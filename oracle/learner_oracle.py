"""numpy float64 restatement of the learner arithmetic (agent.py:90-116, 209-264) -- TEST INFRASTRUCTURE ONLY.

NN PARITY UNPINNED: Keras/TensorFlow are not installed and the reference pins no learner output, so this
follows the documented semantics of Dense/relu/softmax, the reference's huber_loss (agent.py:91-99), Keras'
categorical_crossentropy (target used as is) and plain SGD.  Each row gets its own TD target (the reference's
row-0-only overwrite, agent.py:241, is a bug that is not reproduced -- see DESIGN.md).
"""
import numpy as np

NET_PARAMS = 2179


def split(w):
    w = np.asarray(w, np.float64)
    return w[:1920].reshape(30, 64), w[1920:1984], w[1984:2176].reshape(64, 3), w[2176:2179]


def bits(m):
    return ((np.asarray(m, np.uint32)[:, None] >> np.arange(30)) & 1).astype(np.float64)


def br_grad(w, w_target, s, s2, a, r, t, gamma, terminal_bootstraps=False, others_to_target=False):
    """Mean gradient (flat, 2179) of the Huber loss on the taken action; also the exploitability proxy sum."""
    g, expl, loss, _ = _br(w, w_target, s, s2, a, r, t, gamma, terminal_bootstraps, others_to_target)
    return g, expl, loss


def avg_grad(w, s, y):
    g, loss, _ = _avg(w, s, y)
    return g, loss


def _br(w, w_target, s, s2, a, r, t, gamma, terminal_bootstraps, others_to_target):
    W1, b1, W2, b2 = split(w)
    T1, tb1, T2, tb2 = split(w_target)
    x, x2 = bits(s), bits(s2)
    pre = x @ W1 + b1
    h = np.maximum(pre, 0)
    z = h @ W2 + b2
    q = np.maximum(z, 0)
    qn = np.maximum(np.maximum(x2 @ T1 + tb1, 0) @ T2 + tb2, 0).max(1)
    expl = np.maximum(np.maximum(x @ T1 + tb1, 0) @ T2 + tb2, 0).max(1).sum()
    live = np.ones(len(s)) if terminal_bootstraps else 1.0 - np.asarray(t, np.float64)
    y = np.asarray(r, np.float64) + gamma * live * qn
    n = len(s)
    rows = np.arange(n)
    a = np.asarray(a, np.int64)
    qs = np.maximum(np.maximum(x @ T1 + tb1, 0) @ T2 + tb2, 0)       # target net on s: agent.py:220
    tgt = qs.copy() if others_to_target else q.copy()                   # outputs not taken: to qs, or zero error
    tgt[rows, a] = y
    err = tgt - q
    dz = -np.where(np.abs(err) > 1, np.sign(err), err) / 3.0 * (z > 0)
    loss = (np.where(np.abs(err) > 1, np.abs(err) - 0.5, 0.5 * err * err) / 3.0).sum()
    on = np.ones(z.shape, bool) if others_to_target else np.arange(3) == a[:, None]   # outputs with a derivative
    seen = {"margin": min(np.abs(pre).min(), np.abs(z[on]).min()), "huber_linear": int((np.abs(err[on]) > 1).sum()),
            "huber_quadratic": int((np.abs(err[on]) <= 1).sum()), "log_clamped": 0}
    return _backprop(x, h, W2, dz, n), expl, loss, seen


def _avg(w, s, y):
    W1, b1, W2, b2 = split(w)
    x = bits(s)
    pre = x @ W1 + b1
    h = np.maximum(pre, 0)
    z = h @ W2 + b2
    e = np.exp(z - z.max(1, keepdims=True))
    p = e / e.sum(1, keepdims=True)
    y = np.asarray(y, np.float64)
    dz = p * y.sum(1, keepdims=True) - y
    loss = -(y * np.log(np.maximum(p, 1e-7))).sum()
    seen = {"margin": np.abs(pre).min(), "huber_linear": 0, "huber_quadratic": 0,
            "log_clamped": int(((p < 1e-7) & (y != 0)).sum())}
    return _backprop(x, h, W2, dz, len(s)), loss, seen


def _backprop(x, h, W2, dz, n):
    dh = (dz @ W2.T) * (h > 0)
    g = np.concatenate([(x.T @ dh).ravel(), dh.sum(0), (h.T @ dz).ravel(), dz.sum(0)]) / n
    return g


def fit(w, w_target, rl, sl, minibatch, fit_batch, epochs, lr, gamma, net_mask=0xF, terminal_bootstraps=False,
        others_to_target=False, peers=()):
    """Keras' fit() of the four nets as the one-launch fit runs it: every epoch takes the sampled rows in slices
    [row0, min(row0 + fit_batch, minibatch)), and after each slice w -= lr * mean gradient.

    w [4, 2179]: net k = player * 2 + {0 average policy, 1 best response}; w_target [2, 2179]: the players' target nets.
    rl[p], sl[p]: player p's sampled records in row order (fields of orc.RL_DT / orc.SL_DT, at least `minibatch` rows).
    lr[k]: the learning rate of net k.  Nets whose net_mask bit is clear keep their weights.
    peers: the (rl, sl) of further ranks training together.  Every step then applies the mean of the ranks' mean
    gradients, and the statistics are sums over the ranks.

    Returns (weights [4, 2179], stats [8], margin, seen):
    - stats: those of the first step, laid out as the kernels write them: [0,1] exploitability-proxy sums and [2,3] row
      counts of the best-response nets, [4..7] loss sums of the nets.  NaN where a net does not train.
    - margin: the smallest |hidden pre-activation| of a trained net and |output z| of a best-response output with a
      derivative, over every step and row.  These are the only points where the derivative jumps: Huber's derivative is
      continuous at |e| = 1, and the target net and its max are only evaluated.  An fp32 run of the same fit can only
      take another branch where this margin is within its rounding.
    - seen: over every step, the errors that took the linear / quadratic Huber branch, and the average-policy
      probabilities with a non-zero target that fell under the log's 1e-7 clamp."""
    W = np.array(w, np.float64).reshape(4, NET_PARAMS)
    T = np.asarray(w_target, np.float64).reshape(2, NET_PARAMS)
    lr = np.asarray(lr, np.float64)
    ranks = [(rl, sl)] + list(peers)
    stats = np.full(8, np.nan)
    margin = np.inf
    seen = {"huber_linear": 0, "huber_quadratic": 0, "log_clamped": 0}
    first = True
    for _ in range(epochs):
        for row0 in range(0, minibatch, fit_batch):
            rows = slice(row0, min(row0 + fit_batch, minibatch))
            for k in range(4):
                if not (net_mask >> k) & 1:
                    continue
                p = k >> 1
                g, loss, expl, n = 0.0, 0.0, 0.0, 0
                for rl_r, sl_r in ranks:
                    if k & 1:
                        b = rl_r[p][rows]
                        gr, ex, ls, info = _br(W[k], T[p], b["s"], b["s2"], b["a"], b["r"], b["t"], gamma,
                                               terminal_bootstraps, others_to_target)
                        expl += ex
                    else:
                        b = sl_r[p][rows]
                        gr, ls, info = _avg(W[k], b["s"], b["a"])
                    g, loss, n = g + gr, loss + ls, n + len(b)
                    margin = min(margin, info["margin"])
                    for key in seen:
                        seen[key] += info[key]
                if first:
                    stats[4 + k] = loss
                    if k & 1:
                        stats[p], stats[2 + p] = expl, n
                W[k] = W[k] - lr[k] * (g / len(ranks))
            first = False
    return W, stats, margin, seen


def dyadic_net(rng):
    """One net whose step-0 forward pass is exact in fp32 and whose pre-activations all start >= 1/64 from zero:
    W1 and W2 entries multiples of 1/32 in [-1/4, 1/4], b1 odd multiples of 1/64, b2 odd multiples of 1/4096 plus 1/4.
    With such weights an fp32 fit and a float64 one take the same relu branches for many more steps than with
    Glorot-uniform weights, whose pre-activations come arbitrarily close to zero."""
    w = np.zeros(NET_PARAMS)
    w[:1920] = rng.randint(-8, 9, 1920) / 32.0
    w[1920:1984] = (2 * rng.randint(-8, 8, 64) + 1) / 64.0
    w[1984:2176] = rng.randint(-8, 9, 192) / 32.0
    w[2176:] = (2 * rng.randint(-64, 64, 3) + 1) / 4096.0 + 0.25
    return w


def fit_case(seed, minibatch, slots=256):
    """A seeded fit input with every edge a learner kernel must handle, built by hand rather than by a rollout.

    - Four dyadic acting nets and two dyadic target nets.  The output biases of player 1's average-policy net are
      offset by +64 / -64 chips, so its logits span more than 100: exp underflows in fp32 and the log clamp is hit.
    - `slots` RL and SL records per player: observations 0 and 0x3FFFFFFF (all 30 bits, in slots 0 and 1) beside ones
      with about a quarter of the bits set; rewards from -13 to +13 chips in half-chip steps; terminal flags 0 and 1; random bytes
      in the record's player / flags fields, which the learner must ignore; one-hot SL targets beside unnormalised ones
      and an all-zero one (slot 2).  Every value is exact in fp32.
    - Sampled slot indices per memory: `minibatch` draws that repeat and run out of order, slots 0, 1 and 2 among them.
    Returns a dict: w [4, 2179], w_target [2, 2179], rl_slots / sl_slots (per player, orc.RL_DT / orc.SL_DT),
    idx_rl / idx_sl (per player, int64), rl / sl (per player, the sampled records in row order) and lr [4] (four
    different learning rates, so that one applied to the wrong net shows)."""
    from .orc import RL_DT, SL_DT

    rng = np.random.RandomState(seed)
    w = np.stack([dyadic_net(rng) for _ in range(4)])
    w[2, 2176:2178] += (64.0, -64.0)
    wt = np.stack([dyadic_net(rng) for _ in range(2)])

    def obs():
        o = (rng.randint(0, 1 << 30, slots) & rng.randint(0, 1 << 30, slots)).astype(np.uint32)
        o[:2] = (0, 0x3FFFFFFF)
        return o

    def draws():
        idx = rng.randint(0, slots, minibatch).astype(np.int64)
        idx[rng.choice(minibatch, 3, replace=False)] = (0, 1, 2)
        return idx

    rl_slots, sl_slots = [], []
    for _ in range(2):
        rl = np.zeros(slots, RL_DT)
        rl["s"], rl["s2"] = obs(), obs()
        rl["r"] = rng.randint(-26, 27, slots) * 0.5
        rl["a"] = rng.randint(0, 3, slots)
        rl["t"] = rng.rand(slots) < 0.3
        rl["player"], rl["flags"] = rng.randint(0, 256, slots), rng.randint(0, 256, slots)
        sl = np.zeros(slots, SL_DT)
        sl["s"] = obs()
        y = rng.randint(0, 33, (slots, 3)) / 32.0                 # unnormalised
        one_hot = rng.rand(slots) < 0.5
        y[one_hot] = np.eye(3)[rng.randint(0, 3, int(one_hot.sum()))]
        y[2] = 0.0
        sl["a"] = y
        rl_slots.append(rl)
        sl_slots.append(sl)
    idx_rl, idx_sl = [draws() for _ in range(2)], [draws() for _ in range(2)]
    return {"w": w, "w_target": wt, "rl_slots": rl_slots, "sl_slots": sl_slots, "idx_rl": idx_rl, "idx_sl": idx_sl,
            "rl": [rl_slots[p][idx_rl[p]] for p in range(2)], "sl": [sl_slots[p][idx_sl[p]] for p in range(2)],
            "lr": np.array([0.02, 0.05, 0.01, 0.03])}
