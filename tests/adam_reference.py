"""numpy float64 restatement of the learner's Adam fit -- TEST INFRASTRUCTURE ONLY.

The gradients are oracle/learner_oracle's (the same mean gradients its SGD `fit` applies); what this adds is Keras 2's
Adam update with its fixed constants and the optimizer state of the four nets:

    m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;  w -= lr sqrt(1 - b2^t) / (1 - b1^t) m / (sqrt(v) + eps)

with b1 = 0.9, b2 = 0.999, eps = 1e-7 and t = 1, 2, ... counted per net (only over the steps the net takes).
"""
import numpy as np

from oracle.learner_oracle import NET_PARAMS, _avg, _br

BETA1, BETA2, EPS = 0.9, 0.999, 1e-7


def adam_step(w, m, v, g, lr, t):
    """One Adam step of float64 arrays; returns the new (w, m, v)."""
    m = BETA1 * m + (1 - BETA1) * g
    v = BETA2 * v + (1 - BETA2) * g * g
    lr_t = lr * np.sqrt(1 - BETA2 ** t) / (1 - BETA1 ** t)
    return w - lr_t * m / (np.sqrt(v) + EPS), m, v


def fit(w, w_target, rl, sl, minibatch, fit_batch, epochs, lr, gamma, m=None, v=None, t=(0, 0, 0, 0), net_mask=0xF,
        terminal_bootstraps=False, others_to_target=False, peers=()):
    """learner_oracle.fit with Adam steps: the same slices, gradients, statistics and peers.  m, v [4, 2179] (default
    zero) and t [4] are the optimizer state before the fit; nets whose net_mask bit is clear keep their weights, m, v and
    t.  Returns (weights, m, v, t, stats, margin): the first four are the state the next fit takes; stats and margin are
    learner_oracle.fit's (the first step's statistics; the smallest distance of a relu gate from its kink)."""
    W = np.array(w, np.float64).reshape(4, NET_PARAMS)
    T = np.asarray(w_target, np.float64).reshape(2, NET_PARAMS)
    M = np.zeros((4, NET_PARAMS)) if m is None else np.array(m, np.float64).reshape(4, NET_PARAMS)
    V = np.zeros((4, NET_PARAMS)) if v is None else np.array(v, np.float64).reshape(4, NET_PARAMS)
    t = [int(x) for x in t]
    lr = np.asarray(lr, np.float64)
    ranks = [(rl, sl)] + list(peers)
    stats = np.full(8, np.nan)
    first, margin = True, np.inf
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
                if first:
                    stats[4 + k] = loss
                    if k & 1:
                        stats[p], stats[2 + p] = expl, n
                t[k] += 1
                W[k], M[k], V[k] = adam_step(W[k], M[k], V[k], g / len(ranks), lr[k], t[k])
            first = False
    return W, M, V, t, stats, margin
