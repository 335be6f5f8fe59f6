"""float64 restatement of the acting nets with a rounding bound -- TEST INFRASTRUCTURE ONLY.

forward64 is the two heads of agent.py:101-112 (Dense 30 -> 64 relu -> 3, then relu for the best response, softmax
for the average policy) in float64.  bound() is a per-element bound on how far ANY fp32 evaluation of the same net may
land from it, whatever the summation order, derived (not measured) as follows.  For an observation with s set bits:

    A_j = |b1_j| + sum_{i set} |W1_ij|              (the first layer's sum of magnitudes; relu is 1-Lipschitz)
    M_c = |b2_c| + sum_j A_j |W2_jc|                (the logit's, through both layers)
    e_c = gamma_n M_c,   gamma_n = n u / (1 - n u)  (Higham's bound for a sum of n terms in any order)

CUDA cores (every forward and rollout variant but the tcgen05 ones, the factorised first layer's two precombined rows
included): the hidden unit is a sum of s + 1 terms and the logit one of 65, so n = s + 66 covers both, u = 2^-24.
tcgen05: every first-layer weight enters the tensor core as three exact bf16 terms (hi + mid + lo = w) multiplied by an
exact 0/1 input, so the hidden unit is a sum of 3 (s + 1) terms: n = 3 (s + 1) + 65.  The tensor core's fp32
accumulation is not documented to round to nearest, so u = 2^-23 there (one full ulp per addition: truncation is
covered too).
Relu heads: e_c.  Softmax heads: the softmax is 1/2-Lipschitz in the infinity norm (row i of its Jacobian has
infinity-norm 2 p_i (1 - p_i) <= 1/2), so 0.5 max_c e_c, plus 2^-20 for expf (<= 2 ulp on each of the three
exponentials) and the sum, reciprocal and product after it (relative 2^-22 + 2^-22 + 4 * 2^-24 < 2^-20 of an output
<= 1).

families() are host-built weight sets [4, 2179] float32 (avg0, br0, avg1, br1), each for the edge it contains; see
its docstring.
"""
from __future__ import annotations

import functools
import os

import numpy as np

NET_PARAMS = 2179
U_FP32, U_TC = 2.0 ** -24, 2.0 ** -23
SOFTMAX_SLACK = 2.0 ** -20
EXACT = ("exact", "tied", "dead", "saturated")   # every path computes every logit of these exactly
TRAINED_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "trained_nets.npz")


def bits(obs):
    """observation masks -> float64 [n, 30] inputs (newenv.py:118 bit order)."""
    return ((np.asarray(obs, np.int64)[:, None] >> np.arange(30)) & 1).astype(np.float64)


def split(w):
    """flat [2179] -> W1 (30,64), b1 (64,), W2 (64,3), b2 (3,) in float64."""
    w = np.asarray(w, np.float64)
    return w[:1920].reshape(30, 64), w[1920:1984], w[1984:2176].reshape(64, 3), w[2176:2179]


def logits64(w, obs):
    W1, b1, W2, b2 = split(w)
    return np.maximum(bits(obs) @ W1 + b1, 0.0) @ W2 + b2


def head64(z, net):
    if net & 1:                                        # best response: relu head (agent.py:103)
        return np.maximum(z, 0.0)
    e = np.exp(z - z.max(1, keepdims=True))            # average policy: softmax head (agent.py:112)
    return e / e.sum(1, keepdims=True)


def forward64(w, obs, net):
    """Net `net` (0..3) of a [4, 2179] weight set, or a single [2179] net, on observation masks: float64 [n, 3]."""
    w = np.asarray(w)
    return head64(logits64(w[net] if w.ndim == 2 else w, obs), net)


def bound(w, obs, net, path):
    """Per-element bound [n, 3] on |fp32 evaluation - forward64| for path "cuda" (CUDA cores) or "tc" (tcgen05 first
    layer); see the module docstring."""
    w = np.asarray(w)
    W1, b1, W2, b2 = split(w[net] if w.ndim == 2 else w)
    x = bits(obs)
    s = x.sum(1, keepdims=True)
    A = np.abs(b1) + x @ np.abs(W1)
    M = np.abs(b2) + A @ np.abs(W2)
    n, u = (s + 66, U_FP32) if path == "cuda" else (3 * (s + 1) + 65, U_TC)
    e = n * u / (1 - n * u) * M
    if net & 1:
        return e
    return np.broadcast_to(0.5 * e.max(1, keepdims=True) + SOFTMAX_SLACK, e.shape).copy()


def top_gap(y):
    """Distance between the largest and the second largest entry of each row."""
    s = np.sort(y, axis=1)
    return s[:, -1] - s[:, -2]


# ------------------------------------------------------------------------------------------------ tcgen05 emulation
def bf16_rn(x):
    """float32 -> nearest bf16 (ties to even), returned as float32."""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000
    return b.astype(np.uint32).view(np.float32)


def bf16_splits(w):
    """pack_tc_wide_kernel's split of fp32 weights into hi + mid + lo bf16 terms (each step's remainder is exact)."""
    w = np.asarray(w, np.float32)
    hi = bf16_rn(w)
    r1 = w - hi
    mid = bf16_rn(r1)
    lo = bf16_rn(r1 - mid)
    return hi, mid, lo


def tc_forward32(w, obs, net, drop_lo=False):
    """fp32 emulation of the tcgen05 forward: the first layer as the tensor core's sum of split terms (hi of every k,
    then mid, then lo, accumulated in fp32), layer 2 and the head in fp32.  drop_lo leaves the lo terms out."""
    w = np.asarray(w, np.float32)
    w = w[net] if w.ndim == 2 else w
    x = bits(obs).astype(np.float32)
    W1b = np.concatenate([w[:1920].reshape(30, 64), w[1920:1984][None]], 0)   # the constant 1 input carries b1
    xb = np.concatenate([x, np.ones((len(x), 1), np.float32)], 1)
    h = np.zeros((len(x), 64), np.float32)
    for part in bf16_splits(W1b)[: 2 if drop_lo else 3]:
        for k in range(31):
            h = (h + xb[:, k:k + 1] * part[k]).astype(np.float32)
    h = np.maximum(h, np.float32(0))
    W2, b2 = w[1984:2176].reshape(64, 3), w[2176:2179]
    z = np.zeros((len(x), 3), np.float32)
    for j in range(64):
        z = (z + h[:, j:j + 1] * W2[j]).astype(np.float32)
    z = (z + b2).astype(np.float32)
    if net & 1:
        return np.maximum(z, np.float32(0))
    e = np.exp((z - z.max(1, keepdims=True)).astype(np.float32))
    return (e / e.sum(1, keepdims=True, dtype=np.float32)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ weight families
def game_observations():
    """Every observation a player can be asked to act on (both seats), sorted."""
    from nfsp_b200 import exploitability as ex

    return np.array(sorted(set(ex.information_states()[0]) | set(ex.information_states()[1])), np.uint32)


def random_masks(n=5000, seed=17):
    return np.random.RandomState(seed).randint(0, 1 << 30, n).astype(np.uint32)


def _dyadic_net(rng):
    """oracle/learner_oracle.dyadic_net: W1, W2 multiples of 1/32 in [-1/4, 1/4], b1 odd multiples of 1/64, b2 odd
    multiples of 1/4096 plus 1/4.  Every weight is one bf16 term (mid = lo = 0) and every partial sum of a forward is a
    multiple of 1/4096 far below 2^24 of them: exact in fp32 in any order."""
    w = np.zeros(NET_PARAMS)
    w[:1920] = rng.randint(-8, 9, 1920) / 32.0
    w[1920:1984] = (2 * rng.randint(-8, 8, 64) + 1) / 64.0
    w[1984:2176] = rng.randint(-8, 9, 192) / 32.0
    w[2176:] = (2 * rng.randint(-64, 64, 3) + 1) / 4096.0 + 0.25
    return w


def _lo_split_net(rng):
    """A dyadic net whose first layer needs all three bf16 terms: b1 = +-(2^18 + odd) 2^-16 has 19 significant bits,
    hi and mid hold 16 of them and lo the rest.  W1: multiples of 1/32 in [-1/8, 1/8]; W2: 16 entries of +-1/4 per
    output, the rest 0.  A hidden unit is then a multiple of 2^-16 below 12 and a logit one of 2^-18 below
    16 * 12 / 4 + 1/2 = 48.5 < 2^(24 - 18) (+ 4 for the best-response offset of families()): every partial sum is exact
    in fp32, in any order and on the tensor cores, so dropping the lo term shows as a wrong last bit."""
    w = np.zeros(NET_PARAMS)
    w[:1920] = rng.randint(-4, 5, 1920) / 32.0
    w[1920:1984] = np.where(rng.rand(64) < 0.5, -1, 1) * (2 ** 18 + 2 * rng.randint(0, 2 ** 17, 64) + 1) * 2.0 ** -16
    W2 = np.zeros((64, 3))
    for c in range(3):
        W2[rng.choice(64, 16, replace=False), c] = np.where(rng.rand(16) < 0.5, -0.25, 0.25)
    w[1984:2176] = W2.reshape(-1)
    w[2176:] = (2 * rng.randint(-64, 64, 3) + 1) / 4096.0 + 0.25
    return w


def exactly_computed(w, obs):
    """True when every partial sum of every forward of the four nets on `obs` is exactly representable in fp32 (and so
    computed exactly in any order): each is a multiple of the finest power of two the weights sit on, below 2^24 of
    those in magnitude (M_c, A_j bound every partial sum)."""
    def grid(v):
        v = np.abs(v[v != 0])
        e = 0
        while np.any(v * 2.0 ** e != np.round(v * 2.0 ** e)):
            e += 1
        return 2.0 ** -e

    for k in range(4):
        W1, b1, W2, b2 = split(w[k])
        g1 = min(grid(W1), grid(b1))
        gz = min(g1 * grid(W2), grid(b2))
        x = bits(obs)
        A = np.abs(b1) + x @ np.abs(W1)
        M = np.abs(b2) + A @ np.abs(W2)
        # tcgen05: the split terms of a weight sit on its grid and |hi| + |mid| + |lo| <= |w| (1 + 2^-7)
        if A.max() * (1 + 2.0 ** -7) >= 2.0 ** 24 * g1 or M.max() >= 2.0 ** 24 * gz:
            return False
    return True


def _trained():
    if not os.path.exists(TRAINED_PATH):
        return {}
    with np.load(TRAINED_PATH) as z:
        return {"trained-%s" % str(label): np.ascontiguousarray(w, np.float32) for label, w in zip(z["labels"], z["w"])}


@functools.lru_cache(maxsize=None)
def _families():
    obs = np.concatenate([game_observations(), random_masks()])
    out = {}
    rng = np.random.RandomState(2026)
    # exact: every logit exact on every path, with b1 carrying a lo split
    w = np.stack([_lo_split_net(rng) for _ in range(4)])
    w[[1, 3], 2176:] += 4.0                      # best-response Q-values mostly above 0 (M_c stays below 48.5 + 4 < 64)
    out["exact"] = w
    # tied: best response and average policy of player 0 with W2 columns 0 = 1, of player 1 with 0 = 1 = 2 (b2 too):
    # exact two- and three-way ties at every state, equal softmax outputs
    w = np.stack([_dyadic_net(rng) for _ in range(4)])
    for k in range(4):
        W2 = w[k, 1984:2176].reshape(64, 3)
        tie = (1,) if k < 2 else (1, 2)
        for c in tie:
            W2[:, c] = W2[:, 0]
            w[k, 2176 + c] = w[k, 2176]
    out["tied"] = w
    # dead: best-response b2 lowered (by a multiple of 1/4) to the median over the game's observations of the largest
    # Q-value, so that about half of the states have all three Q-values 0 (the non-zero flag off, agent.py:134)
    w = np.stack([_dyadic_net(rng) for _ in range(4)])
    for k in (1, 3):
        t = np.ceil(4 * np.median(logits64(w[k], game_observations()).max(1))) / 4
        w[k, 2176:] -= t
    out["dead"] = w
    # saturated: average-policy b2 offsets +96 / -64 (logit spans > 104: probabilities exactly 0, and > 17: exactly 1;
    # logits > 88.7, where expf without the max subtraction overflows), best-response Q-values up to +20 and beyond
    w = np.stack([_dyadic_net(rng) for _ in range(4)])
    for k in (0, 2):
        w[k, 2176:2178] += (96.0, -64.0)
    for k in (1, 3):
        w[k, 2176] += 20.0
    out["saturated"] = w
    # full-mantissa: random fp32 weights (every bf16 split in use), hidden sums of tens
    w = np.zeros((4, NET_PARAMS), np.float32)
    for k in range(4):
        w[k, :1920] = rng.uniform(-4, 4, 1920)
        w[k, 1920:1984] = rng.uniform(-3, 3, 64)
        w[k, 1984:2176] = rng.uniform(-0.5, 0.5, 192)
        w[k, 2176:] = rng.uniform(-1, 1, 3)
    out["full-mantissa"] = w
    out = {k: np.ascontiguousarray(v, np.float32) for k, v in out.items()}
    for k in EXACT:
        assert np.array_equal(out[k].astype(np.float64), out[k].astype(np.float64).astype(np.float32)), k
        assert exactly_computed(out[k].astype(np.float64), obs), k
    out.update(_trained())
    return out


def families():
    """{name: float32 [4, 2179]}, each weight set for the edge it contains:

    exact          dyadic weights whose every partial sum is exact in fp32 (so every path computes every logit exactly),
                   with 19-bit first-layer biases that need the lo bf16 term on the tensor cores
    tied           exact (dyadic_net), W2 columns 0 = 1 (player 0's nets) and 0 = 1 = 2 (player 1's), b2 likewise
    dead           exact, best-response b2 lowered so that all three Q-values are 0 on about half of the states
    saturated      exact, average-policy b2 offsets +96 / -64 and a best-response offset of +20
    full-mantissa  random fp32 weights: the rounding of every path at work
    trained-*      snapshots of the engine's own training (tests/golden/trained_nets.npz, oracle/gen_trained_nets.py)
    """
    return {k: v.copy() for k, v in _families().items()}
