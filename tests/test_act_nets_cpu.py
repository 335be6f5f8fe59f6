"""The float64 reference of the acting nets and its rounding bound (tests/act_reference.py) on the CPU.

The bound is only worth something if every correct fp32 evaluation stays inside it and a wrong one does not: the C
oracle's forward and numpy float32 in three summation orders must stay inside it on every family (and be bit-exact on the
exact ones), and an emulated tcgen05 forward must be bit-exact on the exact families with its three bf16 terms and not
with two."""
import numpy as np
import pytest

import act_reference as ar
from oracle import orc


@pytest.fixture(scope="module")
def fam():
    return ar.families()


@pytest.fixture(scope="module")
def obs():
    return np.concatenate([ar.game_observations(), ar.random_masks()])


def _oracle_nets(w):
    return orc.Nets([dict(W1=w[k, :1920].reshape(30, 64), b1=w[k, 1920:1984], W2=w[k, 1984:2176].reshape(64, 3),
                          b2=w[k, 2176:]) for k in range(4)])


def _np32(w, obs, net, order):
    """fp32 forward in numpy: "up" / "down" sum the inputs of each unit in ascending / descending index order, "blas"
    leaves the order (and any FMA) to the matrix product."""
    w = np.asarray(w[net], np.float32)
    x = ar.bits(obs).astype(np.float32)
    W1, b1, W2, b2 = w[:1920].reshape(30, 64), w[1920:1984], w[1984:2176].reshape(64, 3), w[2176:]
    if order == "blas":
        h = np.maximum(x @ W1 + b1, np.float32(0))
        z = h @ W2 + b2
    else:
        idx = range(30) if order == "up" else range(29, -1, -1)
        h = np.zeros((len(x), 64), np.float32) if order == "up" else np.broadcast_to(b1, (len(x), 64)).astype(np.float32)
        for i in idx:
            h = (h + x[:, i:i + 1] * W1[i]).astype(np.float32)
        if order == "up":
            h = (h + b1).astype(np.float32)
        h = np.maximum(h, np.float32(0))
        z = np.zeros((len(x), 3), np.float32)
        for j in (range(64) if order == "up" else range(63, -1, -1)):
            z = (z + h[:, j:j + 1] * W2[j]).astype(np.float32)
        z = (z + b2).astype(np.float32)
    if net & 1:
        return np.maximum(z, np.float32(0))
    e = np.exp((z - z.max(1, keepdims=True)).astype(np.float32))
    return (e / e.sum(1, keepdims=True, dtype=np.float32)).astype(np.float32)


def _check(got, w, obs, k, path, exact):
    ref = ar.forward64(w, obs, k)
    bnd = ar.bound(w, obs, k, path)
    err = np.abs(got.astype(np.float64) - ref)
    assert (err <= bnd).all(), (k, path, float((err / bnd).max()))
    if exact and k & 1:
        assert np.array_equal(got.astype(np.float64), ref), k
    return float((err / bnd).max())


def test_families_have_their_edges(fam, obs):
    assert {"exact", "tied", "dead", "saturated", "full-mantissa"} <= set(fam)
    g = ar.game_observations()
    assert len(g) == 387
    for name, w in fam.items():
        assert w.shape == (4, 2179) and w.dtype == np.float32, name
    # exact: 19-bit first-layer biases, so the tensor cores need the lo term
    assert (ar.bf16_splits(fam["exact"][:, 1920:1984])[2] != 0).mean() > 0.5
    # tied: exact ties at every state
    for k in range(4):
        y = ar.forward64(fam["tied"], g, k)
        assert (y[:, 0] == y[:, 1]).all() and (k < 2 or (y[:, 0] == y[:, 2]).all())
    # dead: all three Q-values 0 on some states, not on all
    for k in (1, 3):
        dead = (ar.forward64(fam["dead"], g, k) == 0).all(1)
        assert 0 < dead.sum() < len(g)
    # saturated: logit spans beyond 104 (probability exactly 0) and 17 (exactly 1), logits beyond expf's overflow,
    # Q-values of 20
    for k in (0, 2):
        z = ar.logits64(fam["saturated"][k], g)
        assert (z.max(1) - z.min(1)).min() > 104 and z.max() > 88.8
    assert max(ar.forward64(fam["saturated"], g, k).max() for k in (1, 3)) >= 20
    # full-mantissa: hidden sums of tens
    W1, b1 = fam["full-mantissa"][0, :1920].reshape(30, 64), fam["full-mantissa"][0, 1920:1984]
    assert np.abs(ar.bits(g) @ W1 + b1).max() > 10


def test_trained_fixture_provenance_and_scale():
    """tests/golden/trained_nets.npz: shapes, provenance, and Q-values of at least one chip on the game's observations
    (what the family is for: outputs far from 1, where a fixed 1e-5 tolerance is a few ulps)."""
    with np.load(ar.TRAINED_PATH) as z:
        d = {k: z[k] for k in z.files}
    S = len(d["labels"])
    assert S >= 4 and d["w"].shape == (S, 4, 2179) and d["w"].dtype == np.float32
    assert d["iterations"].shape == (S,) and d["optimizer"].shape == (S,) and set(d["optimizer"].tolist()) == {"sgd", "adam"}
    for key in ("command", "seed", "games", "commit", "card", "power_limit"):
        assert key in d and str(d[key]), key
    assert int(d["games"]) == 65536
    g = ar.game_observations()
    for label, w in zip(d["labels"], d["w"]):
        q = max(np.abs(ar.logits64(w[k], g)).max() for k in (1, 3))
        assert q >= 1.0, (str(label), q)
    trained = [k for k in ar.families() if k.startswith("trained-")]
    assert len(trained) == S


def test_oracle_forward_within_the_bound(fam, obs):
    """orc.Nets.forward (the C oracle, fp32, inputs in ascending order then the bias)."""
    sub = obs[::4]
    for name, w in fam.items():
        nets = _oracle_nets(w)
        x = ar.bits(sub).astype(np.float32)
        for k in range(4):
            got = nets.forward(k, x, "br" if k & 1 else "avg")
            _check(got, w, sub, k, "cuda", name in ar.EXACT)


@pytest.mark.parametrize("order", ["up", "down", "blas"])
def test_numpy_fp32_orders_within_the_bound(fam, obs, order):
    for name, w in fam.items():
        for k in range(4):
            _check(_np32(w, obs, k, order), w, obs, k, "cuda", name in ar.EXACT)


def test_tcgen05_emulation_needs_all_three_bf16_terms(fam, obs):
    """The tensor-core forward's arithmetic (three bf16 terms per weight, fp32 accumulation) is within the tcgen05 bound
    everywhere and bit-exact on the exact families.  Without the lo term the exact family loses its exactness.

    That is the only place a dropped lo term can show: |lo| <= 2^-8 |mid| <= 2^-16 |w| (in practice below 2^-17 |w|),
    while the tcgen05 bound allows n u >= 71 * 2^-23 > 2^-16.9 of the sum of magnitudes per logit, so on random or
    trained weights a missing lo term stays inside the bound (asserted below, on the full-mantissa family).  Exactness
    is the check that catches it, and the exact family's 19-bit biases are what give it a lo term to lose."""
    sub = obs[::2]
    for name, w in fam.items():
        for k in range(4):
            _check(ar.tc_forward32(w, sub, k), w, sub, k, "tc", name in ar.EXACT)
    w = fam["exact"]
    lost = [not np.array_equal(ar.tc_forward32(w, sub, k, drop_lo=True).astype(np.float64), ar.forward64(w, sub, k))
            for k in (1, 3)]
    assert all(lost)
    w = fam["full-mantissa"]
    for k in range(4):
        ref = ar.forward64(w, sub, k)
        err = np.abs(ar.tc_forward32(w, sub, k, drop_lo=True) - ref)
        assert err.max() > 0 and (err <= ar.bound(w, sub, k, "tc")).all()
