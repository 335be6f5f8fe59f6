"""-m gpu: the acting nets as the rollouts evaluate them, held to float64 (tests/act_reference.py) on trained, saturated,
dead and tied nets.

- Forwards: SelfPlay.forward on the CUDA cores and on tcgen05, every observation of the game plus random masks.
- Scores: every variant's score vector at every decision of the 20 352 reference hands (epsilon 0: each is a net's output),
  which reaches every entry of the "states" variant's table through real launches.
- Production launches (no debug, no forcing) on the exact families, where every decision is determined exactly: records
  and counters equal the oracle's own rollout, also for runs of different families batched in one RunBatch.
- Exploitability: the average policies' tables from the GPU forward equal the float64 ones.

Tolerances are the derived bound of act_reference.bound, never a fixed number: an output of 13 chips and one of 0.3 are
held to what fp32 can do for each.  Exact families (act_reference.EXACT) are held to bit equality of their Q-values.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import act_reference as ar  # noqa: E402
from oracle import orc  # noqa: E402

VARIANTS = ["states", "pairs", "sorted", "cuda", "tcgen05", "tcgen05_ws"]
RATIO = {}   # (path, family) -> largest err / bound seen


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


@pytest.fixture(scope="module")
def fam():
    return ar.families()


@pytest.fixture(scope="module", autouse=True)
def ratio_table():
    yield
    if RATIO:
        print("\nlargest |got - float64| / bound, per path and family:")
        for (path, name), r in sorted(RATIO.items()):
            print("  %-16s %-22s %.3e" % (path, name, r))


def _golden(golden_dir):
    with np.load(os.path.join(golden_dir, "nfsp_exhaustive.npz")) as z:
        return {k: z[k] for k in z.files}


def _canon(recs):
    a = np.ascontiguousarray(recs).view(np.uint32).reshape(-1, 4)
    return a[np.lexsort(a.T[::-1])]


def _oracle_nets(w):
    return orc.Nets([dict(W1=w[k, :1920].reshape(30, 64), b1=w[k, 1920:1984], W2=w[k, 1984:2176].reshape(64, 3),
                          b2=w[k, 2176:]) for k in range(4)])


def _hold(got, w, obs, net, path, name, key):
    """got (fp32 [n, 3]) of net `net` on obs against forward64: within the bound, bit-exact Q-values on an exact family,
    and the first-maximum argmax of float64 wherever its top-two gap exceeds twice the bound (everywhere on an exact
    family)."""
    ref = ar.forward64(w, obs, net)
    bnd = ar.bound(w, obs, net, path)
    err = np.abs(got.astype(np.float64) - ref)
    r = float((err / bnd).max()) if len(obs) else 0.0
    RATIO[(key, name)] = max(RATIO.get((key, name), 0.0), r)
    assert r <= 1.0, (key, name, net, r)
    exact = name in ar.EXACT
    if exact and net & 1:
        bad = np.nonzero((got.astype(np.float64) != ref).any(1))[0]
        assert len(bad) == 0, (key, name, net, obs[bad[:4]], got[bad[:4]], ref[bad[:4]])
    sure = np.ones(len(obs), bool) if exact else ar.top_gap(ref) > 2 * bnd.max(1)
    assert np.array_equal(got[sure].argmax(1), ref[sure].argmax(1)), (key, name, net)


def _all_observations(golden_dir):
    g = _golden(golden_dir)
    dec = np.arange(6)[None, :] < g["n_dec"][:, None]
    seen = np.concatenate([ar.game_observations(), g["obs_before"][dec], g["obs_after"].ravel()])
    return np.concatenate([np.unique(seen), ar.random_masks()])


def test_forwards_every_family(nb, fam, golden_dir):
    """SelfPlay.forward, CUDA cores and tcgen05, per net over all observations (a ragged last tile) and with the four
    nets mixed row by row at 1, 129 and all rows."""
    obs = _all_observations(golden_dir)
    assert len(obs) % 128 != 0
    rng = np.random.RandomState(8)
    mixed = rng.randint(0, 4, len(obs)).astype(np.int8)
    for name, w in fam.items():
        sp = nb.SelfPlay(64, weights=torch.from_numpy(w), rl_capacity=1024, sl_capacity=1024)
        for tc in (False, True):
            path, key = ("tc", "forward-tcgen05") if tc else ("cuda", "forward-cuda")
            for k in range(4):
                got = sp.forward(torch.from_numpy(obs.astype(np.int32)), torch.full((len(obs),), k, dtype=torch.int8),
                                 tensor_cores=tc).cpu().numpy()
                _hold(got, w, obs, k, path, name, key)
            for n in (1, 129, len(obs)):
                got = sp.forward(torch.from_numpy(obs[:n].astype(np.int32)), torch.from_numpy(mixed[:n]),
                                 tensor_cores=tc).cpu().numpy()
                for k in range(4):
                    m = mixed[:n] == k
                    _hold(got[m], w, obs[:n][m], k, path, name, key)


@pytest.mark.parametrize("variant", VARIANTS)
def test_scores_at_every_decision_of_the_reference_hands(nb, fam, golden_dir, variant):
    """The golden-hands launch (set_hands + the reference's scripted vectors) with epsilon 0: out["vec"] holds the score
    vector the kernel read at each decision -- for "states" the table entry -- and must be the acting net's output
    (policy 'a' -> average net, 'b' -> best response) on the observation of that decision.  The hands visit all 387
    observations a player can act on."""
    g = _golden(golden_dir)
    T, D = g["kind"].shape
    forced = np.ascontiguousarray(g["vec"].transpose(1, 0, 2))
    dec = np.arange(D)[None, :] < g["n_dec"][:, None]              # [T, D]: decisions of the reference hand
    gi, di = np.nonzero(dec)
    actor = g["player"][gi, di].astype(np.int64)
    net = 2 * actor + g["policy"][gi, actor].astype(np.int64)
    obs = g["obs_before"][gi, di]
    assert set(ar.game_observations().tolist()) <= set(obs.tolist())
    path = "tc" if variant.startswith("tcgen05") else "cuda"
    for name, w in fam.items():
        sp = nb.SelfPlay(T, weights=torch.from_numpy(w), seed=3, epsilon=0.0, rl_capacity=1024, sl_capacity=1024,
                         max_steps_per_call=D, variant=variant)
        sp.env.set_hands(g["dealer"], g["cards"], g["policy"])
        sp.env.step_counter = 1
        out = sp.rollout(D, insert=False, forced_vec=forced)
        vec = out["vec"].cpu().numpy()[di, gi]
        for k in range(4):
            m = net == k
            _hold(vec[m], w, obs[m], k, path, name, "scores-" + variant)


def _production(nb, w, variant, n, seed, eta, eps, steps, launches):
    sp = nb.SelfPlay(n, weights=torch.from_numpy(w), seed=seed, eta=eta, epsilon=eps, rl_capacity=1 << 12,
                     sl_capacity=1 << 12, max_steps_per_call=steps, variant=variant)
    rl, sl = [[], []], [[], []]
    for _ in range(launches):
        sp.rollout(steps, insert=False)
        r, s = sp.staged()
        for p in range(2):
            rl[p].append(r[p])
            sl[p].append(s[p])
        sp.counts.zero_()
    return sp.read_stats(), [np.concatenate(x) for x in rl], [np.concatenate(x) for x in sl]


def _oracle(w, n, seed, eta, eps, steps, launches):
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(eta))
    nets = _oracle_nets(w)
    refs = [b.rollout_act(1 + k * steps, steps, nets, orc.u32_frac(eta), orc.u32_frac(eps)) for k in range(launches)]
    rl = [np.concatenate([r["rl"][p] for r in refs]) for p in range(2)]
    sl = [np.concatenate([r["sl"][p] for r in refs]) for p in range(2)]
    tot = {k: sum(r[k] for r in refs) for k in ("actions", "played", "reward_half", "hands")}
    return tot, rl, sl


def _same_as_oracle(st, rl, sl, ref, n, steps, launches, tag):
    tot, rrl, rsl = ref
    for p in range(2):
        assert len(rl[p]) == len(rrl[p]) and len(sl[p]) == len(rsl[p]), (tag, p)
        assert np.array_equal(_canon(rl[p]), _canon(rrl[p])), (tag, p)
        assert np.array_equal(_canon(sl[p]), _canon(rsl[p])), (tag, p)
    assert [st["a0_fold"], st["a0_call"], st["a0_raise"]] == list(tot["actions"][0]), tag
    assert [st["a1_fold"], st["a1_call"], st["a1_raise"]] == list(tot["actions"][1]), tag
    assert [st["played0"], st["played1"]] == list(tot["played"]), tag
    to_s = lambda v: v - (1 << 64) if v >= 1 << 63 else v  # noqa: E731
    assert [to_s(st["reward0_half"]), to_s(st["reward1_half"])] == list(tot["reward_half"]), tag
    assert st["hands"] == tot["hands"] and st["transitions"] == n * steps * launches and st["dropped"] == 0, tag


@pytest.mark.parametrize("name", ar.EXACT)
@pytest.mark.parametrize("n", [1, 1000, 50_000])
def test_production_launches_equal_the_oracle(nb, fam, name, n):
    """Every variant's production kernel (kDebug = false: the "states" table's stored action words, no recomputation),
    several launches, epsilon and eta > 0 so that random vectors and both policies occur, against the oracle's own
    rollout (its fp32 forward, no forced vectors).  On an exact family every decision is determined exactly, so the
    staged records (as multisets) and the counters must be equal."""
    w = fam[name]
    steps, launches = (30, 3) if n == 1 else (8, 2)
    seed, eta, eps = 2024 + n, 0.35, 0.2
    ref = _oracle(w, n, seed, eta, eps, steps, launches)
    for variant in VARIANTS:
        st, rl, sl = _production(nb, w, variant, n, seed, eta, eps, steps, launches)
        _same_as_oracle(st, rl, sl, ref, n, steps, launches, (name, n, variant))


def test_runbatch_of_different_families_each_equal_its_oracle(nb, fam):
    """One RunBatch whose runs hold the four exact families (their own seeds, eta and epsilon): two batched rollouts, and
    each run's memories (rings and reservoirs, filled below capacity: every record kept) and counters equal its own
    oracle."""
    from nfsp_b200.learner import Learner
    from nfsp_b200.runs import RunBatch

    n, steps, launches = 4096, 8, 2
    cfg = [(name, 11 + r, 0.1 + 0.1 * r, 0.05 + 0.05 * r) for r, name in enumerate(ar.EXACT)]
    sps = [nb.SelfPlay(n, weights=torch.from_numpy(fam[name]), seed=s, eta=e, epsilon=ep, rl_capacity=1 << 18,
                       sl_capacity=1 << 17, max_steps_per_call=steps) for name, s, e, ep in cfg]
    rb = RunBatch(sps, [Learner(sp) for sp in sps])
    for _ in range(launches):
        rb.rollout(steps)
    torch.cuda.synchronize()
    for sp, (name, s, e, ep) in zip(sps, cfg):
        for m in sp.rl + sp.sl:
            assert int(m.total.item()) == m.size() < m.capacity
        rl, sl = [m.records() for m in sp.rl], [m.records() for m in sp.sl]
        ref = _oracle(fam[name], n, s, e, ep, steps, launches)
        _same_as_oracle(sp.read_stats(), rl, sl, ref, n, steps, launches, name)


def test_policy_tables_from_the_gpu_forward(nb, fam):
    """exploitability.policy_tables over the GPU forward against the float64 forward: identical on the exact families;
    on the trained ones identical wherever the float64 top-two margin exceeds twice the bound (the states left out are
    counted and printed)."""
    from nfsp_b200 import exploitability as ex

    for name, w in fam.items():
        sp = nb.SelfPlay(64, weights=torch.from_numpy(w), rl_capacity=1024, sl_capacity=1024)
        gpu = ex.policy_tables(lambda m, k: sp.forward(torch.from_numpy(m), torch.from_numpy(k)).cpu().numpy())
        ref = ex.policy_tables(lambda m, k: ar.forward64(w, m.astype(np.int64) & 0x3FFFFFFF, int(k[0])))
        excluded = 0
        for p in range(2):
            states = np.array(sorted(ref[p]), np.int64)
            if name in ar.EXACT:
                sure = np.ones(len(states), bool)
            else:
                y = ar.forward64(w, states, 2 * p)
                sure = ar.top_gap(y) > 2 * ar.bound(w, states, 2 * p, "cuda").max(1)
            excluded += int((~sure).sum())
            for s in states[sure]:
                assert gpu[p][int(s)] == ref[p][int(s)], (name, p, int(s))
        if name not in ar.EXACT:
            print("%s: %d of %d states left out of the table comparison (float64 margin within twice the bound)" %
                  (name, excluded, sum(len(t) for t in ref)))
        if name in ar.EXACT:
            assert excluded == 0
