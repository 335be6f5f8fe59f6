"""-m gpu: independent runs side by side (nfsp_b200.runs.RunBatch, nfsp_rollout_runs, nfsp_learner_fit_runs).

Every run of a batch must do exactly what it does alone: the same game words, counters, memories (contents and totals),
acting and target weights and schedules, bit for bit, as the same configuration driven standalone."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import learner_oracle as lo  # noqa: E402


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def _run(nb, n, seed, eta, eps, lr_br=0.05, lr_ar=0.1, **kw):
    from nfsp_b200.learner import Learner

    sp = nb.SelfPlay(n, seed=seed, eta=eta, epsilon=eps, **kw)
    return sp, Learner(sp, lr_br=lr_br, lr_ar=lr_ar)


def _assert_same_run(a, b, la=None, lb=None, tag=""):
    torch.cuda.synchronize()
    assert torch.equal(a.env.state_words(), b.env.state_words()), tag
    assert a.env.step_counter == b.env.step_counter, tag
    assert torch.equal(a.stats, b.stats), tag
    for p in range(2):
        for ma, mb in ((a.rl[p], b.rl[p]), (a.sl[p], b.sl[p])):
            assert torch.equal(ma.total, mb.total), (tag, p)
            assert torch.equal(ma.store, mb.store), (tag, p)
            assert ma.sample_calls == mb.sample_calls, (tag, p)
    assert torch.equal(a.weights, b.weights), tag
    assert a.epsilons == b.epsilons, tag
    if la is not None:
        assert torch.equal(la.target, lb.target), tag
        assert la.iteration == lb.iteration and la.target_update_count == lb.target_update_count, tag
        assert la.lr_br == lb.lr_br and la.temp == lb.temp, tag


CONFIGS = [  # seed, eta, epsilon per player, lr_br, lr_ar
    (1234, 0.1, (0.06, 0.06), 0.05, 0.1),
    (77, 0.3, (0.2, 0.05), 0.02, 0.2),
    (4242, 0.05, (0.1, 0.15), 0.1, 0.05),
]


def test_runs_train_bit_for_bit_like_standalone_runs(nb):
    """Three runs with different seeds, eta, epsilons and learning rates; 10 iterations of rollout(8) with an update
    from the third on.  After every iteration each batched run equals the same configuration driven alone."""
    from nfsp_b200.runs import RunBatch

    kw = dict(rl_capacity=1 << 16, sl_capacity=1 << 16, max_steps_per_call=8, deterministic=True)
    solo = [_run(nb, 4096, s, e, list(ep), lb, la, **kw) for s, e, ep, lb, la in CONFIGS]
    runs = [_run(nb, 4096, s, e, list(ep), lb, la, **kw) for s, e, ep, lb, la in CONFIGS]
    rb = RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])
    trained = 0
    for it in range(10):
        for sp, ln in solo:
            sp.rollout(8)
            if it >= 2:
                trained |= ln.update(sync=False)["trained"]
        rb.rollout(8)
        if it >= 2:
            rb.update(sync=False)
        for r in range(3):
            _assert_same_run(solo[r][0], runs[r][0], solo[r][1], runs[r][1], "iteration %d run %d" % (it, r))
    assert trained == 0xF and all(ln.iteration[0] > 0 for _, ln in runs)
    # the runs really differ from each other
    assert not torch.equal(runs[0][0].weights, runs[1][0].weights)
    # update(sync=True) reads every run's statistics back
    from nfsp_b200.exploitability import exploitability

    out = rb.step(8, sync=True)
    refs = []
    for sp, ln in solo:
        sp.rollout(8)
        refs.append(ln.update(sync=True))
    for r in range(3):
        assert refs[r]["trained"] == 0xF and out[r] == refs[r], r
        _assert_same_run(solo[r][0], runs[r][0], solo[r][1], runs[r][1], "sync step run %d" % r)
    # exact exploitability of each run's average policies (the standalone update rebuilt its images already)
    ex = rb.exploitability()
    for r in range(3):
        assert ex[r] == exploitability(solo[r][0]), r


def test_runs_at_different_counters_train_like_standalone_runs(nb):
    """Runs of one batch at their own step counters, ring tickets and draw counters -- a fresh run, one whose counters
    cross 2^32 during the test and one far past it (a resumed long run): the batched launches take each run's 64-bit
    counters, so every run still equals the same run driven alone, iteration by iteration."""
    from nfsp_b200.runs import RunBatch

    ages = [(0, 0, 0), (2 ** 32 - 20, 2 ** 32 - 40_000, 2 ** 32 - 2), (2 ** 40 + 3, 2 ** 62 + 5, 2 ** 40 + 7)]
    kw = dict(rl_capacity=1 << 16, sl_capacity=1 << 16, max_steps_per_call=8, deterministic=True)

    def aged(r):
        s, e, ep, lb, la = CONFIGS[r]
        sp, ln = _run(nb, 4096, s, e, list(ep), lb, la, **kw)
        step, total, calls = ages[r]
        sp.env.step_counter = sp.env.step_counter + step
        for m in sp.rl:
            m.total.add_(total)
        for m in sp.rl + sp.sl:
            m.sample_calls += calls
        return sp, ln

    solo = [aged(r) for r in range(3)]
    runs = [aged(r) for r in range(3)]
    rb = RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])
    for it in range(6):
        for sp, ln in solo:
            sp.rollout(8)
            if it >= 2:
                ln.update(sync=False)
        rb.rollout(8)
        if it >= 2:
            rb.update(sync=False)
        for r in range(3):
            _assert_same_run(solo[r][0], runs[r][0], solo[r][1], runs[r][1], "iteration %d run %d" % (it, r))
    sp1 = runs[1][0]
    assert sp1.env.step_counter > 2 ** 32 and all(int(m.total.item()) > 2 ** 32 and m.sample_calls > 2 ** 32
                                                  for m in sp1.rl)


def _rows(a):
    return [bytes(x) for x in np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)]


def test_direct_rings_at_sweep_size(nb):
    """Four runs of 65 536 games with direct rings, three rollouts: game words and counters equal the standalone runs',
    and each launch's ring and reservoir records are the same multisets (their order inside a launch follows the
    atomics)."""
    from nfsp_b200.runs import RunBatch

    n, steps = 65536, 8
    kw = dict(rl_capacity=1 << 22, sl_capacity=1 << 21, max_steps_per_call=steps, direct_rings=True)
    solo = [_run(nb, n, s, e, list(ep), lb, la, **kw) for s, e, ep, lb, la in CONFIGS + [(9, 0.2, (0.08, 0.08), 0.05, 0.1)]]
    runs = [_run(nb, n, s, e, list(ep), lb, la, **kw) for s, e, ep, lb, la in CONFIGS + [(9, 0.2, (0.08, 0.08), 0.05, 0.1)]]
    rb = RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])
    for launch in range(3):
        before = [[(int(m.total.item())) for m in sp.rl + sp.sl] for sp, _ in runs]
        for sp, _ in solo:
            sp.rollout(steps)
        rb.rollout(steps)
        torch.cuda.synchronize()
        for r in range(4):
            a, b = solo[r][0], runs[r][0]
            assert torch.equal(a.env.state_words(), b.env.state_words()), (launch, r)
            assert torch.equal(a.stats, b.stats) and a.env.step_counter == b.env.step_counter, (launch, r)
            for k, (ma, mb) in enumerate(zip(a.rl + a.sl, b.rl + b.sl)):
                t0, t1 = before[r][k], int(mb.total.item())
                assert int(ma.total.item()) == t1 and t1 <= ma.capacity, (launch, r, k)
                assert t1 > t0
                assert Counter(_rows(ma.data[t0:t1].cpu().numpy())) == Counter(_rows(mb.data[t0:t1].cpu().numpy())), (launch, r, k)


def _fit_inputs(nb, seed, minibatch, dev):
    """One hand-built learner input (oracle/learner_oracle.fit_case) on the device."""
    c = lo.fit_case(seed, minibatch)
    rng = np.random.RandomState(seed)
    d = {"rl": [], "sl": []}
    for p in range(2):
        rl = np.ascontiguousarray(c["rl_slots"][p]).view(np.int32).reshape(-1, 4)
        sl = np.ascontiguousarray(c["sl_slots"][p]).view(np.int32).reshape(-1, 4)
        tail = rng.randint(-2 ** 31, 2 ** 31, sl.shape, dtype=np.int64).astype(np.int32)
        d["rl"].append(torch.from_numpy(rl.copy()).to(dev))
        d["sl"].append(torch.from_numpy(np.concatenate([sl, tail], 1)).to(dev))
    d["idx_rl"] = [torch.from_numpy(i).to(dev) for i in c["idx_rl"]]
    d["idx_sl"] = [torch.from_numpy(i).to(dev) for i in c["idx_sl"]]
    d["w"] = torch.tensor(c["w"], dtype=torch.float32, device=dev)
    d["wt"] = torch.tensor(c["w_target"], dtype=torch.float32, device=dev)
    return d


def _learner_io(d, flat, mask, tb, ott, gamma):
    from nfsp_b200._lib import LearnerIO
    from nfsp_b200.learner import GRAD

    io = LearnerIO()
    io.d_weights, io.d_target_weights = d["w"].data_ptr(), d["wt"].data_ptr()
    for p in range(2):
        io.d_rl[p], io.d_rl_idx[p] = d["rl"][p].data_ptr(), d["idx_rl"][p].data_ptr()
        io.d_sl[p], io.d_sl_idx[p] = d["sl"][p].data_ptr(), d["idx_sl"][p].data_ptr()
    io.row0, io.rows, io.gamma, io.net_mask = 0, 0, gamma, mask
    io.terminal_bootstraps, io.others_to_target = tb, ott
    io.d_grad, io.d_stats = flat.data_ptr(), flat[GRAD:].data_ptr()
    return io


@pytest.mark.parametrize("geometry", [(128, 32, 2), (320, 80, 2)], ids=["rows-kernel", "register-kernel"])
@pytest.mark.parametrize("aliased", [False, True], ids=["w_out-separate", "w_out-aliased"])
def test_fit_runs_equals_one_fit_per_run(nb, geometry, aliased):
    """nfsp_learner_fit_runs over five runs -- own memories, sampled slots, masks, flags, gamma and learning rates --
    gives the weights and statistics of five nfsp_learner_fit calls, bit for bit."""
    from nfsp_b200._lib import LearnerIO, check
    from nfsp_b200.batched import _ptr, _stream
    from nfsp_b200.learner import GRAD, N_STATS

    dev = torch.device("cuda", torch.cuda.current_device())
    masks, flags = [0xF, 0b0101, 0b1010, 0b0001, 0xF], [(0, 0), (1, 0), (0, 1), (1, 1), (0, 0)]
    gammas = [0.95, 0.9, 0.99, 0.95, 0.5]
    lrs = [[0.1 * (r + 1), 0.05 / (r + 1), 0.2 - 0.01 * r, 0.03 + 0.01 * r] for r in range(5)]
    ins = [_fit_inputs(nb, 100 + r, geometry[0], dev) for r in range(5)]
    # reference: one nfsp_learner_fit per run
    ref_w, ref_s = [], []
    for r, d in enumerate(ins):
        flat = torch.zeros(GRAD + N_STATS, dtype=torch.float32, device=dev)
        w_out = d["w"].clone() if aliased else torch.full_like(d["w"], float("nan"))
        io = _learner_io(dict(d, w=w_out) if aliased else d, flat, masks[r], *flags[r], gammas[r])
        check(nb.lib().nfsp_learner_fit(C.byref(io), *geometry, (C.c_float * 4)(*lrs[r]), _ptr(w_out), _stream(dev)))
        ref_w.append(w_out)
        ref_s.append(flat[GRAD:])
    # the same in one launch
    flats = [torch.zeros(GRAD + N_STATS, dtype=torch.float32, device=dev) for _ in range(5)]
    outs = [d["w"].clone() if aliased else torch.full_like(d["w"], float("nan")) for d in ins]
    ios = (LearnerIO * 5)()
    for r, d in enumerate(ins):
        ios[r] = _learner_io(dict(d, w=outs[r]) if aliased else d, flats[r], masks[r], *flags[r], gammas[r])
    lr = (C.c_float * 20)(*[x for l_ in lrs for x in l_])
    w_ptrs = (C.c_void_p * 5)(*[o.data_ptr() for o in outs])
    check(nb.lib().nfsp_learner_fit_runs(ios, 5, *geometry, lr, w_ptrs, _stream(dev)))
    torch.cuda.synchronize()
    for r in range(5):
        assert torch.equal(outs[r], ref_w[r]), r
        assert torch.equal(flats[r][GRAD:], ref_s[r]), r
        for k in range(4):  # not vacuous: the masked nets trained, the others were copied / left alone
            assert torch.equal(outs[r][k], ins[r]["w"][k]) != bool((masks[r] >> k) & 1), (r, k)


def _io_array(sps):
    from nfsp_b200._lib import RolloutIO

    arr = (RolloutIO * len(sps))()
    for r, sp in enumerate(sps):
        arr[r] = sp._rollout_io()
    return arr


def _call_runs(nb, sps, n_steps=2, n_runs=None, ios=None, weights=False):
    from nfsp_b200.batched import _stream

    R = len(sps)
    h = (C.c_void_p * R)(*[sp.env._h.value for sp in sps])
    eta = (C.c_double * R)(*[sp.eta for sp in sps])
    eps = (C.c_double * R)(*[sp.epsilons[0] for sp in sps])
    w = (C.c_void_p * R)(*[sp.weights.data_ptr() for sp in sps]) if weights else None
    return nb.lib().nfsp_rollout_runs(h, R if n_runs is None else n_runs, n_steps, eta, eps,
                                      _io_array(sps) if ios is None else ios, w, _stream(sps[0].device))


def test_one_run_equals_a_plain_rollout(nb):
    from nfsp_b200.runs import RunBatch

    kw = dict(rl_capacity=1 << 15, sl_capacity=1 << 15, max_steps_per_call=8, deterministic=True)
    (a, la), (b, lb) = _run(nb, 3000, 5, 0.2, [0.1, 0.04], **kw), _run(nb, 3000, 5, 0.2, [0.1, 0.04], **kw)
    rb = RunBatch([b], [lb])
    for it in range(4):
        a.rollout(8)
        rb.rollout(8)
        if it >= 1:
            la.update(sync=False)
            rb.update()
        _assert_same_run(a, b, la, lb, "iteration %d" % it)


def test_as_many_runs_as_the_limit_allows(nb):
    """n_runs = min(NFSP_MAX_RUNS, SMs): every run equals its standalone twin."""
    from nfsp_b200._lib import MAX_RUNS
    from nfsp_b200.runs import RunBatch

    sms = C.c_int()
    nb.lib().nfsp_device_info(torch.cuda.current_device(), C.byref(sms), None, None, None, 0)
    R = min(MAX_RUNS, sms.value)
    kw = dict(rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=4, deterministic=True)
    solo = [_run(nb, 100, 1000 + r, 0.1 + 0.01 * r, 0.06, **kw) for r in range(R)]
    runs = [_run(nb, 100, 1000 + r, 0.1 + 0.01 * r, 0.06, **kw) for r in range(R)]
    rb = RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])
    for _ in range(3):
        for sp, _ in solo:
            sp.rollout(4)
        rb.rollout(4)
    for r in range(R):
        _assert_same_run(solo[r][0], runs[r][0], tag="run %d" % r)
    if R == MAX_RUNS:
        with pytest.raises(ValueError):
            RunBatch([sp for sp, _ in runs] + [solo[0][0]], [ln for _, ln in runs] + [solo[0][1]])


def test_mismatched_runs_are_refused_before_anything_runs(nb):
    """Each difference of shape returns NFSP_E_ARG and leaves every handle's game words and step counter as they were."""
    from nfsp_b200._lib import MAX_RUNS
    from nfsp_b200.learner import Learner
    from nfsp_b200.runs import RunBatch

    base = dict(rl_capacity=1 << 14, sl_capacity=1 << 14, max_steps_per_call=2)
    a = nb.SelfPlay(256, seed=1, **base)
    cases = {
        "games": nb.SelfPlay(288, seed=2, **base),
        "record mode": nb.SelfPlay(256, seed=3, direct_rings=True, **base),
        "ring capacity": nb.SelfPlay(256, seed=4, direct_rings=True, **dict(base, rl_capacity=1 << 13)),
    }
    torch.cuda.synchronize()

    def snapshot(sps):
        return [(sp.env.state_words().clone(), sp.env.step_counter) for sp in sps]

    def same(before, sps):
        torch.cuda.synchronize()
        return all(torch.equal(w, sp.env.state_words()) and c == sp.env.step_counter for (w, c), sp in zip(before, sps))

    for name, b in cases.items():
        pair = [cases["record mode"], b] if name == "ring capacity" else [a, b]
        before = snapshot(pair)
        assert _call_runs(nb, pair) == -1, name
        assert _call_runs(nb, pair, weights=True) == -1, name
        assert same(before, pair), name
        with pytest.raises(ValueError):
            RunBatch(pair, [Learner(sp) for sp in pair])
    # n_segments and reserve_sms differ
    pair = [a, nb.SelfPlay(256, seed=6, **base)]
    before = snapshot(pair)
    for field, value in (("n_segments", pair[1].n_seg // 2), ("reserve_sms", 4)):
        ios = _io_array(pair)
        setattr(ios[1], field, value)
        assert _call_runs(nb, pair, ios=ios) == -1 and same(before, pair), field
    # the same handle twice, a debug output, n_runs out of range
    assert _call_runs(nb, [a, a]) == -1
    ios = _io_array(pair)
    ios[0].d_trace = ios[0].d_counts
    assert _call_runs(nb, pair, ios=ios) == -1
    assert _call_runs(nb, pair, n_runs=0) == -1
    assert _call_runs(nb, pair, n_runs=MAX_RUNS + 1) == -1
    assert same(before, pair)
    # and a valid call still works: both step counters advance
    assert _call_runs(nb, pair, n_steps=2) == 0
    torch.cuda.synchronize()
    assert [sp.env.step_counter for sp in pair] == [c + 2 for _, c in before]


def test_sampling_many_memories_in_one_launch_draws_like_per_memory_calls(nb):
    """4R requests (beyond the eight the parameter block used to hold) in one launch: the positions of
    nfsp_sample_indices / DeviceRing.sample_slots, memory by memory, and the expanded rows of the per-memory gathers."""
    from nfsp_b200._lib import MAX_SAMPLE_REQS, SampleReq, check
    from nfsp_b200.batched import DeviceReservoir, DeviceRing, _ptr, _stream

    dev = torch.device("cuda", torch.cuda.current_device())
    R, b = 10, 64
    g = torch.Generator().manual_seed(3)
    mems = []
    for r in range(R):
        for k in range(4):
            cap = 300 + 37 * r + k
            m = (DeviceRing if k < 2 else DeviceReservoir)(cap, 50 + 4 * r + k, dev)
            m.store.copy_(torch.randint(0, 1 << 30, m.store.shape, generator=g, dtype=torch.int32))
            m.total.fill_([0, 40, cap - 5, 5 * cap][(r + k) % 4])  # empty, partly filled, nearly full, wrapped
            m.sample_calls = 3 * r + k
            mems.append(m)
    reqs = (SampleReq * len(mems))()
    outs = []
    for q, m in zip(reqs, mems):
        q.d_mem, q.d_total, q.cap, q.seed, q.call_idx, q.is_ring = m.store.data_ptr(), m.total.data_ptr(), m.capacity, \
            m.seed, m.sample_calls, int(m.is_ring)
        out = torch.full((b * (65 if m.is_ring else 33),), float("nan"), dtype=torch.float32, device=dev)
        q.d_out = out.data_ptr()
        outs.append(out)
    assert len(mems) > 8 and len(mems) <= MAX_SAMPLE_REQS
    idx = torch.empty((len(mems), b), dtype=torch.int64, device=dev)
    cnt = torch.empty(len(mems), dtype=torch.int32, device=dev)
    check(nb.lib().nfsp_sample_minibatches(reqs, len(mems), b, _ptr(idx), _ptr(cnt), _stream(dev)))
    for k, m in enumerate(mems):
        if m.is_ring:
            s, a, r_, s2, t, i, n = m.sample(b)
            dense = torch.cat([s.reshape(-1), a.reshape(-1), r_, s2.reshape(-1), t])
        else:
            s, a, i, n = m.sample(b)
            dense = torch.cat([s.reshape(-1), a.reshape(-1)])
        assert torch.equal(idx[k], i), k
        assert int(cnt[k].item()) == int(n.item()), k
        assert torch.equal(outs[k].view(torch.int32), dense.view(torch.int32)), k  # bit patterns: random words may be NaNs
