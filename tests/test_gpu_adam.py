"""-m gpu: the learner's Adam (Learner(optimizer="adam")) on every path, against the float64 Adam reference
(tests/adam_reference.py) and against itself across paths.

Tolerances.  The kernels are fp32 and the reference float64.  The gradients agree to fp32 rounding (test_gpu_learner_fit);
Adam then divides each first moment by the root of the second, so an element whose gradient is small compared with the
terms it is summed from keeps a relative error far above fp32's: a gradient of 1e-8 that is really 0 still moves its
weight by lr * 1e-8 / (1e-8 + 3.2e-6) at the first step.  Where the gradient is large the step is ~lr whatever its
error.  So the weights are held to a tolerance in units of the learning rate per step (W_TOL_LR * lr * steps; relative
for the few weights above 1 in magnitude),
the moments to fp32 rounding of their own size plus the error the gradient carries into them.  The learning rates are
Adam-sized (~1e-3), and each case's seed keeps the reference's relu gates >= MARGIN from their kinks over the whole
trajectory (a flip there moves a gradient by ~1e-3): fp32 evaluates a pre-activation of up to 31 terms of magnitude
<= 1 to within ~2e-6, so MARGIN = 1e-5 leaves no branch to chance."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import adam_reference as ar  # noqa: E402
from oracle import learner_oracle as lo  # noqa: E402
from test_gpu_learner_fit import GAMMA, SLOTS, DeviceCase, _slot_words, f32  # noqa: E402

MARGIN = 1e-5
LR_SCALE = 0.05      # fit_case's rates (0.01 .. 0.05) scaled to Adam's usual 5e-4 .. 2.5e-3
W_TOL_LR = 1e-3      # weights: |w - w_ref| <= W_TOL_LR * lr * steps of the net
M_RTOL, V_RTOL = 1e-4, 1e-4


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


class DeviceAdam:
    """Adam's state of one run on the device and the nfsp_adam_state that points at it."""

    def __init__(self, dev, m=None, v=None, t=(0, 0, 0, 0)):
        from nfsp_b200 import _lib

        z = np.zeros((4, lo.NET_PARAMS))
        self.m = torch.tensor(z if m is None else m, dtype=torch.float32, device=dev)
        self.v = torch.tensor(z if v is None else v, dtype=torch.float32, device=dev)
        self.s = _lib.AdamState(self.m.data_ptr(), self.v.data_ptr(), (C.c_int64 * 4)(*t))


def _fit(nb, d, a, geometry, lr, mask=0xF, tb=0, ott=0, w_in=None, w_out=None):
    from nfsp_b200._lib import check
    from nfsp_b200.batched import _ptr, _stream

    w_out = d.w.clone() if w_out is None else w_out
    check(nb.lib().nfsp_learner_fit_adam(C.byref(d.io(mask, tb, ott, w_in=w_in)), *geometry, (C.c_float * 4)(*lr),
                                         _ptr(w_out), C.byref(a.s), _stream(d.dev)))
    torch.cuda.synchronize()
    return w_out


def _compare(tag, w, m, v, ref, lr, steps, mask=0xF):
    """Weights and moments against the reference state (w, m, v); returns the largest weight error in units of lr."""
    w_ref, m_ref, v_ref = ref
    w, m, v = (x.cpu().numpy().astype(np.float64) for x in (w, m, v))
    worst = 0.0
    for k in range(4):
        if not (mask >> k) & 1:
            continue
        # relative where |w| > 1: the wide-logit net's output biases near +-64 keep only 2^-18 of absolute precision
        ew = (np.abs(w[k] - w_ref[k]) / np.maximum(np.abs(w_ref[k]), 1.0)).max() / (lr[k] * steps[k])
        em = np.abs(m[k] - m_ref[k]) - M_RTOL * np.abs(m_ref[k]).max()
        ev = np.abs(v[k] - v_ref[k]) - V_RTOL * np.abs(v_ref[k]).max()
        print("%s net %d: max |w - w_ref| = %.3e lr/step; max |m - m_ref| = %.2e (max |m| %.2e); max |v - v_ref| = %.2e "
              "(max |v| %.2e)" % (tag, k, ew, np.abs(m[k] - m_ref[k]).max(), np.abs(m_ref[k]).max(),
                                  np.abs(v[k] - v_ref[k]).max(), np.abs(v_ref[k]).max()))
        assert ew <= W_TOL_LR, (tag, k, ew)
        assert em.max() <= 0, (tag, k)
        assert ev.max() <= 0, (tag, k)
        worst = max(worst, ew)
    return worst


# (minibatch, fit_batch, epochs), terminal_bootstraps, others_to_target, seed (gate margin >= MARGIN over two fits)
CASES = [
    ((128, 32, 2), 0, 0, 1),   # production: the row-parallel kernel, all four flag combinations
    ((128, 32, 2), 0, 1, 8),
    ((128, 32, 2), 1, 0, 11),
    ((128, 32, 2), 1, 1, 1),
    ((256, 65, 2), 0, 1, 77),  # the register kernel with prefetched rows
    ((256, 65, 2), 1, 0, 29),
    ((320, 80, 1), 1, 1, 22),  # the register kernel reading its rows through the indices
]


@pytest.mark.parametrize("geometry,tb,ott,seed", CASES, ids=["%d-%d-%d-tb%d-ott%d" % (g + (t, o)) for g, t, o, _ in CASES])
def test_adam_fit_matches_float64_reference_over_two_chained_fits(nb, geometry, tb, ott, seed):
    """Two fits in a row: the second starts from the first's weights, moments and step counts (t0 = 8 or 4)."""
    c = lo.fit_case(seed, geometry[0])
    lr = c["lr"] * LR_SCALE
    d = DeviceCase(nb, c)
    a = DeviceAdam(d.dev)
    w, m, v, t = c["w"], None, None, (0, 0, 0, 0)
    steps = geometry[2] * -(-geometry[0] // geometry[1])
    for fit in range(2):
        w, m, v, t, stats, margin = ar.fit(w, c["w_target"], c["rl"], c["sl"], *geometry, f32(lr), f32(GAMMA), m=m, v=v,
                                           t=t, terminal_bootstraps=bool(tb), others_to_target=bool(ott))
        assert margin >= MARGIN, "the data sits on a relu kink (gate margin %.2e): choose another seed" % margin
        _fit(nb, d, a, geometry, lr, tb=tb, ott=ott, w_out=d.w)
        a.s.t0[:] = t    # the host advances t
        _compare("fit %d %s tb=%d ott=%d" % (fit, geometry, tb, ott), d.w, a.m, a.v, (w, m, v), lr, [(fit + 1) * steps] * 4)
        if fit == 0:
            got = d.flat[d.GRAD:].cpu().numpy().astype(np.float64)
            assert np.allclose(got[4:], stats[4:], rtol=1e-4, atol=1e-6)   # the statistics are the SGD fit's
    assert t == [2 * steps] * 4


@pytest.mark.parametrize("geometry,seed", [((128, 32, 2), 0), ((320, 80, 1), 1)], ids=["rows-kernel", "register-kernel"])
@pytest.mark.parametrize("mask", [0b0101, 0b1010, 0b0001, 0b1110])
@pytest.mark.parametrize("aliased", [False, True], ids=["w_out-separate", "w_out-aliased"])
def test_adam_fit_net_mask(nb, geometry, seed, mask, aliased):
    """A net outside net_mask keeps its weights, m and v bit for bit (under Adam a zero gradient would still move them);
    the others train as in the reference, from non-zero moments and step counts."""
    c = lo.fit_case(seed, geometry[0])
    lr = c["lr"] * LR_SCALE
    rng = np.random.RandomState(7)
    m0, v0, t0 = rng.randn(4, lo.NET_PARAMS) * 1e-3, rng.rand(4, lo.NET_PARAMS) * 1e-6, (3, 5, 7, 9)
    m0, v0 = f32(m0), f32(v0)
    d = DeviceCase(nb, c)
    a = DeviceAdam(d.dev, m0, v0, t0)
    w_in, m_in, v_in = d.w.clone(), a.m.clone(), a.v.clone()
    w_out = d.w if aliased else torch.full_like(d.w, float("nan"))
    _fit(nb, d, a, geometry, lr, mask=mask, w_out=w_out)
    for k in range(4):
        if not (mask >> k) & 1:
            assert torch.equal(w_out[k], w_in[k]) and torch.equal(a.m[k], m_in[k]) and torch.equal(a.v[k], v_in[k]), k
    w, m, v, t, _, margin = ar.fit(c["w"], c["w_target"], c["rl"], c["sl"], *geometry, f32(lr), f32(GAMMA), m=m0, v=v0,
                                   t=t0, net_mask=mask)
    assert margin >= MARGIN
    steps = geometry[2] * -(-geometry[0] // geometry[1])
    assert t == [t0[k] + (steps if (mask >> k) & 1 else 0) for k in range(4)]
    _compare("mask %s %s" % (bin(mask), geometry), w_out, a.m, a.v, (w, m, v), lr, [steps] * 4, mask)


def test_adam_apply_is_one_step_of_the_fit(nb):
    """nfsp_learner_grads + nfsp_adam_apply, step by step, equals the one-launch Adam fit on the same rows (the register
    and row kernels compute the same mean gradients; only fused multiply-adds may differ), and a net outside the mask
    stays as it was."""
    from nfsp_b200._lib import check
    from nfsp_b200.batched import _ptr, _stream

    geometry = (128, 32, 2)
    c = lo.fit_case(CASES[0][3], 128)
    lr = c["lr"] * LR_SCALE
    d1, d2 = DeviceCase(nb, c), DeviceCase(nb, c)
    a1, a2 = DeviceAdam(d1.dev, t=(2, 2, 2, 2)), DeviceAdam(d2.dev, t=(2, 2, 2, 2))
    mask = 0b1011
    _fit(nb, d1, a1, geometry, lr, mask=mask, w_out=d1.w)
    lr_c = (C.c_float * 4)(*lr)
    for _ in range(2):
        for row0 in range(0, 128, 32):
            check(nb.lib().nfsp_learner_grads(C.byref(d2.io(mask, row0=row0, rows=32)), _stream(d2.dev)))
            check(nb.lib().nfsp_adam_apply(_ptr(d2.w), _ptr(d2.flat), C.byref(lr_c), 1.0, mask, C.byref(a2.s), _stream(d2.dev)))
            for k in range(4):
                if (mask >> k) & 1:
                    a2.s.t0[k] += 1
    torch.cuda.synchronize()
    assert torch.equal(d2.w[2], d1.w[2]) and not a2.m[2].any() and not a2.v[2].any()
    dw = (d1.w - d2.w).abs().max().item()
    print("one launch vs step by step: max |dw| = %.3e" % dw)
    assert dw <= W_TOL_LR * float(lr.max()) * 8
    assert torch.allclose(a1.m, a2.m, rtol=M_RTOL, atol=1e-7) and torch.allclose(a1.v, a2.v, rtol=V_RTOL, atol=1e-10)


UPDATE_SEED = 5    # gate margin >= MARGIN over the rows SelfPlay(seed=5)'s memories draw in the first three updates


def test_learner_update_with_adam_matches_the_chained_reference(nb):
    """Learner(optimizer="adam").update() three times on crafted memories (as test_gpu_learner_fit does for SGD), against
    the reference chained over the rows each update sampled, with the learning rates and target nets each update had
    (the BR rates decay between updates; the first update copies the BR nets into the targets)."""
    from nfsp_b200.learner import Learner

    c = lo.fit_case(UPDATE_SEED, 128)
    sp = nb.SelfPlay(64, seed=5, rl_capacity=SLOTS, sl_capacity=SLOTS)
    sp.set_weights(torch.tensor(c["w"], dtype=torch.float32, device=sp.device))
    rng = np.random.RandomState(99)
    total = 3 * SLOTS + 17
    head = total % SLOTS
    for p in range(2):
        rl, sl = _slot_words(c, p, rng)
        sp.rl[p].store.copy_(torch.roll(rl, head, 0))
        sp.sl[p].store.copy_(sl)
        sp.rl[p].total.fill_(total)
        sp.sl[p].total.fill_(total)
    L = Learner(sp, gamma=GAMMA, optimizer="adam", lr_br=0.002, lr_ar=0.001)
    L.target = torch.tensor(c["w_target"], dtype=torch.float32, device=sp.device)
    w, m, v, t = c["w"], None, None, (0, 0, 0, 0)
    for u in range(3):
        lr = [L.lr_ar, L.lr_br[0], L.lr_ar, L.lr_br[1]]
        wt = L.target.cpu().numpy().astype(np.float64)
        assert L.update()["trained"] == 0xF
        slots = L._pos.cpu().numpy()
        rl = [c["rl_slots"][p][(slots[p] - head) % SLOTS] for p in range(2)]
        sl = [c["sl_slots"][p][slots[2 + p]] for p in range(2)]
        w, m, v, t, _, margin = ar.fit(w, wt, rl, sl, 128, 32, 2, f32(lr), f32(GAMMA), m=m, v=v, t=t)
        assert margin >= MARGIN
        assert L.adam_t == t == [8 * (u + 1)] * 4
        _compare("update %d" % u, sp.weights, L.adam_m, L.adam_v, (w, m, v), np.array(lr), [8 * (u + 1)] * 4)
    assert L.lr_br[0] < 0.002


def _filled(nb, n=4096, seed=1234):
    from test_gpu_learner import _filled_selfplay

    return _filled_selfplay(nb, n=n)


@pytest.mark.parametrize("minibatch,fit_batch", [(128, 32), (320, 80)])
def test_adam_one_launch_equals_the_step_by_step_path(nb, minibatch, fit_batch):
    """Learner(fused=True) (one Adam fit launch) against Learner(fused=False) (grads + nfsp_adam_apply per step) over three
    updates on the same memories: the same statistics, step counts, and weights and moments to fp32 rounding."""
    from nfsp_b200.learner import Learner

    a, b = _filled(nb), _filled(nb)
    La, Lb = (Learner(x, minibatch=minibatch, fit_batch=fit_batch, fused=f, optimizer="adam", lr_br=0.002, lr_ar=0.001)
              for x, f in ((a, True), (b, False)))
    for k in range(3):
        ra, rb = La.update(), Lb.update()
        assert ra["trained"] == rb["trained"] == 0xF
        assert np.allclose(ra["loss"], rb["loss"], rtol=1e-4, atol=1e-5)
        assert La.adam_t == Lb.adam_t
        d = (a.weights - b.weights).abs().max().item()
        print("update %d: max |dw| = %.3e" % (k, d))
        assert d <= W_TOL_LR * 0.002 * La.adam_t[0], (k, d)
        assert torch.allclose(La.adam_m, Lb.adam_m, rtol=M_RTOL, atol=1e-6)
        assert torch.allclose(La.adam_v, Lb.adam_v, rtol=V_RTOL, atol=1e-9)


def test_adam_peer_exchange_two_ranks_on_one_gpu(nb):
    """nfsp_learner_fit_peers_adam with two ranks played by two kernels side by side on one GPU: weights, m and v
    bit-identical on both ranks, and equal to the single-GPU Adam step on the mean gradient (nfsp_learner_grads of both
    ranks summed on the device, nfsp_adam_apply with scale 1/2) to fp32 rounding."""
    from nfsp_b200 import _lib
    from nfsp_b200._lib import check
    from nfsp_b200.batched import _ptr, _stream
    from nfsp_b200.learner import Learner

    sps = [_filled(nb), _filled(nb, n=2048)]
    w0 = sps[0].weights.clone()
    sps[1].set_weights(w0.clone())
    Ls = [Learner(sp, fused=False, optimizer="adam") for sp in sps]
    idx = [L._sample_positions() for L in Ls]
    lr = (C.c_float * 4)(0.001, 0.002, 0.001, 0.002)
    refs = [DeviceAdam(sps[0].device) for _ in range(2)]
    for _ in range(2):
        for row0 in range(0, 128, 32):
            for L, (irl, isl) in zip(Ls, idx):
                check(nb.lib().nfsp_learner_grads(C.byref(L._io(irl, isl, row0, 32, 0xF)), _stream(L.device)))
            total = Ls[0].flat + Ls[1].flat
            for L, ref in zip(Ls, refs):   # each rank applies the same mean gradient to its own replica
                check(nb.lib().nfsp_adam_apply(_ptr(L.sp.weights), _ptr(total), C.byref(lr), 0.5, 0xF, C.byref(ref.s),
                                               _stream(L.device)))
                for k in range(4):
                    ref.s.t0[k] += 1
    w_ref, ref = Ls[0].sp.weights.clone(), refs[0]
    assert torch.equal(w_ref, Ls[1].sp.weights)
    dev = sps[0].device
    bufs = [torch.zeros(_lib.PEER_BUF_FLOATS, dtype=torch.float32, device=dev) for _ in range(2)]
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    streams = [torch.cuda.Stream(dev) for _ in range(2)]
    states = [DeviceAdam(dev) for _ in range(2)]
    for L in Ls:
        L.sp.weights.copy_(w0)
    torch.cuda.synchronize()
    for r, (L, (irl, isl)) in enumerate(zip(Ls, idx)):
        p = _lib.Peers()
        p.world, p.rank, p.epoch0, p.d_err = 2, r, 0, err.data_ptr()
        for q in range(2):
            p.d_buf[q] = bufs[q].data_ptr()
        with torch.cuda.stream(streams[r]):
            check(nb.lib().nfsp_learner_fit_peers_adam(C.byref(L._io(irl, isl, 0, 128, 0xF)), 128, 32, 2, lr,
                                                       _ptr(L.sp.weights), C.byref(p), C.byref(states[r].s), _stream(dev)))
    torch.cuda.synchronize()
    assert int(err.item()) == 0, "a rank timed out waiting for its peer"
    assert torch.equal(Ls[0].sp.weights, Ls[1].sp.weights)
    assert torch.equal(states[0].m, states[1].m) and torch.equal(states[0].v, states[1].v)
    d = (Ls[0].sp.weights - w_ref).abs().max().item()
    print("peers vs mean-gradient Adam: max |dw| = %.3e" % d)
    assert d <= W_TOL_LR * 0.002 * 8
    assert torch.allclose(states[0].m, ref.m, rtol=M_RTOL, atol=1e-6)
    assert torch.allclose(states[0].v, ref.v, rtol=V_RTOL, atol=1e-9)
    assert not torch.equal(w0, w_ref)


def test_adam_runs_train_bit_for_bit_like_standalone_runs(nb):
    """Three Adam runs with their own seeds, eta, epsilons and learning rates, batched, against the same runs driven alone:
    weights, memories, schedules and every run's moments and step counts, after every iteration."""
    from nfsp_b200.learner import Learner
    from nfsp_b200.runs import RunBatch
    from test_gpu_runs import _assert_same_run

    configs = [(1234, 0.1, [0.06, 0.06], 0.002, 0.001), (77, 0.3, [0.2, 0.05], 0.0005, 0.002),
               (4242, 0.05, [0.1, 0.15], 0.001, 0.0005)]
    kw = dict(rl_capacity=1 << 16, sl_capacity=1 << 16, max_steps_per_call=8, deterministic=True)

    def run(s, e, ep, lb, la):
        sp = nb.SelfPlay(4096, seed=s, eta=e, epsilon=list(ep), **kw)
        return sp, Learner(sp, lr_br=lb, lr_ar=la, optimizer="adam")

    solo = [run(*cf) for cf in configs]
    runs = [run(*cf) for cf in configs]
    rb = RunBatch([sp for sp, _ in runs], [ln for _, ln in runs])
    for it in range(8):
        for sp, ln in solo:
            sp.rollout(8)
            if it >= 2:
                ln.update(sync=False)
        rb.rollout(8)
        if it >= 2:
            rb.update(sync=False)
        for r in range(3):
            _assert_same_run(solo[r][0], runs[r][0], solo[r][1], runs[r][1], "iteration %d run %d" % (it, r))
            assert torch.equal(solo[r][1].adam_m, runs[r][1].adam_m) and torch.equal(solo[r][1].adam_v, runs[r][1].adam_v)
            assert solo[r][1].adam_t == runs[r][1].adam_t
    assert all(ln.adam_t[0] > 0 for _, ln in runs)
    assert not torch.equal(runs[0][1].adam_m, runs[1][1].adam_m)
    # a batch refuses runs whose learners differ in optimizer
    sp = nb.SelfPlay(4096, seed=9, **kw)
    with pytest.raises(ValueError, match="optimizer"):
        RunBatch([runs[0][0], sp], [runs[0][1], Learner(sp)])


def test_adam_pipelined_trainer_equals_the_sequential_loop_with_one_update_of_lag(nb):
    """test_gpu_train's lag check under Adam: the moments are updated in place on the learner's stream beside the next
    rollout, and the result is bit-identical to the sequential loop acting one update behind."""
    from nfsp_b200.learner import Learner, PipelinedTrainer

    def make():
        sp = nb.SelfPlay(4096, seed=21, eta=0.3, epsilon=0.2, rl_capacity=1 << 15, sl_capacity=1 << 15, max_steps_per_call=8,
                         deterministic=True)
        for _ in range(3):
            sp.rollout(8)
        return sp

    K = 7
    a, b = make(), make()
    La, Lb = (Learner(x, cfg=nb.load_config(None), optimizer="adam") for x in (a, b))
    chain = a.weights.clone()
    hist = [chain.clone()]
    for j in range(K):
        a.set_weights(hist[j - 1 if j >= 1 else 0].clone())
        a.rollout(8)
        a.set_weights(chain)
        assert La.update(sync=False)["trained"] == 0xF
        hist.append(chain.clone())
    T = PipelinedTrainer(b, Lb)
    for j in range(K):
        assert T.step(8)["trained"] == 0xF
    final = T.finish()
    torch.cuda.synchronize()
    assert torch.equal(final, hist[K]) and not torch.equal(hist[K], hist[0])
    assert torch.equal(La.adam_m, Lb.adam_m) and torch.equal(La.adam_v, Lb.adam_v) and La.adam_t == Lb.adam_t == [8 * K] * 4
    assert torch.equal(a.env.state_words(), b.env.state_words())


def test_adam_checkpoint_resume_is_bit_for_bit(nb, tmp_path):
    """Saved after 5 iterations and resumed: the resumed Adam run equals the one that never stopped, moments and step
    counts included; an SGD learner refuses the state, naming the optimizer."""
    from nfsp_b200 import checkpoint
    from nfsp_b200.learner import Learner
    from test_gpu_checkpoint import _assert_same, _iterate, _make, _resumed

    def make():
        return _make(nb, rl_capacity=1 << 14, sl_capacity=1 << 13, max_steps_per_call=8, deterministic=True,
                     lr_br=0.002, lr_ar=0.001, learner=dict(optimizer="adam"))

    def same(x, lx, y, ly, tag):
        _assert_same(x, y, lx, ly, tag)
        assert torch.equal(lx.adam_m, ly.adam_m) and torch.equal(lx.adam_v, ly.adam_v) and lx.adam_t == ly.adam_t, tag

    a, la = make()
    b, lb = make()
    for it in range(5):
        assert _iterate(a, la, it) == _iterate(b, lb, it)
    c, lc = _resumed(nb, tmp_path, b, lb, 5, make)
    same(a, la, c, lc, "resumed")
    for it in range(5, 9):
        assert _iterate(a, la, it) == _iterate(c, lc, it), it
        same(a, la, c, lc, "iteration %d" % it)
    assert la.adam_t[1] > 0
    d = str(tmp_path / "ck2")
    checkpoint.save(d, 9, selfplay=a, learner=la)
    sp = nb.SelfPlay(4096, seed=1234, eta=0.3, epsilon=0.2, rl_capacity=1 << 14, sl_capacity=1 << 13, max_steps_per_call=8,
                     deterministic=True)
    with pytest.raises(ValueError, match="optimizer"):
        checkpoint.load(d, selfplay=sp, learner=Learner(sp))


@pytest.mark.parametrize("runs", [1, 3], ids=["sequential", "runs-3"])
def test_cli_adam_checkpoint_and_resume(nb, tmp_path, runs):
    """main.py --optimizer adam --checkpoint DIR, then --resume DIR with a larger --episodes: the resumed rows are the
    rows of the run that never stopped, and they say "optimizer": "adam".  A resume without --optimizer adam is refused."""
    from test_gpu_checkpoint import _cli, _strip

    extra = ["--optimizer", "adam"] + (["--runs", str(runs)] if runs > 1 else [])
    ref = _strip(_cli(tmp_path, extra + ["--episodes", "250000"]))
    assert len(ref) >= 5 and all(r["optimizer"] == "adam" for r in ref)
    stop = ref[len(ref) // 2]
    e1 = stop["hands"] if runs == 1 else min(r["hands"] for r in stop["runs"])
    d = str(tmp_path / "ck")
    first = _strip(_cli(tmp_path, extra + ["--episodes", str(e1), "--checkpoint", d, "--checkpoint-every", "5"]))
    assert first == ref[:len(ref) // 2 + 1]
    with pytest.raises(ValueError, match="optimizer"):
        _cli(tmp_path, extra[2:] + ["--episodes", "250000", "--resume", d])
    rest = _strip(_cli(tmp_path, extra + ["--episodes", "250000", "--resume", d]))
    assert rest == ref[len(ref) // 2 + 1:] and rest


def test_adam_sweep_runs_equal_their_standalone_runs(nb, tmp_path):
    """A one-rank --optimizer adam sweep over two Adam-sized BR learning rates: each run's state (moments and step counts
    included) and rows equal main.py --optimizer adam trained alone with the run's values."""
    import json

    import test_gpu_sweep as sw

    d = str(tmp_path / "ck")
    rows = sw._cli(["--optimizer", "adam", "--sweep", "LearningRateBR=0.001,0.0001", "--config",
                    sw._config(tmp_path / "config.ini"), "--episodes", str(sw.EPISODES), "--checkpoint", d])
    runs = [r for r in rows if r["kind"] == "run"]
    assert runs and all(r["optimizer"] == "adam" for r in rows)
    last = max(r["calls"] for r in rows)
    saved = torch.load(os.path.join(d, "rank0-of-1.pt"), weights_only=True)
    for i, state in enumerate(saved["runs"]["runs"]):
        mine = [r for r in runs if r["run"] == i]
        hp, seed = mine[0]["hparams"], mine[0]["seed"]
        cfg = sw._config(tmp_path / ("run%d.ini" % i), "".join("%s = %r\n" % kv for kv in hp.items()) +
                         "[Utils]\nSeed = %d\n" % seed)
        solo_dir = str(tmp_path / ("solo%d" % i))
        solo = sw._cli(["--optimizer", "adam", "--config", cfg, "--episodes", str(mine[-1]["hands"]), "--checkpoint", solo_dir])
        assert len(solo) == len(mine) and solo[-1]["calls"] == last, i
        for a, b in zip(sw._strip(solo), sw._strip(mine)):
            assert a == {k: b[k] for k in a}, (i, a["calls"])
        alone = torch.load(os.path.join(solo_dir, "rank0-of-1.pt"), weights_only=True)
        sw._same_state(state["selfplay"], alone["selfplay"], "run %d selfplay" % i)
        sw._same_state(state["learner"], alone["learner"], "run %d learner" % i)
        assert alone["learner"]["shape"]["optimizer"] == "adam" and max(alone["learner"]["adam_t"]) > 0
    json.dumps(rows)


def test_adam_peer_exchange_on_real_gpus_when_there_are_two():
    """tests/mgpu_adam_check.py under torchrun: Adam weights and moments identical on both ranks; needs >= 2 GPUs."""
    import subprocess

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29537", os.path.join(root, "tests", "mgpu_adam_check.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "mgpu adam check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
