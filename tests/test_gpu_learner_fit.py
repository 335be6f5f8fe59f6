"""-m gpu: the learner's one-launch fit against the float64 reference of the whole fit (oracle/learner_oracle.fit).

The memories are built by hand (oracle/learner_oracle.fit_case), not by a rollout, so that every edge is there on
purpose: observations 0 and 0x3FFFFFFF, rewards of both Huber branches, terminal flags 0 and 1, unnormalised and all-zero
SL targets, an average-policy net whose logits span more than 100, sampled indices that repeat and run out of order, and
random words in the unused half of every 32-byte reservoir slot (a wrong slot stride reads garbage).

The kernels are fp32 and the reference is float64: where a relu pre-activation sits within rounding of zero, the two can
take different branches, and one such flip moves a W1 gradient by ~1e-3.  The nets are dyadic (lo.dyadic_net), so the
first forward pass is exact in fp32 and every pre-activation starts >= 1/64 from zero, and each case's seed was chosen so
that the reference's gate margin stays >= 1e-4 over the whole trajectory; a precondition asserts it.  Then the weights
must agree within 2e-6 (relative for the few weights above 1 in magnitude) and the first step's statistics within
1e-4 relative."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import learner_oracle as lo  # noqa: E402
from oracle import orc  # noqa: E402

SLOTS = 256          # records per hand-built memory
GAMMA = 0.95
MARGIN = 1e-4        # the smallest gate margin of the reference trajectory a comparison accepts
W_TOL = 2e-6         # fp32 rounding over up to 64 updates: absolute for weights of magnitude <= 1, relative above
                     # (the wide-logit net's output biases near +-64 keep only 2^-17 of absolute precision)
STATS_RTOL = 1e-4


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def f32(x):
    """What the kernel sees of a host float: the reference runs on the same values."""
    return np.float32(x).astype(np.float64)


def _slot_words(c, p, rng):
    """Player p's records as the memories store them: a ring slot is the 16-byte record, a reservoir slot the record and
    16 bytes the learner must never read (here random words)."""
    rl = np.ascontiguousarray(c["rl_slots"][p]).view(np.int32).reshape(SLOTS, 4)
    sl = np.ascontiguousarray(c["sl_slots"][p]).view(np.int32).reshape(SLOTS, 4)
    tail = rng.randint(-2 ** 31, 2 ** 31, (SLOTS, 4), dtype=np.int64).astype(np.int32)
    return torch.from_numpy(rl.copy()), torch.from_numpy(np.concatenate([sl, tail], 1))


class DeviceCase:
    """One fit_case on the device: the memories, the sampled indices, weights, target nets and the learner's flat
    gradient + statistics buffer, and the LearnerIO that points at them."""

    def __init__(self, nb, c, w=None, w_target=None):
        from nfsp_b200._lib import LearnerIO
        from nfsp_b200.batched import DeviceReservoir, DeviceRing
        from nfsp_b200.learner import GRAD, N_STATS

        self.dev = torch.device("cuda", torch.cuda.current_device())
        rng = np.random.RandomState(99)
        self.rings = [DeviceRing(SLOTS, 11 + p, self.dev) for p in range(2)]
        self.res = [DeviceReservoir(SLOTS, 13 + p, self.dev) for p in range(2)]
        for p in range(2):
            rl, sl = _slot_words(c, p, rng)
            self.rings[p].store.copy_(rl)
            self.res[p].store.copy_(sl)
        self.idx_rl = [torch.from_numpy(i).to(self.dev) for i in c["idx_rl"]]
        self.idx_sl = [torch.from_numpy(i).to(self.dev) for i in c["idx_sl"]]
        self.w = torch.tensor(c["w"] if w is None else w, dtype=torch.float32, device=self.dev)
        self.wt = torch.tensor(c["w_target"] if w_target is None else w_target, dtype=torch.float32, device=self.dev)
        self.flat = torch.zeros(GRAD + N_STATS, dtype=torch.float32, device=self.dev)
        self.GRAD = GRAD
        self.LearnerIO = LearnerIO

    def io(self, mask=0xF, tb=0, ott=0, row0=0, rows=0, w_in=None):
        io = self.LearnerIO()
        io.d_weights, io.d_target_weights = (self.w if w_in is None else w_in).data_ptr(), self.wt.data_ptr()
        for p in range(2):
            io.d_rl[p], io.d_rl_idx[p] = self.rings[p].store.data_ptr(), self.idx_rl[p].data_ptr()
            io.d_sl[p], io.d_sl_idx[p] = self.res[p].store.data_ptr(), self.idx_sl[p].data_ptr()
        io.row0, io.rows, io.gamma, io.net_mask = row0, rows, GAMMA, mask
        io.terminal_bootstraps, io.others_to_target = tb, ott
        io.d_grad, io.d_stats = self.flat.data_ptr(), self.flat[self.GRAD:].data_ptr()
        return io

    def fit(self, nb, geometry, lr, mask=0xF, tb=0, ott=0, w_out=None):
        from nfsp_b200._lib import check
        from nfsp_b200.batched import _ptr, _stream

        w_out = self.w.clone() if w_out is None else w_out
        lr_c = (C.c_float * 4)(*lr)
        check(nb.lib().nfsp_learner_fit(C.byref(self.io(mask, tb, ott)), *geometry, lr_c, _ptr(w_out), _stream(self.dev)))
        torch.cuda.synchronize()
        return w_out, self.flat[self.GRAD:].cpu().numpy().astype(np.float64)


def _reference(c, geometry, mask=0xF, tb=0, ott=0, rl=None, sl=None, lr=None, peers=()):
    lr = c["lr"] if lr is None else lr
    return lo.fit(c["w"], c["w_target"], c["rl"] if rl is None else rl, c["sl"] if sl is None else sl, *geometry,
                  f32(lr), f32(GAMMA), mask, bool(tb), bool(ott), peers)


def _compare(tag, w_got, stats_got, ref, w_in, mask=0xF):
    """The kernel's weights and first-step statistics against the reference; returns the largest weight deviation."""
    w_ref, stats_ref, margin, seen = ref
    assert margin >= MARGIN, "%s: the data sits on a relu kink (gate margin %.2e): choose another seed" % (tag, margin)
    w_got = w_got.cpu().numpy().astype(np.float64)
    err = np.abs(w_got - w_ref)
    dev = (err / np.maximum(np.abs(w_ref), 1.0)).max()
    print("%s: max |w - w_ref| = %.3e where |w| <= 1, %.3e relative where |w| > 1; gate margin %.2e"
          % (tag, err[np.abs(w_ref) <= 1].max(), dev if (np.abs(w_ref) > 1).any() else 0.0, margin))
    assert dev <= W_TOL, (tag, dev, np.unravel_index(np.argmax(err / np.maximum(np.abs(w_ref), 1.0)), err.shape))
    for k in range(4):
        if (mask >> k) & 1:
            assert np.abs(w_got[k] - w_in[k]).max() >= 1e-3, (tag, k)           # not vacuous: the net trained
            idx = [4 + k] + ([k >> 1, 2 + (k >> 1)] if k & 1 else [])
            assert np.allclose(stats_got[idx], stats_ref[idx], rtol=STATS_RTOL, atol=1e-6), (tag, k, stats_got, stats_ref)
    return dev


# (minibatch, fit_batch, epochs), terminal_bootstraps, others_to_target, seed of the fit_case (gate margin >= 1e-4)
CASES = [
    ((128, 32, 2), 0, 0, 86),   # production: the row-parallel kernel, all four flag combinations
    ((128, 32, 2), 0, 1, 86),
    ((128, 32, 2), 1, 0, 86),
    ((128, 32, 2), 1, 1, 86),
    ((256, 64, 2), 1, 1, 26),  # the row-parallel kernel at both shared-memory limits; two ballot chunks in phase 2
    ((100, 24, 2), 0, 0, 0),   # ragged last slice of 4 rows
    ((129, 32, 2), 1, 0, 15),   # last slice of 1 row
    ((256, 65, 2), 0, 0, 30),  # the register kernel with prefetched rows, all four flag combinations
    ((256, 65, 2), 0, 1, 30),
    ((256, 65, 2), 1, 0, 30),
    ((256, 65, 2), 1, 1, 30),
    ((100, 128, 1), 0, 1, 10),  # the register kernel with prefetched rows, one ragged step
    ((320, 80, 2), 1, 0, 127),   # the register kernel reading its rows through the indices
    ((64, 1, 1), 0, 0, 63),     # exactly NFSP_MAX_FIT_STEPS steps of one row
]


@pytest.mark.parametrize("geometry,tb,ott,seed", CASES, ids=["%d-%d-%d-tb%d-ott%d" % (g + (t, o)) for g, t, o, _ in CASES])
def test_fit_matches_float64_sgd(nb, geometry, tb, ott, seed):
    c = lo.fit_case(seed, geometry[0])
    d = DeviceCase(nb, c)
    w_got, stats = d.fit(nb, geometry, c["lr"], tb=tb, ott=ott)
    ref = _reference(c, geometry, tb=tb, ott=ott)
    _compare("fit %s tb=%d ott=%d seed=%d" % (geometry, tb, ott, seed), w_got, stats, ref, c["w"])
    _, _, _, seen = ref
    assert seen["huber_linear"] > 0 and seen["huber_quadratic"] > 0 and seen["log_clamped"] > 0


@pytest.mark.parametrize("geometry,seed", [((128, 32, 2), 86), ((320, 80, 2), 127)], ids=["rows-kernel", "register-kernel"])
@pytest.mark.parametrize("mask", [0b0101, 0b1010, 0b0001])
@pytest.mark.parametrize("aliased", [False, True], ids=["w_out-separate", "w_out-aliased"])
def test_fit_net_mask(nb, geometry, seed, mask, aliased):
    """Nets outside net_mask: with a separate output they are copied bit for bit, with the output aliased to the input
    they are left alone; the others train as in the reference."""
    c = lo.fit_case(seed, geometry[0])
    d = DeviceCase(nb, c)
    w_in = d.w.clone()
    w_out = d.w if aliased else torch.full_like(d.w, float("nan"))
    d.fit(nb, geometry, c["lr"], mask=mask, w_out=w_out)
    for k in range(4):
        if not (mask >> k) & 1:
            assert torch.equal(w_out[k], w_in[k]), k
    _compare("mask %s %s aliased=%d" % (bin(mask), geometry, aliased), w_out, d.flat[d.GRAD:].cpu().numpy().astype(np.float64),
             _reference(c, geometry, mask=mask), c["w"], mask)


def test_fit_is_deterministic(nb):
    for geometry, seed in (((128, 32, 2), 86), ((320, 80, 2), 127)):
        c = lo.fit_case(seed, geometry[0])
        d = DeviceCase(nb, c)
        w1, s1 = d.fit(nb, geometry, c["lr"], tb=1, ott=1)
        w2, s2 = d.fit(nb, geometry, c["lr"], tb=1, ott=1)
        assert torch.equal(w1, w2) and np.array_equal(s1, s2), geometry


def test_fit_refuses_more_than_max_fit_steps(nb):
    """64 x 1 rows x 2 epochs = 128 SGD steps: an argument error, and w_out is not touched."""
    from nfsp_b200._lib import NfspError

    c = lo.fit_case(63, 64)
    d = DeviceCase(nb, c)
    w_out = torch.full_like(d.w, 7.0)
    with pytest.raises(NfspError, match="more than 64 SGD steps"):
        d.fit(nb, (64, 1, 2), c["lr"], w_out=w_out)
    assert bool((w_out == 7.0).all())


@pytest.mark.parametrize("tb,ott", [(0, 0), (1, 1), (0, 1), (1, 0)])
@pytest.mark.parametrize("row0,rows", [(17, 300), (8, 1)], ids=["300-rows-through-indices", "one-row"])
def test_gradient_kernel_matches_reference(nb, row0, rows, tb, ott):
    """nfsp_learner_grads beyond its prefetch buffer (300 rows are read through the indices) and on a single row."""
    from nfsp_b200._lib import check
    from nfsp_b200.batched import _stream

    c = lo.fit_case(4, 320)
    d = DeviceCase(nb, c)
    check(nb.lib().nfsp_learner_grads(C.byref(d.io(0xF, tb, ott, row0, rows)), _stream(d.dev)))
    flat = d.flat.cpu().numpy().astype(np.float64)
    sel = slice(row0, row0 + rows)
    for p in range(2):
        b = c["rl"][p][sel]
        g, expl, loss = lo.br_grad(c["w"][2 * p + 1], c["w_target"][p], b["s"], b["s2"], b["a"], b["r"], b["t"], f32(GAMMA),
                                   bool(tb), bool(ott))
        got = flat[(2 * p + 1) * 2179:(2 * p + 2) * 2179]
        assert np.abs(got - g).max() < 1e-5 and np.abs(g).max() > 1e-3, (p, np.abs(got - g).max())
        assert np.isclose(flat[d.GRAD + p], expl, rtol=STATS_RTOL) and flat[d.GRAD + 2 + p] == rows
        assert np.isclose(flat[d.GRAD + 4 + 2 * p + 1], loss, rtol=STATS_RTOL, atol=1e-6)
        b = c["sl"][p][sel]
        g, loss = lo.avg_grad(c["w"][2 * p], b["s"], b["a"])
        got = flat[(2 * p) * 2179:(2 * p + 1) * 2179]
        assert np.abs(got - g).max() < 1e-5 and np.abs(g).max() > 1e-3, (p, np.abs(got - g).max())
        assert np.isclose(flat[d.GRAD + 4 + 2 * p], loss, rtol=STATS_RTOL, atol=1e-6)


UPDATE_SEED = 12   # fit_case seed of the Learner.update() test (gate margin >= 1e-4 on the rows SelfPlay(seed=5) samples)


def test_learner_update_trains_each_net_with_its_learning_rate(nb):
    """Learner.update() end to end on crafted memories: the host's learning-rate-to-net mapping, its minibatch slicing
    and the sampled positions, against the reference run on the rows the update sampled and the learning rates it had
    before its decay."""
    from nfsp_b200.learner import GRAD, Learner

    c = lo.fit_case(UPDATE_SEED, 128)
    sp = nb.SelfPlay(64, seed=5, rl_capacity=SLOTS, sl_capacity=SLOTS)
    sp.set_weights(torch.tensor(c["w"], dtype=torch.float32, device=sp.device))
    rng = np.random.RandomState(99)
    for p in range(2):
        rl, sl = _slot_words(c, p, rng)
        sp.rl[p].store.copy_(rl)
        sp.sl[p].store.copy_(sl)
        sp.rl[p].total.fill_(SLOTS)    # full memories: every net trains and every draw lands on a crafted slot
        sp.sl[p].total.fill_(SLOTS)
    L = Learner(sp, gamma=GAMMA)
    L.target = torch.tensor(c["w_target"], dtype=torch.float32, device=sp.device)
    L.lr_ar, L.lr_br = 0.01, [0.05, 0.02]
    lr = [L.lr_ar, L.lr_br[0], L.lr_ar, L.lr_br[1]]
    out = L.update()
    assert out["trained"] == 0xF and L.lr_br[0] < 0.05       # the rates decayed after the fit
    pos = L._pos.cpu().numpy()
    for k, mem in enumerate((sp.rl[0], sp.rl[1], sp.sl[0], sp.sl[1])):   # full ring: deque position == slot
        assert np.array_equal(pos[k], orc.sample_indices(mem.seed, 0, SLOTS, 128)), k
    rl = [c["rl_slots"][p][pos[p]] for p in range(2)]
    sl = [c["sl_slots"][p][pos[2 + p]] for p in range(2)]
    ref = _reference(c, (128, 32, 2), rl=rl, sl=sl, lr=lr)
    _compare("Learner.update", sp.weights, L.flat[GRAD:].cpu().numpy().astype(np.float64), ref, c["w"])


PEER_SEEDS = (116, 1116)   # fit_case seeds of the two ranks' memories (gate margin >= 1e-4)


def test_peer_exchange_fit_matches_float64_sgd_on_the_mean_gradient(nb):
    """nfsp_learner_fit_peers with two ranks played by two kernels side by side on two streams of one GPU (as in
    test_gpu_learner.test_peer_exchange_protocol_two_ranks_on_one_gpu), each on its own memories, against float64 SGD on
    the mean of the two ranks' mean gradients.  The statistics are sums over the ranks."""
    from nfsp_b200 import _lib
    from nfsp_b200._lib import check
    from nfsp_b200.batched import _ptr, _stream

    a, b = (lo.fit_case(s, 128) for s in PEER_SEEDS)
    ranks = [DeviceCase(nb, a), DeviceCase(nb, b, w=a["w"], w_target=a["w_target"])]
    dev = ranks[0].dev
    bufs = [torch.zeros(_lib.PEER_BUF_FLOATS, dtype=torch.float32, device=dev) for _ in range(2)]
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    streams = [torch.cuda.Stream(dev) for _ in range(2)]
    outs = [torch.full_like(r.w, float("nan")) for r in ranks]
    lr = (C.c_float * 4)(*a["lr"])
    torch.cuda.synchronize()
    for r, d in enumerate(ranks):
        p = _lib.Peers()
        p.world, p.rank, p.epoch0, p.d_err = 2, r, 0, err.data_ptr()
        for q in range(2):
            p.d_buf[q] = bufs[q].data_ptr()
        with torch.cuda.stream(streams[r]):
            check(nb.lib().nfsp_learner_fit_peers(C.byref(d.io()), 128, 32, 2, lr, _ptr(outs[r]), C.byref(p), _stream(dev)))
    torch.cuda.synchronize()
    assert int(err.item()) == 0, "a rank timed out waiting for its peer"
    assert torch.equal(outs[0], outs[1])
    ref = _reference(a, (128, 32, 2), peers=[(b["rl"], b["sl"])])
    for r, d in enumerate(ranks):
        _compare("peers rank %d" % r, outs[r], d.flat[d.GRAD:].cpu().numpy().astype(np.float64), ref, a["w"])
