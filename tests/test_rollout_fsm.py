"""The default rollout (variant 6, rollout_states_kernel) on its state-machine image (csrc/nfsp_fsm.cuh, nfsp_rollout_image).

CPU: the image is walked on the host with the kernel's per-step recipe -- deal and policy entries, the two entry loads,
the reward word, the masks, the swap -- on the oracle's own score vectors, and the trace words (bit for bit), the RL / SL
records (as multisets), the counters and the state-table address of every decision are held against the CPU
restatement of Agent.play / main.train and the table's slot formula.

GPU: the instantiation the benchmark times (no debug outputs, RL records appended straight into the rings, several
blocks of games per warp, record buffers carried across blocks) against the oracle, launch after launch."""
import ctypes
import os

import numpy as np
import pytest

from oracle import orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "neural-ficititious-self-play-in-imperfect-information-games_b200")

# layout constants of csrc/nfsp_fsm.cuh ("the fused rollout's image") and csrc/rollout_states.cu
ROW, ENTRY, INFO, LIVE_ROWS = 112, 32, 96, 36
TERM_OFF = LIVE_ROWS * ROW
DEAL_OFF = TERM_OFF + 16 * 16
DEAL_HALF = 18 * ROW
POL_OFF = 120 * 16
REWARD_OFF = DEAL_OFF + 2 * DEAL_HALF
NET_SLOTS = 72 * 18
AT = 4 * NET_SLOTS * 16  # the image follows the state table
P_CLEAR, NZ, OVER, CM0 = 0x7E000, 1 << 15, 1 << 30, 0x07000000
M32 = 0xFFFFFFFF


@pytest.fixture(scope="module")
def image():
    import __graft_entry__ as g

    if not os.path.exists(os.path.join(PKG, "libnfsp_b200.so")):
        g.build()
    import nfsp_b200

    L = nfsp_b200.lib()
    n = L.nfsp_rollout_image(None, 0)
    assert n * 4 == REWARD_OFF + 4 * 1024
    buf = np.zeros(n, np.uint32)
    assert L.nfsp_rollout_image(buf.ctypes.data_as(ctypes.c_void_p), n) == n
    return buf


def f32(x):
    return int(np.float32(x).view(np.uint32))


def i8(v):
    return v - 256 if v & 0x80 else v


def score_word(v):
    """states_pack_kernel's fourth word: np.argmax * the entry size | (np.average != 0) << 15."""
    a = 0 if (v[1] <= v[0] and v[2] <= v[0]) else (1 if v[2] <= v[1] else 2)
    return a * ENTRY | (NZ if (v != 0).any() else 0)


def seq_id(rnd):
    s0, s1, s2 = rnd & 3, (rnd >> 2) & 3, (rnd >> 4) & 3
    return 6 + s0 if s2 else (2 * s0 + s1 if s1 else s0)


def formula_slot(net, card, pub, dealer, obs):
    """The state-table slot of a decision as the register formulation computed it from the game's fields."""
    h = obs & 0xFFFFFF
    both = h | (h >> 12)
    r = 1 if (obs >> 27) & 7 else 0
    fin0 = (seq_id(both & 63) >> 1) - 1 if r else 0
    sigma = 9 + seq_id((both >> 6) & 63) if r else seq_id(both & 63)
    return net * NET_SLOTS + ((((card * 3 + pub) * 2 + dealer) * 4 + fin0) * 18 + sigma)


class RolloutWalker:
    """One game, stepped the way rollout_states_kernel steps it (addresses: byte offsets from the state table)."""

    def __init__(self, img, seed, game, eta_u32):
        self.img, self.game, self.eta = img, game, eta_u32
        self.key = (seed & M32, seed >> 32)

    def words(self, addr, count):
        return [int(v) for v in self.img[(addr - AT) // 4: (addr - AT) // 4 + count]]

    def block(self, step):
        return [int(v) for v in orc.philox((self.game & M32, step & M32, step >> 32, 0), self.key)]

    def deal(self, x, dealer):
        self.dealer = dealer
        self.dl = AT + DEAL_OFF + dealer * DEAL_HALF
        D = self.words(self.dl + ((x[1] * 120) >> 32) * 16, 4)
        pa = self.dl + POL_OFF + (16 if x[2] < self.eta else 0) + (32 if x[3] < self.eta else 0)
        P = self.words(pa, 4)
        self.PA, self.PO = D[0] | P[0], D[1] | P[1]
        self.FA, self.FO = (D[2] + P[2]) & M32, (D[3] + P[3]) & M32
        self.SA = self.SO = 0
        self.tix, self.HX = self.dl - DEAL_OFF, CM0

    def reset(self, step):  # nfsp_reset_kernel: game g starts with dealer g & 1
        self.deal(self.block(step), self.game & 1)

    def step(self, step, vec):
        x = self.block(step)
        started = 0
        if self.HX & OVER:
            self.deal(x, 1 - self.dealer)
            started = 1
        q = (self.PA >> 23) & 1
        obs = self.HX & (self.PA | 0xFFFFFF)
        pol = (self.PA >> 12) & 1
        # the address the walk carries against the slot formula, from fields the walk does not use to address the table
        card, pub = (self.PA >> 19) & 3, (self.PA >> 21) & 3
        assert self.FA == 16 * formula_slot(2 * q + pol, card, pub, self.dealer, obs)
        recs = []
        if self.PA & NZ:
            recs.append(("rl", q, (self.SA, obs, 0, ((self.PA >> 13) & 3) | q << 16)))
        aw = score_word(vec)
        ea = self.tix + (aw & 0x60)
        hc, pa, pm, nx, ds, mx, rm, inc = self.words(ea, 8)
        self.PA = (((self.PA & ~P_CLEAR & M32) | (aw & NZ)) + pa) & M32
        self.HX = (self.HX & 0xFFFFFF) | hc
        term = self.HX & OVER
        rw = self.words(AT + REWARD_OFF + (rm & ((self.PA & 0xFF) | (self.PO & 0xF00))), 1)[0]
        ra, ro = i8(rw & 0xFF), i8((rw >> 8) & 0xFF)
        if term and aw & NZ:
            recs.append(("rl", q, (obs, self.HX & (self.PA | 0xFFFFFF), f32(0.5 * ra), mx & 0x10103)))
        if term and self.PO & NZ:
            recs.append(("rl", q ^ 1, (self.SO, self.HX & (self.PO | 0xFFFFFF), f32(0.5 * ro),
                                       ((self.PO >> 13) & 3) | ((mx & 0x10100) ^ 0x10000))))
        if pol:
            recs.append(("sl", q, (obs,) + tuple(int(v) for v in np.asarray(vec, np.float32).view(np.uint32))))
        P0, P1 = (self.PO, self.PA) if q else (self.PA, self.PO)
        misc = ((mx & 0x101F) | self.dealer << 5 | ((P0 >> 19) & 3) << 6 | ((P1 >> 19) & 3) << 8 | ((P0 >> 21) & 3) << 10 |
                ((P0 >> 2) & 15) << 13 | ((P1 >> 2) & 15) << 17 | started << 21 | ((P0 >> 12) & 1) << 22 | ((P1 >> 12) & 1) << 23)
        trace = (self.HX & (self.PA | 0xC0FFFFFF), f32(0.5 * ra), misc)
        fa, fo = (self.FA + ds) & M32, (self.FO + ds) & M32
        if pm:
            self.PA, self.PO = self.PO, self.PA
            self.SA, self.SO = self.SO, obs
            self.FA, self.FO = fo, fa
        else:
            self.SA, self.FA, self.FO = obs, fa, fo
        self.tix = nx
        rew = (ro, ra) if q else (ra, ro)
        return trace, recs, inc, rew


def ref_rows(recs):
    return sorted(tuple(int(v) for v in r) for r in np.ascontiguousarray(recs).view(np.uint32).reshape(-1, 4))


def forced_vectors(rng, steps, n):
    """Scores with exact ties, all-zero vectors and plain random ones."""
    v = rng.uniform(0, 1, (steps, n, 3)).astype(np.float32)
    kind = rng.randint(0, 8, (steps, n))
    v[kind == 0] = 0.0
    v[kind == 1, 1] = v[kind == 1, 0]
    v[kind == 2] = 0.25
    return v


def random_nets(rng):
    return [{"W1": rng.uniform(-0.25, 0.25, (30, 64)).astype(np.float32), "b1": rng.uniform(-0.2, 0.2, 64).astype(np.float32),
             "W2": rng.uniform(-0.3, 0.3, (64, 3)).astype(np.float32), "b2": rng.uniform(-0.2, 0.2, 3).astype(np.float32)}
            for _ in range(4)]


@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("seed,eta,eps", [(1234, 0.1, 0.06), (0xDEADBEEFCAFE, 0.5, 0.3), (77, 0.9, 0.9)])
def test_walking_the_rollout_image_reproduces_the_oracle(image, seed, eta, eps, forced):
    """forced=False: the oracle's nets and epsilon branch choose; forced=True: score vectors with exact ties and
    all-zero vectors (no records, no non-zero flag)."""
    n, steps = 120, 24
    eta_u32, eps_u32 = orc.u32_frac(eta), orc.u32_frac(eps)
    rng = np.random.RandomState(seed & 0xFFFF)
    b = orc.NfspBatch(n, seed)
    b.reset(0, eta_u32)
    fv = forced_vectors(rng, steps, n) if forced else None
    ref = b.rollout_act(1, steps, orc.Nets(random_nets(rng)), eta_u32, eps_u32, forced_vec=fv)
    vec = fv if forced else ref["vec"]
    rl, sl = [[], []], [[], []]
    actions, reward = np.zeros((2, 3), np.int64), [0, 0]
    for g in range(n):
        w = RolloutWalker(image, seed, g, eta_u32)
        w.reset(0)
        for t in range(steps):
            trace, recs, inc, rew = w.step(1 + t, vec[t, g])
            where = "game %d step %d" % (g, t)
            assert trace == (int(ref["trace"]["obs"][t, g]), int(ref["trace"]["reward"][t, g].view(np.uint32)),
                             int(ref["trace"]["misc"][t, g])), where
            for kind, p, r in recs:
                (rl if kind == "rl" else sl)[p].append(r)
            k = inc.bit_length() - 1
            actions[k // 15, (k // 5) % 3] += 1
            reward[0] += rew[0]
            reward[1] += rew[1]
    for p in range(2):
        assert sorted(rl[p]) == ref_rows(ref["rl"][p])
        assert sorted(sl[p]) == ref_rows(ref["sl"][p])
    assert np.array_equal(actions, ref["actions"]) and reward == list(ref["reward_half"])
    assert ref["hands"] > n * steps // 8
    assert not forced or (vec == 0).all(axis=2).sum() > n * steps // 16


def test_rollout_image_structure(image):
    """Each live entry leads to a row of the same dealer or to a terminal pseudo-row that says so, moves the state-table
    offset to the next row's, and counts its own (player, action)."""
    words = lambda off, k: [int(v) for v in image[off // 4: off // 4 + k]]  # noqa: E731
    seen_term = set()
    for row in range(LIVE_ROWS):
        sigma = row % 18
        if sigma % 9 >= 7:
            assert not image[row * ROW // 4: (row + 1) * ROW // 4].any()
            continue
        q = (words(row * ROW + INFO, 1)[0] >> 4) & 1
        for raw in range(3):
            hc, pa, pm, nx, ds, mx, rm, inc = words(row * ROW + raw * ENTRY, 8)
            assert (hc >> 31) == q and (mx & 3) == raw and ((pa >> 13) & 3) == raw and not pa & NZ
            assert inc == 1 << (5 * (3 * q + raw)) and (mx >> 16) == q
            nx -= AT
            info = words(nx + INFO, 1)[0]
            if (hc >> 30) & 1:
                assert nx >= TERM_OFF - INFO and (nx + INFO - TERM_OFF) % 16 == 0 and pm == 0
                assert (info >> 16) & 1 and ((info >> 4) & 1) == q
                assert rm in (0x3C, 0xFFC)
                seen_term.add(nx)
            else:
                assert nx % ROW == 0 and nx // ROW < LIVE_ROWS and (nx // ROW) // 18 == row // 18
                assert pm == (M32 if ((info >> 4) & 1) != q else 0) and rm == 0
                nsig = (nx // ROW) % 18
                assert nsig == sigma + ds // 16 if sigma < 9 and nsig < 9 or sigma >= 9 else nsig == 9
    assert len(seen_term) == 16
    rew = image[REWARD_OFF // 4:]
    assert rew[0] == 0


# --------------------------------------------------------------------------------------------------------------- GPU
def _rows(a):
    return [tuple(r) for r in np.ascontiguousarray(a).view(np.uint32).reshape(-1, 4).tolist()]


def _canon(a):
    a = np.ascontiguousarray(a).view(np.uint32).reshape(-1, 4)
    return a[np.lexsort(a.T[::-1])]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1 << 20, 1 << 16])
def test_benchmarked_instantiation_vs_oracle(n):
    """The production launch (no debug outputs, direct rings) over several launches: the rings hold the oracle's RL
    records, the staged SL records are the oracle's, game words and counters equal.  The oracle acts on the score
    vectors of a debug launch of the same kernel from the same state, so a last-bit difference between the state table
    and the oracle's forward cannot make the two take different actions in a near-tie."""
    torch = pytest.importorskip("torch")
    import nfsp_b200 as nb

    steps, seed, launches, eta, eps = 8, 99, 3, 0.2, 0.1
    cap = 1 << 25
    mk = lambda direct: nb.SelfPlay(n, seed=seed, eta=eta, epsilon=eps, rl_capacity=cap, sl_capacity=1 << 24,  # noqa: E731
                                    max_steps_per_call=steps, variant="states", direct_rings=direct)
    sd, ss = mk(True), mk(False)
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(eta))
    nets = orc.Nets([nb.split_net(w) for w in nb.glorot_nets(seed, "cuda").cpu().numpy()])
    want_rl = [[], []]
    stats = None
    for k in range(launches):
        out = ss.rollout(steps, insert=False, debug=True)
        ref = b.rollout_act(1 + k * steps, steps, nets, orc.u32_frac(eta), orc.u32_frac(eps),
                            forced_vec=out["vec"].cpu().numpy())
        ss.staged()  # the debug launch's own records are checked against the oracle by tests/test_gpu_act.py
        ss.flush()
        sd.rollout(steps, insert=False)
        _, sl = sd.staged()
        for p in range(2):
            want_rl[p].append(ref["rl"][p])
            assert len(sl[p]) == len(ref["sl"][p]) and np.array_equal(_canon(sl[p]), _canon(ref["sl"][p])), (k, p)
            total = int(sd.rl[p].total.item())
            assert total == sum(len(r) for r in want_rl[p]) and total <= cap
            assert np.array_equal(_canon(sd.rl[p].data[:total].cpu().numpy()), _canon(np.concatenate(want_rl[p]))), (k, p)
        sd.flush()
        st = sd.read_stats()
        if stats is not None:
            st = {key: st[key] - stats[key] for key in st}
        stats = sd.read_stats()
        assert [st["a0_fold"], st["a0_call"], st["a0_raise"]] == list(ref["actions"][0])
        assert [st["a1_fold"], st["a1_call"], st["a1_raise"]] == list(ref["actions"][1])
        to_s = lambda v: v - (1 << 64) if v >= 1 << 63 else v  # noqa: E731
        assert [to_s(st["reward0_half"]) & M32, to_s(st["reward1_half"]) & M32] == [v & M32 for v in ref["reward_half"]]
        assert st["hands"] == ref["hands"] and st["transitions"] == n * steps and st["dropped"] == 0
        assert np.array_equal(sd.env.state_words().cpu().numpy(), ss.env.state_words().cpu().numpy())
    assert torch.cuda.is_available()
