"""-m gpu: the CUDA environments (K1) against the golden fixtures produced by the reference and against
the CPU oracle on identical seeded inputs.  Everything is integer / byte work => bit-exact."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402


def load(golden_dir, name):
    with np.load(os.path.join(golden_dir, name)) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


# ------------------------------------------------------------------------------- ENV_NFSP
def test_nfsp_env_golden_exhaustive(nb, golden_dir):
    """All 20 352 reference hands as one batch: every env.step compared field by field."""
    g = load(golden_dir, "nfsp_exhaustive.npz")
    T = len(g["dealer"])
    env = nb.BatchedNfspEnv(T, seed=1)
    env.set_hands(g["dealer"], g["cards"], g["policy"])
    code = g["kind"].copy()  # 0 F, 1 C, 2 R, 3 Z == kernel action codes
    for d in range(6):
        live = g["n_dec"] > d
        acts = np.where(live, code[:, d], 4).astype(np.int8)
        pl = np.where(live, g["player"][:, d], 0).astype(np.int8)
        s, a, r, s2, t = env.get_state(pl)
        assert np.array_equal(s2.cpu().numpy().view(np.uint32)[live], g["obs_before"][live, d])
        env.step(acts[None], pl[None], n_steps=1, auto_reset=False)
        e = _np(env.export())
        assert np.array_equal(e["terminated"][live], g["terminated"][live, d])
        assert np.array_equal(e["round"][live], g["round"][live, d])
        assert np.array_equal(e["k"][live], g["round_raises"][live, d])
        assert np.array_equal(e["bets0"][live], (2 * g["bets"][live, d, 0]).astype(np.int32))
        assert np.array_equal(e["bets1"][live], (2 * g["bets"][live, d, 1]).astype(np.int32))
        assert np.array_equal(e["rew0_half"][live], (2 * g["reward"][live, d, 0]).astype(np.int32))
        assert np.array_equal(e["rew1_half"][live], (2 * g["reward"][live, d, 1]).astype(np.int32))
        assert np.array_equal(e["obs0"].view(np.uint32)[live], g["obs_after"][live, d, 0])
        assert np.array_equal(e["obs1"].view(np.uint32)[live], g["obs_after"][live, d, 1])
        assert np.array_equal(e["snap0"].view(np.uint32)[live], g["snap"][live, d, 0])
        assert np.array_equal(e["snap1"].view(np.uint32)[live], g["snap"][live, d, 1])
        assert int(e["anomaly"][live].sum()) == 0


def test_nfsp_env_golden_call_order_fuzz(nb, golden_dir):
    """Arbitrary players, repeated calls, steps after the terminal: the single-game API contract."""
    g = load(golden_dir, "fuzz_nfsp_calls.npz")
    N, K = g["op"].shape
    env = nb.BatchedNfspEnv(N, seed=1)
    env.set_hands(g["dealer"], g["cards"])
    from nfsp_b200.leduc.newenv import action_code

    for c in range(K):
        is_step = g["op"][:, c] == 0
        pl = g["player"][:, c].astype(np.int8)
        acts = np.where(is_step, action_code(g["vec"][:, c]), 4).astype(np.int8)
        s, a, r, s2, t = env.get_state(pl)  # the reference's get_state, before this call's step
        rr = np.where(t.cpu().numpy() > 0, r.cpu().numpy(), 0)
        env.step(acts[None], pl[None], n_steps=1, auto_reset=False)
        e = _np(env.export())
        assert np.array_equal(e["terminated"], g["terminated"][:, c]), c
        assert np.array_equal(e["round"], g["round"][:, c])
        assert np.array_equal(e["bets0"], (2 * g["bets"][:, c, 0]).astype(np.int32))
        assert np.array_equal(e["bets1"], (2 * g["bets"][:, c, 1]).astype(np.int32))
        assert np.array_equal(e["rew0_half"], (2 * g["reward"][:, c, 0]).astype(np.int32))
        assert np.array_equal(e["rew1_half"], (2 * g["reward"][:, c, 1]).astype(np.int32))
        assert np.array_equal(e["obs0"].view(np.uint32), g["obs"][:, c, 0])
        assert np.array_equal(e["obs1"].view(np.uint32), g["obs"][:, c, 1])
        assert np.array_equal(e["snap0"].view(np.uint32), g["snap"][:, c, 0])
        assert np.array_equal(e["snap1"].view(np.uint32), g["snap"][:, c, 1])
        gs = ~is_step  # get_state(p) results of the reference at this call
        assert np.array_equal(rr[gs], g["gs_r"][gs, c])


def test_nfsp_do_action_alone_golden(nb, golden_dir):
    """newenv.Env.do_action (newenv.py:131-178) called on its own, against the reference's method: 2 400 hands brought
    somewhere by step() calls, then bare do_action calls by arbitrary players (a hand ends with its first fold) -- return value, history, round_raises,
    chips, `terminated` untouched, last_action -- and the single-game drop-in class on the first hands."""
    g = load(golden_dir, "do_action.npz")
    N, C = g["op"].shape
    from nfsp_b200.leduc.newenv import Env, action_code

    env = nb.BatchedNfspEnv(N, seed=1)
    env.set_hands(g["dealer"], g["cards"])
    n_calls = 0
    for c in range(C):
        op, pl = g["op"][:, c], g["player"][:, c].astype(np.int8)
        code = action_code(g["vec"][:, c])
        env.step(np.where(op == 0, code, 4).astype(np.int8)[None], pl[None], n_steps=1, auto_reset=False)
        fold = env.do_action(np.where(op == 1, code, -1).astype(np.int8), pl).cpu().numpy()
        e = _np(env.export())
        live, bare = op >= 0, op == 1
        n_calls += int(bare.sum())
        assert np.array_equal(fold[bare], g["ret"][bare, c].astype(bool)), c
        assert not fold[~bare].any()
        assert np.array_equal(e["hist"][live].view(np.uint32), g["hist"][live, c]), c
        assert np.array_equal(e["round"][live], g["round"][live, c]) and np.array_equal(e["k"][live], g["round_raises"][live, c])
        assert np.array_equal(e["bets0"][live], (2 * g["bets"][live, c, 0]).astype(np.int32))
        assert np.array_equal(e["bets1"][live], (2 * g["bets"][live, c, 1]).astype(np.int32))
        assert np.array_equal(e["terminated"][live], g["terminated"][live, c]) and not e["anomaly"][live].any()
        for q in (0, 1):  # last_action[q] (newenv.py:136): its argmax and whether it is the zero vector
            la = g["last_action"][live, c, q]
            assert np.array_equal(e["last_a%d" % q][live], np.argmax(la, axis=1))
            assert np.array_equal(e["nz%d" % q][live].astype(bool), (la != 0).any(axis=1))
    assert n_calls == int((g["op"] == 1).sum()) > 2000 and int(g["ret"].sum()) > 500
    for i in range(40):  # the reference-shaped class, one game at a time
        one = Env(n_games=1, seed=1, config_path=None)
        one.load_hand(int(g["dealer"][i]), g["cards"][i])
        for c in range(C):
            if g["op"][i, c] == 0:
                one.step(g["vec"][i, c].reshape(1, 1, 3), int(g["player"][i, c]))
            elif g["op"][i, c] == 1:
                assert one.do_action(g["vec"][i, c].reshape(1, 1, 3), int(g["player"][i, c])) is bool(g["ret"][i, c])
                assert np.array_equal(one.last_action[0], g["last_action"][i, c])


def _with_step0(cases):
    """Each case at step counters 1 (a fresh run), 2^32 - 5 (the launch crosses 2^32, where the counter's high word
    enters Philox counter word 2) and 2^40 + 3 (a resumed run of a long life); a fresh run keeps its old test id."""
    params = []
    for case in cases:
        for step0 in (1, 2 ** 32 - 5, 2 ** 40 + 3):
            tag = "-".join(map(str, case)) + ("" if step0 == 1 else "-step0=%d" % step0)
            params.append(pytest.param(*case, step0, id=tag))
    return params


@pytest.mark.parametrize("n,steps,step0", _with_step0([(1, 40), (257, 33), (100_000, 24)]))
def test_nfsp_env_seeded_rollout_vs_oracle(nb, n, steps, step0):
    """Philox deals + uniform-random actions + auto re-deal: trace planes bit-exact vs the oracle, from step counter
    step0 on."""
    seed, eta = 1234, 0.1
    env = nb.BatchedNfspEnv(n, seed=seed, eta=eta)
    env.reset()
    env.step_counter = step0
    tr = env.step(n_steps=steps, trace=True)["raw"].cpu().numpy().view(np.uint32)
    assert env.step_counter == step0 + steps
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(eta))
    ref = b.rollout_env(step0, steps, orc.u32_frac(eta))
    assert np.array_equal(tr[0], ref["obs"])
    assert np.array_equal(tr[1].view(np.float32), ref["reward"])
    assert np.array_equal(tr[2], ref["misc"])
    # the same rollout, one launch per step, lands in the same packed words
    env2 = nb.BatchedNfspEnv(n, seed=seed, eta=eta)
    env2.reset()
    env2.step_counter = step0
    for _ in range(steps):
        env2.step(n_steps=1)
    assert torch.equal(env.state_words(), env2.state_words())


def test_state_machine_and_packed_word_kernels_agree_at_full_size(nb):
    """BASELINE config 2 size (2^20 games), 32 transitions per game: the table-driven kernel (Philox actions) and the
    packed-word kernel (the same actions passed explicitly) must leave identical trace planes and game words, launch
    after launch -- every (dealer, betting sequence, action) entry, deal and re-deal is hit tens of thousands of times."""
    n, steps = 1 << 20, 16
    a, b = nb.BatchedNfspEnv(n, seed=2024, eta=0.3), nb.BatchedNfspEnv(n, seed=2024, eta=0.3)
    a.reset()
    b.reset()
    for _ in range(2):
        ta = a.step(n_steps=steps, trace=True)
        tb = b.step(actions=ta["action"].to(torch.int8), n_steps=steps, auto_reset=True, trace=True)
        assert torch.equal(ta["raw"], tb["raw"])
        assert torch.equal(a.state_words(), b.state_words())
    hands = int(ta["terminated"].sum())
    assert 2.4 < n * steps / hands < 2.8


def test_legacy_state_machine_agrees_with_call_by_call_kernels_at_full_size(nb):
    """2^20 games of the README loop: the table-driven rollout kernel against the SAME actions played through
    nfsp_legacy_step / nfsp_legacy_get_new_state (the packed-word rules, one call per README line) until each game's
    first hand ends; records and exported fields must match for every live game."""
    n, iters = 1 << 20, 6
    roll, manual = nb.BatchedLegacyEnv(n, seed=31), nb.BatchedLegacyEnv(n, seed=31)
    roll.reset()
    manual.load_state_words(roll.state_words())
    rec = roll.rollout(iters, trace=True)
    live = torch.ones(n, dtype=torch.bool, device=roll.device)
    for k in range(iters):
        acts = rec["action"][k].to(torch.int8)           # [n, 2]
        sit = torch.full((n,), 4, dtype=torch.int8, device=roll.device)
        manual.step(torch.where(live, acts[:, 0], sit), 0)
        manual.step(torch.where(live, acts[:, 1], sit), 1)
        out = [manual.get_new_state(torch.where(live, torch.full_like(sit, p), torch.full_like(sit, 2))) for p in (0, 1)]
        for p in (0, 1):
            got = torch.stack([rec["card"][k, :, p], rec["pub"][k, :, p], rec["pot"][k, :, p], rec["reward"][k, :, p],
                               rec["terminal"][k, :, p]], 1)
            assert torch.equal(got[live], out[p][live].to(got.dtype)), (k, p)
        live &= ~(rec["terminal"][k, :, 0].bool() | rec["terminal"][k, :, 1].bool())
    assert int(live.sum()) < n // 50  # nearly every first hand is over after 6 iterations


def test_nfsp_env_sharding_invariance(nb):
    """SURVEY 8e: a game's trace depends on its GLOBAL id only -- two shards == one batch."""
    n, steps = 4096, 20
    whole = nb.BatchedNfspEnv(n, seed=7)
    whole.reset()
    tw = whole.step(n_steps=steps, trace=True)["raw"]
    parts = []
    for k in range(2):
        sh = nb.BatchedNfspEnv(n // 2, seed=7, game0=k * (n // 2))
        sh.reset()
        parts.append(sh.step(n_steps=steps, trace=True)["raw"])
    assert torch.equal(tw, torch.cat(parts, dim=2))


def test_nfsp_env_properties_at_scale(nb):
    """BASELINE config 2 size (1M games): size-independent invariants of the domain."""
    n, steps = 1 << 20, 16
    env = nb.BatchedNfspEnv(n, seed=99)
    env.reset()
    tr = env.step(n_steps=steps, trace=True)
    term = tr["terminated"].bool()
    r2 = (tr["reward"] * 2).round().to(torch.int32)
    assert bool((tr["reward"][~term] == 0).all())
    assert set(torch.unique(r2[term].abs()).tolist()) <= {0, 1, 2, 4, 6, 8, 10}
    # zero-sum: the loser's loss is the winner's gain -> over many hands the two seats' totals cancel
    e = env.export()
    assert int(e["anomaly"].sum()) == 0
    hands = int(term.sum())
    assert 2.4 < n * steps / hands < 2.8  # 2.58 transitions / hand under uniform play (SURVEY 6)
    # deal law (deck.py): 24 reachable rank triples, all-distinct twice as likely as one pair
    first = tr["started"][1:].bool()
    key = (tr["c0"][1:] * 16 + tr["c1"][1:] * 4 + tr["pub"][1:])[first]
    cnt = torch.bincount(key, minlength=64).cpu().numpy()
    assert (cnt > 0).sum() == 24
    tot = cnt.sum()
    for k in np.nonzero(cnt)[0]:
        c = (k >> 4, (k >> 2) & 3, k & 3)
        exp = tot * (8 if len(set(c)) == 3 else 4) / 120.0
        assert abs(cnt[k] - exp) < 6 * np.sqrt(exp)


# ------------------------------------------------------------------------------- ENV_LEGACY
def test_legacy_env_golden_exhaustive(nb, golden_dir):
    g = load(golden_dir, "legacy_exhaustive.npz")
    T, I = g["actions"].shape[:2]
    env = nb.BatchedLegacyEnv(T, seed=1)
    env.set_hands(g["cards"])
    e = _np(env.export())
    assert np.array_equal(np.stack([e["c0"], e["c1"]], 1), g["cards"])
    for k in range(I):
        live = g["n_it"] > k
        for p in (0, 1):
            env.step(np.where(live, g["actions"][:, k, p], 4).astype(np.int8), p)
        e = _np(env.export())
        for p in (0, 1):
            assert np.array_equal(e["left%d" % p][live], g["left"][live, k, p])
            assert np.array_equal(e["pot%d" % p][live], g["pot"][live, k, p])
            assert np.array_equal(e["term%d" % p][live], g["term_step"][live, k, p])
        for p in (0, 1):
            pl = np.where(live, p, 2).astype(np.int8)
            out = env.get_new_state(pl).cpu().numpy()
            assert np.array_equal(out[live], g["out"][live, k, p]), (k, p)


def test_legacy_rollout_kernel_golden(nb, golden_dir):
    """The fused README-iteration kernel on the same exhaustive traces (first hand of every game)."""
    g = load(golden_dir, "legacy_exhaustive.npz")
    T, I = g["actions"].shape[:2]
    env = nb.BatchedLegacyEnv(T, seed=1)
    env.set_hands(g["cards"])
    acts = np.where(g["actions"] < 0, 1, g["actions"]).astype(np.int8).transpose(1, 0, 2).copy()
    rec = env.rollout(I, acts, trace=True)
    out = np.stack([_np(rec)[k] for k in ("card", "pub", "pot", "reward", "terminal")], -1)  # [I, T, 2, 5]
    for k in range(I):
        live = g["n_it"] > k
        assert np.array_equal(out[k][live], g["out"][live, k]), k


def test_legacy_env_golden_call_order_fuzz(nb, golden_dir):
    g = load(golden_dir, "fuzz_legacy_calls.npz")
    N, K = g["op"].shape
    env = nb.BatchedLegacyEnv(N, seed=1)
    env.set_hands(g["cards"])
    for c in range(K):
        is_step = g["op"][:, c] == 0
        pl = g["player"][:, c].astype(np.int8)
        env.step(np.where(is_step, g["action"][:, c], 4).astype(np.int8), pl)
        env.get_new_state(np.where(is_step, 2, pl).astype(np.int8), want_out=False)
        e = _np(env.export())
        for q in (0, 1):
            assert np.array_equal(e["left%d" % q], g["left"][:, c, q]) and np.array_equal(e["pot%d" % q], g["pot"][:, c, q])
            st = np.stack([e["c%d" % q], np.full(N, -1), e["st_pot%d" % q], e["rew%d" % q], e["term%d" % q]], 1)
            assert np.array_equal(st, g["st"][:, c, q]), (c, q)


@pytest.mark.parametrize("n,iters,step0", _with_step0([(1, 30), (1000, 17), (100_000, 12)]))
def test_legacy_seeded_rollout_vs_oracle(nb, n, iters, step0):
    seed = 4321
    env = nb.BatchedLegacyEnv(n, seed=seed)
    env.reset()
    env.step_counter = step0
    rec = env.rollout(iters, trace=True)["raw"].cpu().numpy()
    b = orc.LegacyBatch(n, seed)
    b.reset(0)
    ref = b.rollout(step0, iters)
    w = rec[0].view(np.uint32)
    sb = lambda x: ((x & 0xFF).astype(np.int16) ^ 0x80) - 0x80  # noqa: E731
    assert np.array_equal(sb(w), ref["card"]) and np.array_equal(sb(w >> 8), ref["pub"])
    assert np.array_equal(sb(w >> 16), ref["pot"]) and np.array_equal(sb(w >> 24), ref["terminal"])
    assert np.array_equal(rec[1], ref["reward"])
    assert np.array_equal(rec[2].view(np.uint32), ref["misc"])
    for gi in (0, n // 2, n - 1):
        e, o = _np(env.export()), b.env(gi)
        assert [e["left0"][gi], e["left1"][gi], e["pot0"][gi], e["pot1"][gi]] == [o.left[0], o.left[1], o.pot[0], o.pot[1]]


def test_legacy_rollout_is_independent_of_launch_batching(nb):
    """One launch of 12 README iterations == launches of 7 + 5 == twelve launches of 1: between launches a live hand
    travels as the packed word and comes back through the state-key table of the table-driven kernel."""
    n = 50_000
    envs = [nb.BatchedLegacyEnv(n, seed=8) for _ in range(4)]
    for e in envs:
        e.reset()
    envs[3].rollout(12)  # the kernel variant that writes no records must leave the same words
    whole = envs[0].rollout(12, trace=True)["raw"]
    parts = torch.cat([envs[1].rollout(7, trace=True)["raw"], envs[1].rollout(5, trace=True)["raw"]], dim=1)
    ones = torch.cat([envs[2].rollout(1, trace=True)["raw"] for _ in range(12)], dim=1)
    assert torch.equal(whole, parts) and torch.equal(whole, ones)
    for e in envs[1:]:
        assert torch.equal(envs[0].state_words(), e.state_words())
    live = int((whole[0, -1, :, 0] >> 24 & 1).eq(0).sum())
    assert live > n // 4  # plenty of hands were still live at the launch boundaries


def _deal_ranks(idx):  # deck.py:35-50: ordered draw of 3 of the 6 cards -> ranks
    i0, r = divmod(idx, 20)
    j1, j2 = r >> 2, r & 3
    i1 = j1 + (j1 >= i0)
    lo, hi = min(i0, i1), max(i0, i1)
    i2 = j2 + (j2 >= lo)
    i2 += i2 >= hi
    return i0 >> 1, i1 >> 1, i2 >> 1


def test_legacy_rollout_from_hand_stepped_states(nb, golden_dir):
    """Hands stepped by hand in the fuzz fixture's call orders (terminal flags and accumulated rewards a rollout can
    never produce), THEN handed to the rollout kernel: such words are played by its packed-word path, ordinary ones by
    the table path, and every record must equal the reference rules driven call by call on the same Philox stream."""
    g = load(golden_dir, "fuzz_legacy_calls.npz")
    N, K = g["op"].shape
    seed, iters, step0 = 99, 10, 5
    env = nb.BatchedLegacyEnv(N, seed=seed)
    env.set_hands(g["cards"])
    for c in range(K):
        is_step = g["op"][:, c] == 0
        pl = g["player"][:, c].astype(np.int8)
        env.step(np.where(is_step, g["action"][:, c], 4).astype(np.int8), pl)
        env.get_new_state(np.where(is_step, 2, pl).astype(np.int8), want_out=False)
    before = _np(env.export())
    env.step_counter = step0
    rec = env.rollout(iters, trace=True)["raw"].cpu().numpy()
    after = _np(env.export())
    key = (seed & 0xFFFFFFFF, seed >> 32)
    odd = 0
    for gi in range(0, N, 3):
        e = orc.LegacySingle()
        e.reset(int(g["cards"][gi, 0]), int(g["cards"][gi, 1]))
        for c in range(K):
            if g["op"][gi, c] == 0:
                e.step(int(g["action"][gi, c]), int(g["player"][gi, c]))
            else:
                e.get_new_state(int(g["player"][gi, c]))
        odd += int(before["term0"][gi] | before["term1"][gi] | (before["rew0"][gi] not in (0, -1)) | (before["rew1"][gi] not in (0, -1)))
        need = False
        for t in range(iters):
            x = [int(v) for v in orc.philox((gi, step0 + t, 0, 0), key)]
            started = 0
            if need:
                c0, c1, _ = _deal_ranks((x[2] * 120) >> 32)
                e.reset(c0, c1)
                started = 1 << 8
            a = ((x[0] * 3) >> 32, (x[1] * 3) >> 32)
            e.step(a[0], 0)
            e.step(a[1], 1)
            out = [e.get_new_state(0)]
            left0, pot0 = e.e.left[0], e.e.pot[0]
            out.append(e.get_new_state(1))
            for p in (0, 1):
                w, where = int(rec[0, t, gi, p]) & 0xFFFFFFFF, "game %d iteration %d player %d" % (gi, t, p)
                card, pub, pot, reward, term = out[p]
                assert (w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFF, (w >> 24) & 0xFF) == (card, pub & 0xFF, pot, term), where
                assert int(rec[1, t, gi, p]) == reward, where
                misc = a[p] | ((e.e.left[p] + 1) << 2) | (e.e.pot[p] << 5) | started
                assert int(rec[2, t, gi, p]) & 0xFFFFFFFF == misc, where
            assert (left0, pot0) == (e.e.left[0], e.e.pot[0])
            need = bool(out[0][4] | out[1][4])
        assert [after["left0"][gi], after["left1"][gi], after["pot0"][gi], after["pot1"][gi]] == [e.e.left[0], e.e.left[1], e.e.pot[0], e.e.pot[1]]
        assert [after["rew0"][gi], after["rew1"][gi]] == [e.e.st_reward[0], e.e.st_reward[1]]
    assert odd > 20  # the packed-word path was exercised


# ------------------------------------------------------------------------------- drop-in classes
def test_dropin_newenv_single_game(nb, golden_dir):
    """leduc.newenv.Env with the reference's shapes, replaying a slice of the golden hands."""
    nb.install_dropin()
    import leduc.newenv as leduc

    g = load(golden_dir, "nfsp_exhaustive.npz")
    env = leduc.Env()
    assert env.observation_space == (1, 30) and env.action_space == (3,)
    for i in range(0, len(g["dealer"]), 997):
        env.load_hand(int(g["dealer"][i]), g["cards"][i])
        for d in range(int(g["n_dec"][i])):
            p = int(g["player"][i, d])
            s, a, r, s2, t = env.get_state(p)
            assert s.shape == (1, 30) and a.shape == (1, 1, 3) and s2.shape == (1, 1, 30) and t is False
            assert orc_mask(s2) == g["obs_before"][i, d]
            env.step(g["vec"][i, d].reshape(1, 1, 3), p)
            assert env.round_index == g["round"][i, d]
        for p in (0, 1):
            s, a, r, s2, t = env.get_state(p)
            d = int(g["n_dec"][i]) - 1
            assert t is True and r == g["reward"][i, d, p] and orc_mask(s) == g["snap"][i, d, p]


def orc_mask(v):
    v = np.asarray(v).reshape(-1)
    return sum(1 << i for i in range(30) if v[i] != 0)


def test_dropin_legacy_env_readme_flow(nb, golden_dir):
    """README.md:15-38 usage of leduc.env.Env against golden traces."""
    nb.install_dropin()
    import leduc.env as leduc

    g = load(golden_dir, "legacy_exhaustive.npz")
    env = leduc.Env()
    assert env.dim_shape == (1, 3) and env.observation_space == 3 and env.action_space == 3
    for i in range(0, len(g["n_it"]), 1409):
        env.load_hand(int(g["cards"][i, 0]), int(g["cards"][i, 1]))
        assert env.init_state(0).tolist() == [[int(g["cards"][i, 0]), -1, 0]]
        for k in range(int(g["n_it"][i])):
            for p in (0, 1):
                v = np.zeros(3)
                v[g["actions"][i, k, p]] = 1
                env.step(v, p)
            for p in (0, 1):
                s, a, r, t, info = env.get_new_state(p)
                assert s.tolist() == [list(g["out"][i, k, p][:3])] and (r, t) == tuple(g["out"][i, k, p][3:])
                assert info == ""
    env.reset()  # Philox deal path
    assert env.init_state(1).shape == (1, 3)


def test_lean_and_general_kernels_agree_after_manual_hands(nb):
    """Hands played to the end WITHOUT auto re-deal, then handed to the auto re-deal paths: the lean kernel
    (Philox actions) and the general kernel (the same actions passed explicitly) re-deal them and stay word for
    word identical, traces included."""
    n, steps = 5000, 10
    rng = np.random.RandomState(4)
    envs = [nb.BatchedNfspEnv(n, seed=77) for _ in range(2)]
    dealer = rng.randint(0, 2, n).astype(np.int8)
    cards = np.stack([rng.randint(0, 3, n), rng.randint(0, 3, n), rng.randint(0, 3, n)], 1).astype(np.int8)
    manual = rng.randint(0, 3, (6, n)).astype(np.int8)
    for e in envs:
        e.set_hands(dealer, cards)
        for k in range(6):   # some games finish early and then refuse further steps (anomaly flag), as in the reference
            e.step(manual[k:k + 1], n_steps=1, auto_reset=False)
        e.step_counter = 100
    lean = envs[0].step(n_steps=steps, trace=True)
    acts = lean["action"].to(torch.int8)
    gen = envs[1].step(actions=acts, n_steps=steps, auto_reset=True, trace=True)
    assert torch.equal(lean["raw"], gen["raw"])
    assert torch.equal(envs[0].state_words(), envs[1].state_words())
