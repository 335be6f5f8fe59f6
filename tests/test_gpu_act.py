"""-m gpu: NFSP acting (K2) and the memories (K3/K4/K5) against the CPU oracle.

Integer work (records, slots, indices, counters) is bit-exact; the MLP outputs (Q-values and
policy probabilities) are compared at 1e-5 absolute in fp32, the tolerance BASELINE.json states.
Action selection is checked on the kernel's OWN score vectors (teacher forcing), so a last-bit
difference in a near-tie cannot derail the env trace comparison.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

TOL = 1e-5  # BASELINE.json north_star: "within 1e-5 absolute (fp32)"


def load(golden_dir, name):
    with np.load(os.path.join(golden_dir, name)) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def canon(recs):
    """16-byte records as a lexicographically sorted [n,4] uint32 matrix (order-free comparison)."""
    a = np.ascontiguousarray(recs).view(np.uint32).reshape(-1, 4)
    return a[np.lexsort(a.T[::-1])]


def raw16(recs):
    return np.ascontiguousarray(recs).view(np.uint32).reshape(-1, 4)


def random_nets(seed, scale=1.0):
    rng = np.random.RandomState(seed)
    w = np.zeros((4, 2179), np.float32)
    for k in range(4):
        w[k, :1920] = rng.uniform(-0.2526, 0.2526, 1920) * scale
        w[k, 1920:1984] = rng.uniform(-0.2, 0.2, 64)
        w[k, 1984:2176] = rng.uniform(-0.2993, 0.2993, 192) * scale
        w[k, 2176:] = rng.uniform(-0.2, 0.2, 3)
    return w


def oracle_nets(nb, w):
    return orc.Nets([nb.split_net(w[k]) for k in range(4)])


def test_forward_q_values_and_policy_probabilities(nb, golden_dir):
    """Every observation the game can produce x four nets: |GPU - oracle| <= 1e-5, and the fp32 oracle
    itself is bounded by a float64 evaluation."""
    g = load(golden_dir, "nfsp_exhaustive.npz")
    obs = np.unique(np.concatenate([g["obs_before"].ravel(), g["obs_after"].ravel()])).astype(np.uint32)
    for seed, scale in ((0, 1.0), (1, 4.0)):
        w = random_nets(seed, scale)
        sp = nb.SelfPlay(64, weights=torch.from_numpy(w), rl_capacity=1024, sl_capacity=1024)
        nets = oracle_nets(nb, w)
        x = ((obs[:, None] >> np.arange(30)) & 1).astype(np.float32)
        for k, tc in [(k, tc) for k in range(4) for tc in (False, True)]:
            got = sp.forward(torch.from_numpy(obs.astype(np.int32)), torch.full((len(obs),), k, dtype=torch.int8),
                             tensor_cores=tc)
            got = got.cpu().numpy()
            ref = nets.forward(k, x, "br" if k & 1 else "avg")
            assert np.abs(got - ref).max() <= TOL, (seed, k, tc, np.abs(got - ref).max())
            # float64 bound
            wk = {a: b.astype(np.float64) for a, b in nb.split_net(w[k]).items()}
            h = np.maximum(x @ wk["W1"] + wk["b1"], 0)
            z = h @ wk["W2"] + wk["b2"]
            if k & 1:
                ref64 = np.maximum(z, 0)
            else:
                e = np.exp(z - z.max(1, keepdims=True))
                ref64 = e / e.sum(1, keepdims=True)
                assert np.abs(got.sum(1) - 1).max() < 1e-5
            assert np.abs(got - ref64).max() <= TOL


def test_forward_tensor_core_mixed_nets_ragged(nb):
    """tcgen05 forward with every tile holding a random mix of the four nets, and a ragged last tile."""
    rng = np.random.RandomState(4)
    w = random_nets(2, 2.0)
    sp = nb.SelfPlay(64, weights=torch.from_numpy(w), rl_capacity=1024, sl_capacity=1024)
    nets = oracle_nets(nb, w)
    for n in (1, 127, 128, 129, 5000):
        obs = rng.randint(0, 1 << 30, n).astype(np.int32)
        k = rng.randint(0, 4, n).astype(np.int8)
        got = sp.forward(torch.from_numpy(obs), torch.from_numpy(k), tensor_cores=True).cpu().numpy()
        base = sp.forward(torch.from_numpy(obs), torch.from_numpy(k)).cpu().numpy()
        x = ((obs.astype(np.uint32)[:, None] >> np.arange(30)) & 1).astype(np.float32)
        ref = np.zeros((n, 3), np.float32)
        for kk in range(4):
            m = k == kk
            if m.any():
                ref[m] = nets.forward(kk, x[m], "br" if kk & 1 else "avg")
        assert np.abs(got - ref).max() <= TOL and np.abs(base - ref).max() <= TOL, n


@pytest.mark.parametrize("variant", ["states", "pairs", "sorted", "cuda", "tcgen05", "tcgen05_ws"])
@pytest.mark.parametrize("n,steps,eta,eps,step0", [
    pytest.param(1, 30, 0.5, 0.5, 1, id="1-30-0.5-0.5"),
    pytest.param(1000, 12, 0.1, 0.06, 1, id="1000-12-0.1-0.06"),
    pytest.param(1000, 12, 0.1, 0.06, 2 ** 32 - 5, id="1000-12-0.1-0.06-step0=4294967291"),
    pytest.param(50_000, 8, 0.3, 0.2, 1, id="50000-8-0.3-0.2")])
def test_fused_rollout_vs_oracle(nb, n, steps, eta, eps, step0, variant):
    """The fused act+step+remember kernel vs the oracle's restatement of Agent.play/main.train, from step counter
    step0 on (2^32 - 5: the launch crosses 2^32, where the counter's high word enters Philox counter word 2)."""
    seed = 2024
    w = random_nets(5)
    sp = nb.SelfPlay(n, weights=torch.from_numpy(w), seed=seed, eta=eta, epsilon=eps, rl_capacity=1 << 12,
                     sl_capacity=1 << 12, max_steps_per_call=steps, variant=variant)
    sp.env.step_counter = step0
    out = sp.rollout(steps, insert=False, debug=True)
    rl, sl = sp.staged()
    vec = out["vec"].cpu().numpy()
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(eta))
    ref = b.rollout_act(step0, steps, oracle_nets(nb, w), orc.u32_frac(eta), orc.u32_frac(eps), forced_vec=vec)
    tr = out["raw"].cpu().numpy().view(np.uint32)
    assert np.array_equal(tr[0], ref["trace"]["obs"])
    assert np.array_equal(tr[1].view(np.float32), ref["trace"]["reward"])
    assert np.array_equal(tr[2], ref["trace"]["misc"])
    assert np.abs(vec - ref["vec"]).max() <= TOL
    for p in range(2):
        assert len(rl[p]) == len(ref["rl"][p]) and len(sl[p]) == len(ref["sl"][p])
        assert np.array_equal(canon(rl[p]), canon(ref["rl"][p]))
        assert np.array_equal(canon(sl[p]), canon(ref["sl"][p]))
    st = sp.read_stats()
    assert [st["a0_fold"], st["a0_call"], st["a0_raise"]] == list(ref["actions"][0])
    assert [st["a1_fold"], st["a1_call"], st["a1_raise"]] == list(ref["actions"][1])
    assert [st["played0"], st["played1"]] == list(ref["played"])
    to_s = lambda v: v - (1 << 64) if v >= 1 << 63 else v  # noqa: E731
    assert [to_s(st["reward0_half"]), to_s(st["reward1_half"])] == list(ref["reward_half"])
    assert st["hands"] == ref["hands"] and st["transitions"] == n * steps and st["dropped"] == 0
    # the per-hand policy draws of main.py:38-45 come out with P('b') = eta
    if n >= 1000:
        started = out["started"][1:].bool()
        pol = torch.cat([out["pol0"][1:][started], out["pol1"][1:][started]]).float()
        assert abs(float(pol.mean()) - eta) < 5 * (eta * (1 - eta) / pol.numel()) ** 0.5 + 1e-3


@pytest.mark.parametrize("variant", ["states", "pairs", "sorted", "cuda", "tcgen05", "tcgen05_ws"])
def test_fused_rollout_golden_hands(nb, golden_dir, variant):
    """All 20 352 reference hands (incl. zero vectors and argmax ties) through the fused kernel with the
    reference's scripted score vectors; records must equal the oracle's, which is pinned to the
    reference's own Agent.play / main.train on exactly these hands."""
    g = load(golden_dir, "nfsp_exhaustive.npz")
    T, D = g["kind"].shape
    w = random_nets(9)
    sp = nb.SelfPlay(T, weights=torch.from_numpy(w), seed=3, rl_capacity=1024, sl_capacity=1024, max_steps_per_call=D,
                     variant=variant)
    sp.env.set_hands(g["dealer"], g["cards"], g["policy"])
    forced = np.ascontiguousarray(g["vec"].transpose(1, 0, 2))  # [D, T, 3]; zeros after a hand's last decision
    sp.env.step_counter = 1
    out = sp.rollout(D, insert=False, forced_vec=forced)
    rl, sl = sp.staged()
    b = orc.NfspBatch(T, 3)
    for i in range(T):
        b.inject(i, g["dealer"][i], g["cards"][i], g["policy"][i])
    ref = b.rollout_act(1, D, oracle_nets(nb, w), orc.u32_frac(0.1), orc.u32_frac(0.06), forced_vec=forced)
    tr = out["raw"].cpu().numpy().view(np.uint32)
    assert np.array_equal(tr[0], ref["trace"]["obs"]) and np.array_equal(tr[2], ref["trace"]["misc"])
    for p in range(2):
        assert np.array_equal(canon(rl[p]), canon(ref["rl"][p]))
        assert np.array_equal(canon(sl[p]), canon(ref["sl"][p]))
    # and directly against the fixture for the first hand of every game: RL adds of player 0
    first = np.zeros(T, bool)
    n0 = sum(int((g["rl_player"][i, : g["n_rl"][i]] == 0).sum()) for i in range(T))
    assert len(rl[0]) >= n0


# ------------------------------------------------------------------------------- memories
def _stage(nb, recs, dev):
    d = torch.from_numpy(recs.view(np.int32).reshape(-1, 4).copy()).to(dev)
    n = torch.tensor([len(recs)], dtype=torch.int32, device=dev)
    return d, n


def test_ring_insert_vs_oracle_and_reference(nb, golden_dir):
    g = load(golden_dir, "buffers.npz")
    cap, n = int(g["cap"]), int(g["n_add"])
    recs = np.zeros(n, orc.RL_DT)
    recs["s"], recs["s2"], recs["a"], recs["r"], recs["t"] = g["in_s"], g["in_s2"], g["in_a"], g["in_r"], g["in_t"]
    ring = nb.DeviceRing(cap, seed=1)
    # uneven batches, one of them larger than the ring
    for lo, hi in ((0, 7), (7, 40), (40, 41), (41, 120), (120, n)):
        ring.insert(*_stage(nb, recs[lo:hi], ring.device))
    data, count, total = orc.ring_insert_all(recs, cap)
    assert ring.size() == count == cap and int(ring.total.item()) == total
    got = ring.data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.RL_DT)
    assert np.array_equal(raw16(got), raw16(data))
    # deque order == the reference's buffer contents
    head = total % cap
    order = [(head + i) % cap for i in range(cap)]
    assert np.array_equal(got["s"][order], g["ring_s"]) and np.array_equal(got["r"][order], g["ring_r"])
    # one batch much larger than the ring
    big = nb.DeviceRing(16, seed=1)
    big.insert(*_stage(nb, recs, big.device))
    d2, _, _ = orc.ring_insert_all(recs, 16)
    assert np.array_equal(big.data.cpu().numpy().view(np.uint32), raw16(d2))


@pytest.mark.parametrize("mode", ["R", "reference"])
def test_reservoir_insert_vs_oracle(nb, mode):
    """Algorithm R with Philox keyed by ticket; batches with same-slot collisions resolve like the
    sequential algorithm (largest ticket wins)."""
    cap, seed = 97, 77
    rng = np.random.RandomState(3)
    recs = np.zeros(20000, orc.SL_DT)
    recs["s"] = rng.randint(0, 1 << 30, len(recs))
    recs["a"] = rng.rand(len(recs), 3).astype(np.float32)
    res = nb.DeviceReservoir(cap, seed=seed, mode=mode)
    edges = [0, 5, 96, 97, 98, 500, 501, 9000, 20000]
    for lo, hi in zip(edges[:-1], edges[1:]):
        res.insert(*_stage(nb, recs[lo:hi], res.device))
    data, count, total = orc.reservoir_insert_all(recs, cap, seed, mode=0 if mode == "R" else 1)
    assert res.size() == count and int(res.total.item()) == total == len(recs)
    got = res.data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.SL_DT)
    assert np.array_equal(raw16(got), raw16(data))
    if mode == "reference":  # slot 0 is never replaced (ReservoirBuffer.py:26-28)
        assert got[0].tobytes() == recs[0].tobytes()


def test_sample_indices_and_gather(nb):
    seed = 11
    rng = np.random.RandomState(5)
    for cap, n_ins, batch in ((1000, 400, 256), (1000, 2600, 256), (300, 300, 256), (64, 10, 256), (5000, 5000, 1024)):
        recs = np.zeros(n_ins, orc.RL_DT)
        recs["s"] = rng.randint(0, 1 << 30, n_ins)
        recs["s2"] = rng.randint(0, 1 << 30, n_ins)
        recs["a"] = rng.randint(0, 3, n_ins)
        recs["r"] = rng.randint(-10, 11, n_ins) * 0.5
        recs["t"] = rng.randint(0, 2, n_ins)
        ring = nb.DeviceRing(cap, seed=seed)
        ring.insert(*_stage(nb, recs, ring.device))
        for call in range(3):
            b = min(batch, ring.size())
            s, a, r, s2, t, idx, nn = ring.sample(b)
            count, total = ring.size(), n_ins
            pos = orc.sample_indices(seed, call, count, b)
            head = total % cap if total >= cap else 0
            slots = (head + pos) % cap
            assert int(nn.item()) == b and np.array_equal(idx.cpu().numpy(), slots)
            assert len(set(slots.tolist())) == b
            stored = ring.data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.RL_DT)[slots]
            bits = lambda m: ((m[:, None] >> np.arange(30)) & 1).astype(np.float32)  # noqa: E731
            assert np.array_equal(s.cpu().numpy(), bits(stored["s"])) and np.array_equal(s2.cpu().numpy(), bits(stored["s2"]))
            assert np.array_equal(a.cpu().numpy(), np.eye(3, dtype=np.float32)[stored["a"]])
            assert np.array_equal(r.cpu().numpy(), stored["r"]) and np.array_equal(t.cpu().numpy(), stored["t"].astype(np.float32))
    res = nb.DeviceReservoir(500, seed=seed)
    sl = np.zeros(1200, orc.SL_DT)
    sl["s"] = rng.randint(0, 1 << 30, len(sl))
    sl["a"] = rng.rand(len(sl), 3)
    res.insert(*_stage(nb, sl, res.device))
    s, a, idx, nn = res.sample(256)
    pos = orc.sample_indices(seed, 0, 500, 256)
    assert np.array_equal(idx.cpu().numpy(), pos)
    stored = res.data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.SL_DT)[pos]
    assert np.array_equal(a.cpu().numpy(), stored["a"])


def test_set_weights_from_host_never_writes_through_a_callers_tensor(nb):
    """set_weights(pinned host tensor) copies into a buffer the object owns (no allocation per step); a device tensor
    handed in earlier stays the caller's.  The forward must follow whichever weights were set last."""
    sp = nb.SelfPlay(256, seed=5)
    obs = torch.randint(0, 1 << 30, (64,), dtype=torch.int32, device=sp.device)
    net = torch.randint(0, 4, (64,), dtype=torch.int8, device=sp.device)
    mine = nb.glorot_nets(9, sp.device)
    keep = mine.clone()
    sp.set_weights(mine)
    out_a = sp.forward(obs, net).clone()
    host = [nb.glorot_nets(s, sp.device).cpu().pin_memory() for s in (10, 11)]
    outs = []
    for h in host:
        sp.set_weights(h)
        torch.cuda.synchronize()
        assert torch.equal(mine, keep)          # the caller's tensor was not overwritten
        assert torch.equal(sp.weights.cpu(), h)
        outs.append(sp.forward(obs, net).clone())
    ptr = sp.weights.data_ptr()
    sp.set_weights(host[0])                      # second host call: same device buffer, new contents
    assert sp.weights.data_ptr() == ptr and torch.equal(sp.forward(obs, net), outs[0])
    assert not torch.equal(outs[0], outs[1]) and not torch.equal(out_a, outs[0])
    sp.set_weights(mine)
    assert torch.equal(sp.forward(obs, net), out_a)


def test_rollout_variants_agree_without_debug(nb):
    """Production (non-debug) kernels of both variants leave identical game words, counters and record sets
    whenever no decision is a last-bit near-tie (seeded so that none is)."""
    n, steps = 20_000, 8
    res = []
    for variant in ("cuda", "states", "pairs", "sorted", "tcgen05", "tcgen05_ws"):
        sp = nb.SelfPlay(n, seed=77, eta=0.2, epsilon=0.1, rl_capacity=1 << 12, sl_capacity=1 << 12,
                         max_steps_per_call=steps, variant=variant)
        sp.rollout(steps, insert=False)
        rl, sl = sp.staged()
        res.append((sp.env.state_words().cpu().numpy(), sp.read_stats(), [canon(x) for x in rl]))
    for other in res[1:]:
        assert np.array_equal(res[0][0], other[0]) and res[0][1] == other[1]
        for a, b in zip(res[0][2], other[2]):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("variant", ["states", "pairs", "sorted", "cuda", "tcgen05", "tcgen05_ws"])
@pytest.mark.parametrize("n", [1, 31, 129, 1000])
def test_rollout_launch_batching_and_ragged_sizes(nb, n, variant):
    """One launch of 19 steps == 19 launches of one step (game words, counters, record multisets), for sizes that
    leave phantom lanes in the last warp / tile; 19 > 16 also crosses the small-counter spill."""
    steps = 19
    res = []
    for chunks in ([steps], [1] * steps, [7, 12]):
        sp = nb.SelfPlay(n, seed=31, eta=0.25, epsilon=0.2, rl_capacity=1 << 12, sl_capacity=1 << 12,
                         max_steps_per_call=steps, variant=variant)
        rl = [[], []]
        sl = [[], []]
        for c in chunks:
            sp.rollout(c, insert=False)
            r, s_ = sp.staged()
            for p in range(2):
                rl[p].append(r[p])
                sl[p].append(s_[p])
            sp.counts.zero_()
        res.append((sp.env.state_words().cpu().numpy(), sp.read_stats(),
                    [canon(np.concatenate(x)) for x in rl], [canon(np.concatenate(x)) for x in sl]))
    for other in res[1:]:
        assert np.array_equal(res[0][0], other[0]) and res[0][1] == other[1]
        for a, b in zip(res[0][2] + res[0][3], other[2] + other[3]):
            assert np.array_equal(a, b)
    assert res[0][1]["transitions"] == n * steps and res[0][1]["dropped"] == 0


@pytest.mark.parametrize("variant", ["states", "pairs", "sorted", "cuda", "tcgen05", "tcgen05_ws"])
def test_staging_overflow_drops_and_never_writes_past_a_segment(nb, variant):
    """compute-sanitizer is closed on this pool, so the bounds are checked by hand: staging segments far too small
    for the rollout, canary words behind every segment.  Records that do not fit are counted as dropped, the
    canaries survive, and everything that was staged is a record the full-size run staged too."""
    import ctypes as C

    from nfsp_b200 import _lib
    from nfsp_b200.batched import check, lib, _stream

    n, steps, seed, n_seg, cap, guard = 3000, 8, 5, 8, 40, 8
    if variant == "sorted":  # one cursor per memory: a single dense array, just as short of the records produced
        n_seg, cap = 1, 320
    full = nb.SelfPlay(n, seed=seed, eta=0.3, epsilon=0.1, rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=steps,
                       variant=variant)
    full.rollout(steps, insert=False)
    rl_full, sl_full = full.staged()
    sp = nb.SelfPlay(n, seed=seed, eta=0.3, epsilon=0.1, rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=steps,
                     variant=variant)
    dev = sp.device
    # the kernel addresses segment s at s * cap: a dense [n_seg * cap] array followed by one canary block; inside a
    # segment every slot beyond the claimed count must keep the fill value as well
    dense = [torch.full((n_seg * cap + guard, 4), -7, dtype=torch.int32, device=dev) for _ in range(4)]
    counts = torch.zeros((4, n_seg), dtype=torch.int32, device=dev)
    io = _lib.RolloutIO()
    io.d_rl[0], io.d_rl[1], io.d_sl[0], io.d_sl[1] = (t.data_ptr() for t in dense)
    io.cap_rl, io.cap_sl, io.n_segments = cap, cap, n_seg
    io.d_counts, io.d_stats = counts.data_ptr(), sp.stats.data_ptr()
    io.variant = sp.VARIANTS[variant]
    check(lib().nfsp_rollout(sp.env._h, steps, sp.eta, sp.epsilon, C.byref(io), _stream(dev)))
    torch.cuda.synchronize()
    st = sp.read_stats()
    cnt = counts.cpu().numpy()
    assert st["dropped"] > 0 and st["dropped"] == int(np.maximum(cnt - cap, 0).sum())
    for k, t in enumerate(dense):
        a = t.cpu().numpy()
        assert (a[n_seg * cap:] == -7).all(), "canary behind the last segment overwritten"
        ref = canon(np.concatenate([rl_full[0], rl_full[1]]) if k < 2 else np.concatenate([sl_full[0], sl_full[1]]))
        ref_set = set(map(bytes, ref.view(np.uint8).reshape(len(ref), 16)))
        for s_ in range(n_seg):
            kept = min(int(cnt[k, s_]), cap)
            seg = a[s_ * cap:(s_ + 1) * cap]
            assert (seg[kept:] == -7).all(), "slot beyond the claimed count written"
            for row in seg[:kept]:
                assert row.astype(np.int32).tobytes() in ref_set
    assert np.array_equal(sp.env.state_words().cpu().numpy(), full.env.state_words().cpu().numpy())


def test_memories_after_rollout_match_sequential_oracle(nb):
    """rollout -> flush: ring / reservoir contents equal the oracle fed with the staged records in ticket order."""
    n, steps, seed = 3000, 6, 8
    sp = nb.SelfPlay(n, seed=seed, eta=0.4, epsilon=0.1, rl_capacity=5000, sl_capacity=2000, max_steps_per_call=steps)
    rings = [np.zeros(0, orc.RL_DT), np.zeros(0, orc.RL_DT)]
    ress = [np.zeros(0, orc.SL_DT), np.zeros(0, orc.SL_DT)]
    for _ in range(3):
        sp.rollout(steps, insert=False)
        rl, sl = sp.staged()
        for p in range(2):
            rings[p] = np.concatenate([rings[p], rl[p].astype(orc.RL_DT)])
            ress[p] = np.concatenate([ress[p], sl[p].astype(orc.SL_DT)])
        sp.flush()
    for p in range(2):
        data, count, total = orc.ring_insert_all(rings[p], 5000)
        got = sp.rl[p].data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.RL_DT)
        assert int(sp.rl[p].total.item()) == total and np.array_equal(raw16(got), raw16(data))
        data, count, total = orc.reservoir_insert_all(ress[p], 2000, sp.sl[p].seed)
        got = sp.sl[p].data.cpu().numpy().view(np.uint8).reshape(-1).view(orc.SL_DT)
        assert int(sp.sl[p].total.item()) == total and np.array_equal(raw16(got), raw16(data))
    assert int(sp.counts.sum().item()) == 0


def _rows(a):
    return list(map(bytes, np.ascontiguousarray(a).view(np.uint8).reshape(-1, 16)))


@pytest.mark.parametrize("variant", ["cuda", "states", "pairs", "sorted"])
def test_direct_ring_append_equals_the_staged_insert(nb, variant):
    """direct_rings: the rollout kernel writes the RL records into the rings itself (ticket = atomic add on the ring's
    total, slot = ticket % capacity; replay_buffer.py:30-41).  Launch by launch the records are those the staged path
    moves with nfsp_ring_insert (same seed, same games) and those of the oracle; after the rings have wrapped they hold
    every record of the last launches and the most recent part of the launch the wrap cuts.  The rings start a few
    launches below 2^32 tickets, so the kernel's division-free ticket % capacity meets tickets on both sides of it."""
    from collections import Counter

    n, steps, seed, launches = 3000, 4, 21, 11
    cap = 2 * n * steps  # the smallest ring a launch may not lap: holds about 3.6 launches' worth of one player's records
    mk = lambda direct: nb.SelfPlay(n, seed=seed, eta=0.3, epsilon=0.1, rl_capacity=cap, sl_capacity=1 << 12,  # noqa: E731
                                    max_steps_per_call=steps, variant=variant, direct_rings=direct)
    sd, ss = mk(True), mk(False)
    T0 = 2 ** 32 - cap - 5  # three to four launches' worth of one player's records below 2^32
    for sp in (sd, ss):
        for m in sp.rl:
            m.total.fill_(T0)
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(0.3))
    nets = oracle_nets(nb, nb.glorot_nets(seed, "cuda").cpu().numpy())
    per_launch = [[], []]
    for k in range(launches):
        out = ss.rollout(steps, insert=False, debug=True)
        rl, sl = ss.staged()
        ref = b.rollout_act(1 + k * steps, steps, nets, orc.u32_frac(0.3), orc.u32_frac(0.1), forced_vec=out["vec"].cpu().numpy())
        for p in range(2):
            assert np.array_equal(canon(rl[p]), canon(ref["rl"][p]))
            per_launch[p].append(_rows(rl[p]))
        ss.flush()
        before = [int(sd.rl[p].total.item()) for p in range(2)]
        sd.rollout(steps)  # production kernel, rings written in place, flush() only moves the SL records
        for p in range(2):
            assert int(sd.rl[p].total.item()) - before[p] == len(rl[p]) and int(sd.rl[p].total.item()) == int(ss.rl[p].total.item())
            # the launch's tickets [before, total) land in the same span of slots, ticket % cap, as one multiset
            span = torch.from_numpy((before[p] % cap + np.arange(len(rl[p]))) % cap)
            assert np.array_equal(canon(sd.rl[p].data[span].cpu().numpy()), canon(ss.rl[p].data[span].cpu().numpy())), (k, p)
            assert np.array_equal(canon(sd.rl[p].data[span].cpu().numpy()), canon(rl[p]))
    assert np.array_equal(sd.env.state_words().cpu().numpy(), ss.env.state_words().cpu().numpy())
    assert sd.read_stats() == ss.read_stats() and int(sd.counts.sum().item()) == 0
    for p in range(2):
        assert int(sd.rl[p].total.item()) - T0 > 2 * cap and int(sd.rl[p].total.item()) > 2 ** 32 + cap // 2  # wrapped twice
        for q in range(2):  # the reservoirs went through the staged path in both objects, fed in different orders
            assert int(sd.sl[q].total.item()) == int(ss.sl[q].total.item())
        have = Counter(_rows(sd.rl[p].data.cpu().numpy()))
        room = cap
        for k in reversed(range(launches)):
            want = Counter(per_launch[p][k])
            if len(per_launch[p][k]) <= room:  # a launch the ring still holds completely
                assert not (want - have), (p, k)
                have -= want
                room -= len(per_launch[p][k])
            else:  # the launch the wrap cuts: what is left of the ring comes from it
                assert sum(have.values()) == room and not (have - want), (p, k)
                break


def test_direct_ring_refuses_a_ring_one_launch_could_lap(nb):
    with pytest.raises(ValueError):
        nb.SelfPlay(3000, rl_capacity=2 * 3000 * 4 - 1, sl_capacity=1 << 12, max_steps_per_call=4, variant="sorted", direct_rings=True)
    with pytest.raises(ValueError):
        nb.SelfPlay(3000, rl_capacity=1 << 20, sl_capacity=1 << 12, max_steps_per_call=4, variant="tcgen05", direct_rings=True)
    sp = nb.SelfPlay(3000, rl_capacity=1 << 20, sl_capacity=1 << 12, max_steps_per_call=4, direct_rings="auto")
    assert sp.direct_rings and sp.stage_rl[0].shape[0] == 1


def test_sample_minibatches_slab_equals_per_memory_samples(nb):
    """The one-slab / one-copy minibatch path returns exactly what sample_batch of each memory returns."""
    sp = nb.SelfPlay(4000, seed=11, eta=0.3, epsilon=0.1, rl_capacity=3000, sl_capacity=1500, max_steps_per_call=6)
    sp.rollout(6)
    calls = [(sp.rl[p].sample_calls, sp.sl[p].sample_calls) for p in range(2)]
    views, slab = sp.sample_minibatches(64, to_host=True)
    torch.cuda.synchronize()
    assert not slab.is_cuda and slab.is_pinned()
    for p in range(2):
        sp.rl[p].sample_calls, sp.sl[p].sample_calls = calls[p]
        s, a, r, s2, t, _, n = sp.rl[p].sample(64)
        assert int(n.item()) == 64
        for name, ref in (("s", s), ("a", a), ("r", r), ("s2", s2), ("t", t)):
            assert torch.equal(views[p][name], ref.cpu()), name
        s, a, _, n = sp.sl[p].sample(64)
        assert torch.equal(views[p]["sl_s"], s.cpu()) and torch.equal(views[p]["sl_a"], a.cpu())


def test_counters_ride_in_the_minibatch_slab(nb):
    """sample_minibatches(with_stats=True): the rollout counters live at the tail of the slab from then on, so the one
    device->host copy of the minibatches brings them along; they keep accumulating there."""
    sp = nb.SelfPlay(4096, seed=6, eta=0.3, epsilon=0.1, rl_capacity=1 << 16, sl_capacity=1 << 12, max_steps_per_call=4)
    ref = nb.SelfPlay(4096, seed=6, eta=0.3, epsilon=0.1, rl_capacity=1 << 16, sl_capacity=1 << 12, max_steps_per_call=4)
    sp.rollout(4)
    ref.rollout(4)
    before = sp.read_stats()
    for _ in range(2):
        views, slab = sp.sample_minibatches(64, to_host=True, with_stats=True)
        torch.cuda.synchronize()
        got = slab[-2 * sp.stats.numel():].view(torch.int64)
        assert got.tolist() == sp.stats.cpu().tolist() and sp.read_stats() == ref.read_stats()
        sp.rollout(4)
        ref.rollout(4)
    assert sp.read_stats() == ref.read_stats() and sp.read_stats()["transitions"] == 3 * before["transitions"]


def test_segmented_batches_match_dense_order(nb):
    """A batch staged in segments inserts exactly like the same records staged densely in segment order."""
    rng = np.random.RandomState(8)
    n_seg, seg_cap, cap = 8, 40, 97
    counts = rng.randint(0, seg_cap + 1, n_seg).astype(np.int32)
    counts[3] = 0
    stage = rng.randint(0, 1 << 30, (n_seg, seg_cap, 4)).astype(np.int32)
    dense = np.concatenate([stage[s, : counts[s]] for s in range(n_seg)])
    for kind in ("ring", "res"):
        a = nb.DeviceRing(cap, 3) if kind == "ring" else nb.DeviceReservoir(cap, 3)
        b = nb.DeviceRing(cap, 3) if kind == "ring" else nb.DeviceReservoir(cap, 3)
        for rep in range(3):
            a.insert(torch.from_numpy(stage.reshape(-1, 4)).to(a.device), torch.from_numpy(counts.copy()).to(a.device), seg_cap)
            b.insert(torch.from_numpy(dense).to(b.device), torch.tensor([len(dense)], dtype=torch.int32, device=b.device))
        assert int(a.total.item()) == int(b.total.item()) == 3 * len(dense)
        assert torch.equal(a.data, b.data), kind


def test_dropin_buffers_reference_shapes(nb, golden_dir):
    """utils.replay_buffer.ReplayBuffer / utils.ReservoirBuffer.ReservoirBuffer: the reference's call
    signatures, return shapes and FIFO / saturation behaviour."""
    nb.install_dropin()
    import utils.replay_buffer as RB
    import utils.ReservoirBuffer as RS

    g = load(golden_dir, "buffers.npz")
    cap, n = int(g["cap"]), int(g["n_add"])
    bits = lambda m: ((np.uint32(m) >> np.arange(30)) & 1).astype(np.float64)  # noqa: E731
    rb = RB.ReplayBuffer(cap, 1234)
    for i in range(n):
        rb.add(bits(g["in_s"][i]).reshape(1, 1, 30), np.eye(3)[g["in_a"][i]].reshape(1, 1, 3), float(g["in_r"][i]),
               bits(g["in_s2"][i]).reshape(1, 1, 30), bool(g["in_t"][i]))
        if i in (0, 48, 49, 50, n - 1):
            assert rb.size() == g["ring_sizes"][i]
    s, a, r, s2, t = rb.sample_batch(16)
    assert [s.shape, a.shape, s2.shape] == [tuple(x) for x in g["ring_sample_shapes"]] and r.shape == (16,) and t.shape == (16,)
    stored = {(int(x), float(y)) for x, y in zip(g["ring_s"], g["ring_r"])}
    for k in range(16):
        m = sum(1 << j for j in range(30) if s[k, 0, j])
        assert (m, float(r[k])) in stored
    small = RB.ReplayBuffer(cap, 1234)
    for i in range(5):
        small.add(bits(g["in_s"][i]), np.eye(3)[g["in_a"][i]], 0.5, bits(g["in_s2"][i]), False)
    assert small.sample_batch(16)[0].shape[0] == int(g["ring_small_rows"]) == 5
    rb.clear()
    assert rb.size() == 0
    rs = RS.ReservoirBuffer(cap, 1234, mode="reference")
    for i in range(n):
        rs.add(bits(g["in_s"][i]).reshape(1, 1, 30), g["in_avec"][i].reshape(1, 1, 3))
    assert rs.size() == cap
    s, a = rs.sample_batch(16)
    assert [s.shape, a.shape] == [tuple(x) for x in g["res_sample_shapes"]]
    first = rs.memory.records()[0]
    assert first["s"] == g["res_s"][0] and np.array_equal(first["a"], g["res_a"][0])  # slot 0 never replaced
    with pytest.raises(ValueError):
        rb.add(np.full(30, 0.5), np.eye(3)[0], 0.0, np.zeros(30), False)


def test_dropin_agent_play_flow(nb):
    """agent.agent.Agent.play over leduc.newenv.Env: one hand under main.train's call pattern."""
    nb.install_dropin()
    import agent.agent as agent
    import leduc.newenv as leduc

    env = leduc.Env()
    players = [agent.Agent(None, env.observation_space, env.action_space, "Player%d" % i, env) for i in (0, 1)]
    for hand in range(6):
        dealer = hand & 1
        env.reset(dealer)
        lhand = 1 - dealer
        policy = ["a" if (hand >> 1) & 1 else "b", "b" if hand % 3 else "a"]
        d_s = env.get_state(dealer)[3]
        d_t = l_t = False
        first = True
        for _ in range(8):
            rnd = env.round_index
            if not d_t:
                d_t = players[dealer].play(policy[dealer], dealer, d_s if first else None)
                first = False
            if not l_t:
                l_t = players[lhand].play(policy[lhand], lhand)
            if rnd == env.round_index and not d_t:
                d_t = players[dealer].play(policy[dealer], dealer)
            if d_t and l_t:
                break
        assert d_t and l_t and env.terminated
    assert players[0].played + players[1].played > 0
    assert abs(players[0].reward + players[1].reward) < 1e-9  # zero-sum (newenv.py:344-345)
    assert players[0]._rl_memory.size() + players[1]._rl_memory.size() > 0
    q = players[0].best_response_model.predict(np.zeros((1, 1, 30)))
    pi = players[0].avg_strategy_model.predict(np.zeros((1, 1, 30)))
    assert q.shape == pi.shape == (1, 1, 3) and abs(pi.sum() - 1) < 1e-5 and (q >= 0).all()
    assert hasattr(players[0], "act") and hasattr(players[0], "remember_opponent_behaviour")


def test_rollout_with_weights_from_host_equals_set_weights_then_rollout(nb):
    """nfsp_rollout_with_weights (hand-over + rollout in one library call) against the two calls (deterministic=True: one
    staging segment per block of 32 games, so the order of the records, and with it the reservoirs' contents, is fixed)."""
    n, steps = 5000, 6
    mk = lambda: nb.SelfPlay(n, seed=9, eta=0.3, epsilon=0.1, rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=steps,  # noqa: E731
                             deterministic=True)
    a, b = mk(), mk()
    for k in range(3):
        w = torch.from_numpy(random_nets(20 + k)).pin_memory()
        a.set_weights(w)
        a.rollout(steps)
        b.rollout(steps, weights_host=w)
    torch.cuda.synchronize()
    assert torch.equal(a.weights, b.weights) and torch.equal(a.env.state_words(), b.env.state_words())
    assert a.read_stats() == b.read_stats()
    for p in range(2):
        assert torch.equal(a.rl[p].data, b.rl[p].data) and torch.equal(a.sl[p].data, b.sl[p].data)


def test_rollout_refresh_weights_equals_set_weights_then_rollout(nb):
    """nfsp_rollout_with_weights with h_weights = NULL: the nets were written in place on the device (a learner update); the
    kernels' images and the state table are rebuilt by the call that launches the rollout.  Without the refresh the rollout
    would still act on the previous nets."""
    n, steps = 5000, 6
    mk = lambda: nb.SelfPlay(n, seed=9, eta=0.3, epsilon=0.1, rl_capacity=1 << 12, sl_capacity=1 << 12, max_steps_per_call=steps,  # noqa: E731
                             deterministic=True)
    a, b, stale = mk(), mk(), mk()
    for k in range(3):
        w = torch.from_numpy(random_nets(40 + k)).cuda()
        for sp in (a, b, stale):
            sp.weights.copy_(w)   # in place: the handle's images are now out of date
        a.set_weights(a.weights)
        a.rollout(steps)
        b.rollout(steps, refresh_weights=True)
        stale.rollout(steps)
    torch.cuda.synchronize()
    assert torch.equal(a.env.state_words(), b.env.state_words()) and a.read_stats() == b.read_stats()
    for p in range(2):
        assert torch.equal(a.rl[p].data, b.rl[p].data) and torch.equal(a.sl[p].data, b.sl[p].data)
    assert not torch.equal(a.env.state_words(), stale.env.state_words())  # the stale images played other actions


def test_deterministic_record_order_above_one_warp_per_segment(nb):
    """deterministic=True: one staging segment per block of 32 games, so two runs of one seed leave bit-identical
    memories even where the default layout (1 024 segments shared by several warps) does not fix the order."""
    n, steps = 100_000, 8
    runs = []
    for _ in range(2):
        sp = nb.SelfPlay(n, seed=4, eta=0.3, epsilon=0.1, rl_capacity=150_000, sl_capacity=20_000, max_steps_per_call=steps,
                         deterministic=True)
        assert sp.n_seg >= (n + 31) // 32
        for _ in range(3):
            sp.rollout(steps)
        torch.cuda.synchronize()
        runs.append(sp)
    a, b = runs
    assert a.read_stats() == b.read_stats() and a.read_stats()["dropped"] == 0
    for p in range(2):
        assert int(a.rl[p].total.item()) > 150_000 and int(a.sl[p].total.item()) > 20_000   # wrapped / replacing
        assert torch.equal(a.rl[p].store, b.rl[p].store) and torch.equal(a.sl[p].store, b.sl[p].store)
    with pytest.raises(ValueError):
        nb.SelfPlay(4096, rl_capacity=1 << 20, max_steps_per_call=8, direct_rings=True, deterministic=True)


@pytest.mark.parametrize("variant", ["cuda", "states", "pairs", "sorted", "tcgen05", "tcgen05_ws"])
def test_one_epsilon_per_player(nb, variant):
    """Each Agent of the reference decays its own epsilon (agent.py:78,253): epsilon = (0.6, 0.05) against the oracle;
    the random-vector branch (agent.py:125-128) must fire at each player's own rate."""
    n, steps, seed, eta, eps = 6000, 10, 77, 0.5, (0.6, 0.05)
    w = random_nets(3)
    sp = nb.SelfPlay(n, weights=torch.from_numpy(w), seed=seed, eta=eta, epsilon=eps, rl_capacity=1 << 12, sl_capacity=1 << 12,
                     max_steps_per_call=steps, variant=variant)
    assert sp.epsilons == [0.6, 0.05] and sp.epsilon == 0.6
    out = sp.rollout(steps, insert=False, debug=True)
    rl, sl = sp.staged()
    vec = out["vec"].cpu().numpy()
    b = orc.NfspBatch(n, seed)
    b.reset(0, orc.u32_frac(eta))
    ref = b.rollout_act(1, steps, oracle_nets(nb, w), orc.u32_frac(eta), orc.u32_frac(eps[0]), forced_vec=vec,
                        eps1_u32=orc.u32_frac(eps[1]))
    tr = out["raw"].cpu().numpy().view(np.uint32)
    assert np.array_equal(tr[0], ref["trace"]["obs"]) and np.array_equal(tr[2], ref["trace"]["misc"])
    assert np.abs(vec - ref["vec"]).max() <= TOL   # the oracle draws its random vectors at the same decisions
    for p in range(2):
        assert np.array_equal(canon(rl[p]), canon(ref["rl"][p])) and np.array_equal(canon(sl[p]), canon(ref["sl"][p]))
    same = nb.SelfPlay(n, weights=torch.from_numpy(w), seed=seed, eta=eta, epsilon=0.6, rl_capacity=1 << 12, sl_capacity=1 << 12,
                       max_steps_per_call=steps, variant=variant)
    same.rollout(steps, insert=False)
    assert not np.array_equal(same.env.state_words().cpu().numpy(), sp.env.state_words().cpu().numpy())
