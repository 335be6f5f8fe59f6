"""-m gpu: the memories' inserts and draws at 64-bit counters past 2^32, against the CPU oracle.

Every memory slot and every draw is keyed by a 64-bit counter: a memory's ticket `total` picks ring slots and
reservoir draws, its `sample_calls` keys the minibatch positions.  A long or resumed run carries them past 2^32 (a ring
passes 2^32 tickets within seconds at the benchmarked rate), so each memory here is started mid-life through
load_state_dict -- random held slots, a total near or past 2^32, 2^40 or 2^62 -- and a kernel that dropped a high
word would put a record in the wrong slot, draw another reservoir slot or replay an earlier call's positions."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import orc  # noqa: E402

TOTALS = [2 ** 31 - 1, 2 ** 31 + 1, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 7, 2 ** 62 + 3]
CALLS = [0, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 7]
CAPS = [1, 97, 4096, 200_000]
RES_CHUNK = 1 << 21  # buffer_kernels.cu kResChunk: records per stamp / write round of a reservoir insert
MARK = 0x5EC0DE01    # last word of every batch record (prefilled records never carry it)


@pytest.fixture(scope="module")
def nb():
    import nfsp_b200

    assert torch.cuda.is_available()
    return nfsp_b200


def _prefill(mem, total, rng, calls=0):
    """Starts `mem` mid-life through load_state_dict: random held slots, `total` tickets so far.  A reservoir slot's
    stamp is the ticket + 1 of the record that owns it, so it lies in [1, total]."""
    held = min(total, mem.capacity)
    slots = rng.integers(0, 2 ** 32, (held, mem.slot_words), dtype=np.uint64).astype(np.uint32).view(np.int32)
    slots.view(np.uint32)[slots.view(np.uint32)[:, 3] == MARK, 3] = 0
    if not mem.is_ring:
        slots.view(np.int64)[:, 2] = rng.integers(1, total + 1, held, dtype=np.uint64).astype(np.int64)
    mem.load_state_dict(dict(kind="ring" if mem.is_ring else "reservoir", capacity=mem.capacity, seed=mem.seed,
                             mode=getattr(mem, "mode", 0), total=int(total), sample_calls=int(calls),
                             slots=torch.from_numpy(np.ascontiguousarray(slots))))


def _batch(rng, n, n_seg):
    """n records staged in n_seg segments of uneven counts (-> recs int32 [n_seg * seg_cap, 4], counts, and the records
    in batch order).  Record i of the batch carries i in word 0 and MARK in word 3."""
    cuts = np.sort(rng.integers(0, n + 1, n_seg - 1)) if n_seg > 1 else np.zeros(0, np.int64)
    counts = np.diff(np.concatenate([[0], cuts, [n]])).astype(np.int64)
    seg_cap = int(counts.max()) + 3
    order = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    order[:, 0] = np.arange(n, dtype=np.uint32)
    order[:, 3] = MARK
    recs = np.zeros((n_seg, seg_cap, 4), np.uint32)
    recs[...] = 0xFFFFFFFF  # beyond a segment's count: never read
    at = 0
    for s, c in enumerate(counts):
        recs[s, :c] = order[at:at + c]
        at += c
    return recs.reshape(-1, 4).view(np.int32), counts.astype(np.int32), order, seg_cap


def _stage(recs, counts, dev):
    return torch.from_numpy(recs.copy()).to(dev), torch.from_numpy(counts.copy()).to(dev)


def _as(dt, words):
    return np.ascontiguousarray(words).view(np.uint8).reshape(-1).view(dt).copy()


def _expect(mem, store0, total0, order):
    """The oracle's store after inserting `order` into the memory held as store0 (int32 [cap, slot_words]) at total0.
    Reservoir stamps: the slot's prefilled stamp unless a batch record owns it, then that record's ticket + 1."""
    cap = mem.capacity
    if mem.is_ring:
        data, _, total = orc.ring_insert_all(_as(orc.RL_DT, order), cap, total0=total0,
                                             data=_as(orc.RL_DT, store0))
        return np.ascontiguousarray(data).view(np.int32).reshape(cap, 4), total
    data, _, total = orc.reservoir_insert_all(_as(orc.SL_DT, order), cap, mem.seed, mem.mode, total0=total0,
                                              data=_as(orc.SL_DT, store0[:, :4]))
    want = store0.copy()
    want[:, :4] = np.ascontiguousarray(data).view(np.int32).reshape(cap, 4)
    words = want.view(np.uint32)
    batch = words[:, 3] == MARK
    stamps = want.view(np.int64)[:, 2]
    stamps[batch] = total0 + words[batch, 0].astype(np.int64) + 1
    return want, total


def _check_insert(mem, want, total, tag):
    torch.cuda.synchronize()
    assert int(mem.total.item()) == total, tag
    got = mem.store.cpu().numpy()
    if not np.array_equal(got, want):
        bad = np.nonzero((got != want).any(1))[0]
        raise AssertionError("%s: %d slots differ, first %s: got %s want %s" % (tag, len(bad), bad[:4], got[bad[0]],
                                                                               want[bad[0]]))


def _new(nb, kind, cap, seed):
    from nfsp_b200.batched import DeviceReservoir, DeviceRing

    if kind == "ring":
        return DeviceRing(cap, seed=seed)
    return DeviceReservoir(cap, seed=seed, mode="R" if kind == "R" else "reference")


# ------------------------------------------------------------------------------- staged inserts
@pytest.mark.parametrize("kind", ["ring", "R", "reference"])
@pytest.mark.parametrize("cap", CAPS)
def test_staged_insert_past_2_32_vs_oracle(nb, kind, cap):
    """Both segment paths (5 segments: every CTA scans the counts; 40: one scan CTA and a grid barrier), each at every
    total; rings also take a batch larger than themselves."""
    rng = np.random.default_rng(cap * 7 + len(kind))
    mem = _new(nb, kind, cap, seed=0xC0FFEE + cap)
    for total0 in TOTALS:
        for n_seg, n in ((5, min(3 * cap + 17, 5000)), (40, min(cap + 4000, 50_000)), (3, cap + 1000)):
            if kind != "ring" and n > 50_000:
                continue
            _prefill(mem, total0, rng)
            store0 = mem.store.cpu().numpy()
            recs, counts, order, seg_cap = _batch(rng, n, n_seg)
            want, total = _expect(mem, store0, total0, order)
            mem.insert(*_stage(recs, counts, mem.device), seg_cap=seg_cap)
            _check_insert(mem, want, total, (kind, cap, total0, n_seg, n))


@pytest.mark.parametrize("kind,cap", [("R", 200_000), ("reference", 4096)])
def test_reservoir_batch_of_several_stamp_rounds_crossing_2_32(nb, kind, cap):
    """A batch of more than kResChunk records (several stamp / write rounds) whose tickets cross 2^32 in its middle: the
    stamps are 64-bit tickets + 1 on both sides, and the round that straddles 2^32 resolves its collisions like the
    sequential algorithm."""
    rng = np.random.default_rng(11)
    mem = _new(nb, kind, cap, seed=987654321)
    n = 2 * RES_CHUNK + 12345
    total0 = 2 ** 32 - RES_CHUNK - 777
    _prefill(mem, total0, rng)
    store0 = mem.store.cpu().numpy()
    recs, counts, order, seg_cap = _batch(rng, n, 6)
    want, total = _expect(mem, store0, total0, order)
    assert total0 < 2 ** 32 < total and n > 2 * RES_CHUNK
    mem.insert(*_stage(recs, counts, mem.device), seg_cap=seg_cap)
    _check_insert(mem, want, total, (kind, cap))


def test_four_memories_in_one_insert_launch_at_different_totals(nb):
    """nfsp_insert_multi with both rings and both reservoir modes, each at its own total, in both segment paths."""
    from nfsp_b200._lib import InsertReq, check
    from nfsp_b200.batched import _stream

    rng = np.random.default_rng(5)
    kinds = [("ring", 4096, 2 ** 32 - 100), ("R", 97, 2 ** 40 + 7), ("reference", 4096, 2 ** 32 - 1000),
             ("ring", 97, 2 ** 62 + 3)]
    for n_seg in (8, 36):
        mems, wants, keep = [], [], []
        arr = (InsertReq * 4)()
        for r, (kind, cap, total0) in zip(arr, kinds):
            mem = _new(nb, kind, cap, seed=1000 + cap + len(kind))
            _prefill(mem, total0, rng)
            recs, counts, order, seg_cap = _batch(rng, 3000, n_seg)
            wants.append(_expect(mem, mem.store.cpu().numpy(), total0, order))
            d_recs, d_counts = _stage(recs, counts, mem.device)
            keep += [d_recs, d_counts]
            r.d_mem, r.cap, r.d_total = mem.store.data_ptr(), mem.capacity, mem.total.data_ptr()
            r.d_scratch, r.d_recs, r.d_counts = mem.scratch(n_seg).data_ptr(), d_recs.data_ptr(), d_counts.data_ptr()
            r.n_segments, r.seg_cap, r.seed = n_seg, seg_cap, mem.seed
            r.mode, r.reservoir = getattr(mem, "mode", 0), 0 if mem.is_ring else 1
            mems.append(mem)
        check(nb.lib().nfsp_insert_multi(arr, 4, _stream(mems[0].device)))
        for k, (mem, (want, total)) in enumerate(zip(mems, wants)):
            _check_insert(mem, want, total, (n_seg, kinds[k]))
        assert all(int(c.sum().item()) == 0 for c in keep[1::2])  # the staged counts are consumed


# ------------------------------------------------------------------------------- sampling
def _want_sample(mem, store, total, call, b):
    """(slots, n, dense rows) the oracle names: positions of orc.sample_indices, a ring's from its head."""
    cap = mem.capacity
    count = min(total, cap)
    pos = orc.sample_indices(mem.seed, call, count, b)
    head = total % cap if (mem.is_ring and total >= cap) else 0
    slots = (head + pos) % cap if mem.is_ring else pos
    n = len(slots)
    rec = np.zeros((b, 4), np.uint32)
    rec[:n] = store.view(np.uint32)[slots, :4]
    bits = lambda m: ((m[:, None] >> np.arange(30, dtype=np.uint32)) & 1).astype(np.float32)  # noqa: E731
    if mem.is_ring:
        a = ((rec[:, 3] & 0xFF)[:, None] == np.arange(3)).astype(np.float32)
        r = rec[:, 2].view(np.float32)
        t = ((rec[:, 3] >> 8) & 0xFF).astype(np.float32)
        dense = np.concatenate([bits(rec[:, 0]).ravel(), a.ravel(), r, bits(rec[:, 1]).ravel(), t])
    else:
        dense = np.concatenate([bits(rec[:, 0]).ravel(), rec[:, 1:4].view(np.float32).ravel()])
    full = np.full(b, -1, np.int64)
    full[:n] = slots
    return full, n, dense.view(np.int32)


@pytest.mark.parametrize("kind", ["ring", "R"])
@pytest.mark.parametrize("cap", CAPS)
def test_sample_and_gather_past_2_32_vs_oracle(nb, kind, cap):
    """ring.sample / res.sample (nfsp_sample_indices + gather) at every total and call index."""
    rng = np.random.default_rng(cap + 3)
    mem = _new(nb, kind, cap, seed=0xABCDEF0123456789 + cap)
    b = 256
    for total in TOTALS + [cap // 2 + 1]:
        _prefill(mem, total, rng)
        store = mem.store.cpu().numpy()
        for call in CALLS:
            mem.sample_calls = call
            out = mem.sample(b)
            idx, n = out[-2], out[-1]
            rows = out[:-2]
            dense = torch.cat([x.reshape(-1) for x in rows]).cpu().numpy().view(np.int32)
            slots, nn, want = _want_sample(mem, store, total, call, b)
            assert int(n.item()) == nn and np.array_equal(idx.cpu().numpy(), slots), (total, call)
            assert np.array_equal(dense, want), (total, call)  # bit patterns: random words may be NaNs
            assert mem.sample_calls == call + 1


def _minibatches(nb, mems, calls, b):
    """One nfsp_sample_minibatches launch over mems at the given call indices -> (idx [k, b], n [k], rows per memory)."""
    from nfsp_b200._lib import SampleReq, check
    from nfsp_b200.batched import _ptr, _stream

    dev = mems[0].device
    reqs = (SampleReq * len(mems))()
    outs = []
    for q, m, call in zip(reqs, mems, calls):
        m.sample_req(q)
        q.call_idx = call
        out = torch.full((b * (65 if m.is_ring else 33),), float("nan"), dtype=torch.float32, device=dev)
        q.d_out = out.data_ptr()
        outs.append(out)
    idx = torch.empty((len(mems), b), dtype=torch.int64, device=dev)
    cnt = torch.empty(len(mems), dtype=torch.int32, device=dev)
    check(nb.lib().nfsp_sample_minibatches(reqs, len(mems), b, _ptr(idx), _ptr(cnt), _stream(dev)))
    torch.cuda.synchronize()
    return idx.cpu().numpy(), cnt.cpu().numpy(), [o.cpu().numpy().view(np.int32) for o in outs]


@pytest.mark.parametrize("n_reqs", [4, 12])
def test_sample_minibatches_past_2_32_vs_oracle(nb, n_reqs):
    """Four requests (the parameter-block kernel) and twelve (the __grid_constant__ wide kernel), memories at totals
    below and above 2^32 mixed in one launch, each at its own call index."""
    rng = np.random.default_rng(n_reqs)
    b = 128
    mems, totals, calls = [], [], []
    for k in range(n_reqs):
        kind = ("ring", "R", "ring", "reference")[k % 4]
        cap = CAPS[k % len(CAPS)] if k % 3 else 4096
        mem = _new(nb, kind, cap, seed=77 + 13 * k)
        total = [2 ** 32 + 1, 1000, 2 ** 40 + 7, 2 ** 32 - 1, 2 ** 62 + 3, 2 ** 31 + 1][k % 6]
        _prefill(mem, total, rng)
        mems.append(mem)
        totals.append(total)
        calls.append(CALLS[(k * 5) % len(CALLS)] + k // len(CALLS))
    idx, cnt, rows = _minibatches(nb, mems, calls, b)
    for k, m in enumerate(mems):
        slots, n, want = _want_sample(m, m.store.cpu().numpy(), totals[k], calls[k], b)
        assert int(cnt[k]) == n and np.array_equal(idx[k], slots), k
        assert np.array_equal(rows[k], want), k


def test_call_2_32_plus_k_draws_other_positions_than_call_k(nb):
    """The device keys a draw by the whole 64-bit call index: call 2^32 + k is not call k again."""
    from nfsp_b200.batched import DeviceRing

    cap, total = 200_000, 2 ** 32 + 5
    ring = DeviceRing(cap, seed=31)
    _prefill(ring, total, np.random.default_rng(0))
    got = {}
    for call in (3, 2 ** 32 + 3, 2 ** 40 + 3):
        ring.sample_calls = call
        got[call] = ring.sample_slots(256)[0].cpu().numpy()
        assert np.array_equal(got[call], (total % cap + orc.sample_indices(31, call, cap, 256)) % cap), call
    assert not np.array_equal(got[3], got[2 ** 32 + 3]) and not np.array_equal(got[3], got[2 ** 40 + 3])


# ------------------------------------------------------------------------------- refusal
def test_env_refuses_game_ids_past_2_32(nb):
    """Philox counter word 0 holds the low half of the global game id: a shard reaching game 2^32 would replay game 0's
    deals, so nfsp_env_create refuses game0 + n_games > 2^32 (and accepts the shard that ends exactly there)."""
    with pytest.raises(nb.NfspError, match="2\\^32"):
        nb.BatchedNfspEnv(8, seed=1, game0=2 ** 32 - 7)
    with pytest.raises(nb.NfspError, match="2\\^32"):
        nb.BatchedLegacyEnv(1, seed=1, game0=2 ** 32)
    env = nb.BatchedNfspEnv(8, seed=1, game0=2 ** 32 - 8)
    env.reset()
    torch.cuda.synchronize()
    env.close()
