"""The 64-bit counters past 2^32, without a GPU: every random draw and memory slot is keyed by a 64-bit counter (a
memory's ticket `total`, the env step counter, a memory's `sample_calls`), and long or resumed runs carry them past
2^32.  Plain-Python restatements of Philox4x32-10, the reservoir slot, Floyd's sample and the ring slot pin the C
oracle at such counters, and the device's division-free ring modulo (rollout_common.cuh ring_slot) is restated and
checked against `ticket % cap` over the whole 64-bit range.  The GPU side (tests/test_gpu_counters.py) holds the
kernels to the oracle at the same counters."""
import random

import numpy as np
import pytest

from oracle import orc

M32, M64 = 2 ** 32 - 1, 2 ** 64 - 1
STREAM_RESERVOIR, STREAM_SAMPLE = 2, 3
# counters where a dropped or truncated high word shows: both sides of 2^31 and 2^32, and far beyond
COUNTERS = [2 ** 31 - 1, 2 ** 31 + 1, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 7, 2 ** 62 + 3]
CALLS = [0, 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 7, 2 ** 62 + 3]


# ----------------------------------------------------------------------------- restatements
def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11) on Python ints."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & M32, (p0 >> 32) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


def buffer_u64(seed, idx, call, stream):
    """The memories' draw: counter (idx, idx >> 32 | call >> 32, call, stream), key = the seed's two halves."""
    assert idx <= M32 or call <= M32  # no stream uses both high halves
    o = philox4x32_10((idx & M32, ((idx >> 32) | (call >> 32)) & M32, call & M32, stream), (seed & M32, seed >> 32))
    return o[0] | (o[1] << 32)


def mulhi64(a, b):
    return ((a & M64) * (b & M64)) >> 64


def reservoir_slot(seed, ticket, cap, mode):
    """ReservoirBuffer.py:18-28.  Fill phase, then mode 0: Algorithm R (j ~ U[0, ticket], replace iff j < cap); mode
    1: the reference's law (j = randrange(1, cap + 1), replace iff j < cap).  -1: the record is dropped."""
    if ticket < cap:
        return ticket
    u = buffer_u64(seed, ticket, 0, STREAM_RESERVOIR)
    j = 1 + mulhi64(u, cap) if mode == 1 else mulhi64(u, ticket + 1)
    return j if j < cap else -1


def floyd(seed, call, count, batch):
    """random.sample(range(count), batch) as Floyd's algorithm, draw m keyed by (seed; m, call)."""
    b = min(batch, count)
    out = []
    for m, i in enumerate(range(count - b, count)):
        t = mulhi64(buffer_u64(seed, m, call, STREAM_SAMPLE), i + 1)
        out.append(i if t in out else t)
    return out


def ring_head(total, cap):
    """Storage slot of the oldest record a ring holds (deque position 0)."""
    return total % cap if total >= cap else 0


def ring_slot_magic(ticket, cap):
    """rollout_common.cuh ring_slot: q = umulhi(ticket, floor((2^64 - 1) / cap)) is floor(ticket / cap) or one less,
    so ticket - q * cap needs at most one conditional subtraction."""
    magic = M64 // cap
    q = mulhi64(ticket, magic)
    r = (ticket - q * cap) & M64
    if r >= cap:
        r -= cap
    return r


# ----------------------------------------------------------------------------- Philox
def test_philox_restatement_known_answers():
    """The Random123 known-answer vectors that pin the oracle's Philox (test_oracle_golden.py) pin this one too."""
    kat = [(([0, 0, 0, 0], [0, 0]), [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
           (([M32] * 4, [M32] * 2), [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
           (([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]),
            [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])]
    for (ctr, key), want in kat:
        assert list(philox4x32_10(ctr, key)) == want
        assert [int(x) for x in orc.philox(ctr, key)] == want


def test_philox_restatement_equals_the_oracle_on_high_counter_words():
    rng = random.Random(3)
    for _ in range(200):
        ctr = [rng.getrandbits(32) for _ in range(4)]
        key = [rng.getrandbits(32) for _ in range(2)]
        assert [int(x) for x in orc.philox(ctr, key)] == list(philox4x32_10(ctr, key))


def test_sample_stream_below_2_32_calls_is_the_one_it_always_was():
    """Call indices below 2^32 and every reservoir draw (call 0) keep the counter they always had: checkpoints,
    golden files and dumped outputs do not change.  Calls at and above 2^32 get a counter of their own."""
    def old(seed, idx, call, stream):
        o = philox4x32_10((idx & M32, idx >> 32, call & M32, stream), (seed & M32, seed >> 32))
        return o[0] | (o[1] << 32)

    for seed in (0, 1234, 2 ** 64 - 5):
        for call in (0, 1, 2 ** 31, 2 ** 32 - 1):
            for m in (0, 1, 1023):
                assert buffer_u64(seed, m, call, STREAM_SAMPLE) == old(seed, m, call, STREAM_SAMPLE)
        for t in COUNTERS:
            assert buffer_u64(seed, t, 0, STREAM_RESERVOIR) == old(seed, t, 0, STREAM_RESERVOIR)
        for k in (0, 1, 7, 2 ** 31):
            assert buffer_u64(seed, 0, 2 ** 32 + k, STREAM_SAMPLE) != buffer_u64(seed, 0, k, STREAM_SAMPLE)


# ----------------------------------------------------------------------------- reservoir slots
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("cap", [1, 97, 4096, 200_000])
def test_oracle_reservoir_slot_past_2_32(cap, mode):
    """orc.reservoir_slot against the restatement on runs of tickets around each counter, the fill phase's edge too."""
    seed = 0x9E3779B97F4A7C15
    tickets = [t for c in COUNTERS for t in range(c - 3, c + 4)] + list(range(cap - 2, cap + 3))
    for t in tickets:
        if t >= 0:
            assert orc.reservoir_slot(seed, t, cap, mode) == reservoir_slot(seed, t, cap, mode), (t, cap, mode)


def test_reservoir_slot_keys_the_whole_ticket():
    """Tickets t and t + 2^32 draw differently: a slot computed from (uint32_t)ticket would not."""
    seed, cap = 77, 4096
    hi = [reservoir_slot(seed, 2 ** 32 + t, cap, 1) for t in range(cap, cap + 256)]
    lo = [reservoir_slot(seed, t, cap, 1) for t in range(cap, cap + 256)]
    assert hi != lo
    # Algorithm R past 2^32 keeps a record with probability cap / (ticket + 1): about 1e-6 here, so it must drop
    # nearly all -- a draw scaled by a truncated ticket + 1 would keep them all
    kept = sum(reservoir_slot(seed, t, cap, 0) >= 0 for t in range(2 ** 32, 2 ** 32 + 2000))
    assert kept <= 2


@pytest.mark.parametrize("mode", [0, 1])
def test_oracle_reservoir_insert_mid_life(mode):
    seed, cap = 11, 97
    rng = np.random.default_rng(4)
    for total0 in COUNTERS:
        recs = np.zeros(300, orc.SL_DT)
        recs["s"] = rng.integers(0, 2 ** 30, 300)
        data0 = np.zeros(cap, orc.SL_DT)
        data0["s"] = rng.integers(0, 2 ** 30, cap)
        data, count, total = orc.reservoir_insert_all(recs, cap, seed, mode, total0=total0, data=data0.copy())
        want = data0.copy()
        for i in range(len(recs)):
            j = reservoir_slot(seed, total0 + i, cap, mode)
            if j >= 0:
                want[j] = recs[i]
        assert total == total0 + 300 and count == cap
        assert data.tobytes() == want.tobytes(), total0


# ----------------------------------------------------------------------------- sampling
@pytest.mark.parametrize("count,batch", [(1, 4), (97, 97), (4096, 256), (200_000, 128)])
def test_oracle_sample_indices_at_high_calls(count, batch):
    seed = 0xDEADBEEF12345678
    for call in CALLS:
        got = orc.sample_indices(seed, call, count, batch).tolist()
        want = floyd(seed, call, count, batch)
        assert got == want, call
        assert len(set(got)) == len(got) == min(count, batch) and all(0 <= x < count for x in got)


def test_call_2_32_plus_k_is_not_call_k():
    """The whole 64-bit call index keys the draw: call 2^32 + k must not replay call k's positions."""
    seed = 5
    for k in (0, 1, 12345, 2 ** 31):
        for hi in (2 ** 32, 2 ** 40):
            a = orc.sample_indices(seed, hi + k, 200_000, 256)
            b = orc.sample_indices(seed, k, 200_000, 256)
            assert not np.array_equal(a, b), (hi, k)


@pytest.mark.parametrize("cap", [1, 97, 4096, 200_000])
def test_sampled_ring_slots_past_2_32(cap):
    """A ring's sampled deque position p (oldest first) lives in slot (head + p) % cap, head = total % cap once
    full: restated against the FIFO oracle's storage at every total, so the head of a total past 2^32 is right."""
    rng = np.random.default_rng(cap)
    for total in COUNTERS:
        recs = np.zeros(cap + 5, orc.RL_DT)
        recs["s"] = np.arange(cap + 5) + 1  # record of ticket total0 + i carries i + 1
        total0 = total - len(recs)
        data, _, t = orc.ring_insert_all(recs, cap, total0=total0, data=np.zeros(cap, orc.RL_DT))
        assert t == total
        call = int(rng.integers(0, 2 ** 63))
        for p, pos in enumerate(orc.sample_indices(3, call, cap, 64).tolist()):
            slot = (ring_head(total, cap) + pos) % cap
            # deque position pos holds the record of ticket total - cap + pos
            assert int(data["s"][slot]) == total - cap + pos - total0 + 1, (total, p)


# ----------------------------------------------------------------------------- rings
@pytest.mark.parametrize("cap", [1, 97, 4096, 200_000])
def test_oracle_ring_insert_mid_life(cap):
    """orc.ring_insert_all started at total0 against the restatement slot = ticket % cap, batches smaller and larger
    than the ring."""
    rng = np.random.default_rng(7)
    for total0 in COUNTERS:
        for n in (3, cap + 50):
            recs = np.zeros(n, orc.RL_DT)
            recs["s"] = rng.integers(0, 2 ** 30, n)
            recs["r"] = rng.standard_normal(n)
            data0 = np.zeros(cap, orc.RL_DT)
            data0["s2"] = rng.integers(0, 2 ** 30, cap)
            data, count, total = orc.ring_insert_all(recs, cap, total0=total0, data=data0.copy())
            want = data0.copy()
            for i in range(n):
                want[(total0 + i) % cap] = recs[i]
            assert total == total0 + n and count == cap
            assert data.tobytes() == want.tobytes(), (total0, n)


RING_CAPS = [1, 2, 3, 97, 24_000, 200_000, 2 ** 31 - 1, 2 ** 32 - 1]


@pytest.mark.parametrize("cap", RING_CAPS)
def test_division_free_ring_slot_is_ticket_mod_cap(cap):
    """The direct-ring append's slot (rollout_common.cuh ring_slot) equals ticket % cap for every 64-bit ticket."""
    rng = random.Random(cap)
    tickets = [0, cap - 1, cap, cap + 1, 2 * cap - 1, 2 * cap, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 63 - 1, 2 ** 63,
               M64, M64 - cap]
    tickets += [c + d for c in COUNTERS for d in (-1, 0, 1)]
    tickets += [rng.getrandbits(64) for _ in range(2000)] + [rng.getrandbits(rng.randint(1, 64)) for _ in range(2000)]
    # the tickets just below a multiple of cap are where floor(ticket * magic / 2^64) falls one short
    tickets += [(k * cap - 1) & M64 for k in (1, 2, 3, 2 ** 20 + 1, M64 // cap)]
    for t in tickets:
        if 0 <= t <= M64:
            assert ring_slot_magic(t, cap) == t % cap, (t, cap)
