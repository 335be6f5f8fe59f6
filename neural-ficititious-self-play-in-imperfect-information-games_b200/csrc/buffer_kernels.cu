// K3/K4/K5: the agent memories.
//   K3 circular replay insert  (utils/replay_buffer.py:30-41)   16-byte records, streaming copy
//   K4 reservoir insert        (utils/ReservoirBuffer.py:18-28) Philox Algorithm R, two passes
//   K5 minibatch sample        (replay_buffer.py:46-59, ReservoirBuffer.py:33-43) Floyd + gather/expand
// All counts live in device memory: no host synchronisation on the hot path.
#include <cstdlib>

#include "common.cuh"
#include "philox.cuh"

namespace nfsp {

constexpr int kBufThreads = 256;

__device__ __forceinline__ uint64_t mulhi64(uint64_t a, uint64_t b) { return __umul64hi(a, b); }

// ---- staged batches --------------------------------------------------------------------------------
// A batch is n_seg segments of seg_cap slots with a device count each (n_seg = 1: a plain dense array).
// Record i of segment s has batch index prefix(s) + i, where prefix(s) = sum of the counts of the segments
// before s; its ticket is total + that index.
struct Batch {
    const uint4 *recs;
    uint32_t *counts;
    uint32_t n_seg;
    uint64_t seg_cap;
};

// ---- memories of one launch ----------------------------------------------------------------------
// ONE cooperative launch moves the staged batches of up to NFSP_MAX_INSERT_REQS memories (both players' rings and
// reservoirs after a rollout): segment prefixes -> grid barrier -> ring copies + reservoir stamps -> grid barrier ->
// reservoir payloads -> totals and counts committed.  At 64k games the flush used to be five launches on two streams
// (36 us of launch latency for 30 us of work).
struct Mem {
    uint4 *data;        // ring: 16-byte records; reservoir: 32-byte slots {record, u64 stamp, u64 unused}
    uint64_t cap;
    uint64_t *total;
    uint64_t *scratch;  // [0] barrier arrivals, [1] barrier generation, [2 .. 2 + n_seg] exclusive prefix of the counts
    Batch B;
    uint64_t seed;
    int mode;
    int reservoir;
};
struct MemSet {
    Mem m[NFSP_MAX_INSERT_REQS];
    int n;
    uint32_t gx;     // CTAs' worth of work items per segment
    uint64_t chunk;  // records per stamp / write round of the reservoirs
    int small;       // every memory's batch has at most kSmallSegs segments
};
constexpr int kScratchHead = 2;
constexpr uint64_t kResChunk = 1ull << 21;  // records per stamp / write round: the 64 MB of slots they touch stay in L2

// sense-reversing grid barrier on two words of device memory (all CTAs are co-resident: cooperative launch)
__device__ __forceinline__ void grid_sync(uint64_t *ctrl) {
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long *cnt = reinterpret_cast<unsigned long long *>(ctrl);
        volatile unsigned long long *gen = reinterpret_cast<volatile unsigned long long *>(ctrl + 1);
        const unsigned long long g = *gen;
        __threadfence();
        if (atomicAdd(cnt, 1ull) == (unsigned long long)gridDim.x - 1ull) {
            *cnt = 0ull;
            __threadfence();
            atomicAdd(const_cast<unsigned long long *>(gen), 1ull);
        } else {
            while (*gen == g) __nanosleep(32);
        }
        __threadfence();
    }
    __syncthreads();
}

// exclusive prefix of one memory's segment counts (clamped to the segment capacity), by one CTA
__device__ __forceinline__ void scan_counts(const Mem &M) {
    __shared__ unsigned long long s_warp[kBufThreads / 32];
    __shared__ unsigned long long s_run;
    if (threadIdx.x == 0) s_run = 0ull;
    __syncthreads();
    uint64_t *pre = M.scratch + kScratchHead;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t k0 = 0; k0 < M.B.n_seg; k0 += kBufThreads) {
        const uint32_t k = k0 + threadIdx.x;
        unsigned long long c = 0ull;
        if (k < M.B.n_seg) {
            c = M.B.counts[k];
            if (c > M.B.seg_cap) c = M.B.seg_cap;
        }
        unsigned long long incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long before = s_run;
        for (uint32_t w = 0; w < warp; ++w) before += s_warp[w];
        if (k < M.B.n_seg) pre[k] = before + incl - c;
        __syncthreads();
        if (threadIdx.x == kBufThreads - 1) s_run = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) pre[M.B.n_seg] = s_run;
}

// ---- K3 ------------------------------------------------------------------------------------------
constexpr int kRingUnroll = 4;
// slot = ticket % cap; of a batch larger than the ring only the last `cap` records survive (the others
// would be evicted by popleft(), replay_buffer.py:40).  Work item = (segment, x of gx): records x*256 + t, stride gx*256.
__device__ __forceinline__ void ring_item(const Mem &M, uint64_t total, uint32_t seg, uint32_t x, uint32_t gx, uint64_t before,
                                          uint64_t cnt, uint64_t m) {
    const Batch &B = M.B;
    const uint64_t cap = M.cap;
    const uint64_t first = m > cap ? m - cap : 0;
    const uint4 *src = B.recs + (uint64_t)seg * B.seg_cap;
    uint4 *ring = M.data;
    // slot of batch index idx = (total + idx) % cap without a 64-bit division per record: head = total % cap once, then
    // one conditional subtraction (a second reduction only for batches larger than the ring).  kRingUnroll records per
    // thread and iteration, the loads issued before the first store, so several 16-byte reads are in flight per thread.
    const uint64_t head = total % cap;
    const uint64_t stride = (uint64_t)gx * blockDim.x;
    for (uint64_t i0 = x * (uint64_t)blockDim.x + threadIdx.x; i0 < cnt; i0 += stride * kRingUnroll) {
        uint4 v[kRingUnroll];
#pragma unroll
        for (int u = 0; u < kRingUnroll; ++u) {
            const uint64_t i = i0 + (uint64_t)u * stride;
            if (i < cnt) v[u] = __ldcs(src + i);
        }
#pragma unroll
        for (int u = 0; u < kRingUnroll; ++u) {
            const uint64_t i = i0 + (uint64_t)u * stride, idx = before + i;
            if (i < cnt && idx >= first) {
                uint64_t slot = head + idx;
                if (slot >= cap) slot -= cap;
                if (slot >= cap) slot %= cap;
                ring[slot] = v[u];
            }
        }
    }
}

// ---- K4 ------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t reservoir_slot(uint64_t seed, uint64_t ticket, uint64_t cap, int mode) {
    if (ticket < cap) return (int64_t)ticket;  // fill phase, ReservoirBuffer.py:22-24
    const uint64_t u = buffer_u64(seed, ticket, 0, STREAM_RESERVOIR);
    if (mode == 1) {  // the reference's law: j = randrange(1, B+1); replace iff j < B (ReservoirBuffer.py:26-28)
        const uint64_t j = 1u + mulhi64(u, cap);
        return j < cap ? (int64_t)j : -1;
    }
    const uint64_t j = mulhi64(u, ticket + 1u);  // Algorithm R: j ~ U[0, ticket]
    return j < cap ? (int64_t)j : -1;
}

// A reservoir slot is 32 bytes = one DRAM sector: {record, stamp = ticket + 1 of the record that owns it, unused}.
// Two passes over the batch, a grid barrier between them (ReservoirBuffer.py:18-28 for a whole batch at once):
//   stamp  every accepted record raises its slot's stamp to its ticket + 1 (atomicMax keeps the latest)
//   write  the record whose ticket owns the stamp writes the payload -- the outcome of the sequential adds.
// The random 8-byte atomic brings the slot's sector into L2; the stamp check and the 16-byte payload store of the second
// pass then hit that same sector (separate stamp and payload arrays moved four sectors per record: 163 bytes of DRAM
// traffic for 40 algorithmic, ncu r01).  Batches are processed in rounds of kResChunk records so that the sectors of a
// round are still in L2 when its second pass comes.  Both passes are latency-bound with one access in flight per
// thread, so each thread handles kResUnroll records per iteration, all slot draws / atomics / loads issued before the
// first result is needed.
constexpr int kResUnroll = 4;

template <bool kWrite>
__device__ __forceinline__ void reservoir_item(const Mem &M, uint64_t total, uint32_t seg, uint32_t x, uint32_t gx, uint64_t lo,
                                               uint64_t hi, uint64_t before, uint64_t cnt) {
    const Batch &B = M.B;
    if (before >= hi || before + cnt <= lo) return;  // no record of this segment in the round [lo, hi)
    const uint64_t i_lo = lo > before ? lo - before : 0, i_hi = hi - before < cnt ? hi - before : cnt;
    const uint64_t cap = M.cap, seed = M.seed;
    const int mode = M.mode;
    uint4 *res = M.data;
    const uint4 *src = B.recs + (uint64_t)seg * B.seg_cap;
    const uint64_t stride = (uint64_t)gx * blockDim.x;
    for (uint64_t i0 = i_lo + x * (uint64_t)blockDim.x + threadIdx.x; i0 < i_hi; i0 += stride * kResUnroll) {
        int64_t slot[kResUnroll];
#pragma unroll
        for (int u = 0; u < kResUnroll; ++u) {
            const uint64_t i = i0 + (uint64_t)u * stride;
            slot[u] = i < i_hi ? reservoir_slot(seed, total + before + i, cap, mode) : -1;
        }
        if (!kWrite) {
#pragma unroll
            for (int u = 0; u < kResUnroll; ++u)
                if (slot[u] >= 0)
                    atomicMax(reinterpret_cast<unsigned long long *>(res + 2 * slot[u] + 1),
                              (unsigned long long)(total + before + i0 + (uint64_t)u * stride + 1u));
        } else {
            unsigned long long owner[kResUnroll];
#pragma unroll
            for (int u = 0; u < kResUnroll; ++u)
                owner[u] = slot[u] >= 0 ? __ldcg(reinterpret_cast<const unsigned long long *>(res + 2 * slot[u] + 1)) : 0ull;
#pragma unroll
            for (int u = 0; u < kResUnroll; ++u) {
                const uint64_t i = i0 + (uint64_t)u * stride;
                if (slot[u] >= 0 && owner[u] == (unsigned long long)(total + before + i + 1u)) res[2 * slot[u]] = __ldcs(src + i);
            }
        }
    }
}

// work items of memory k: (segment, x) pairs, enumerated CTA-stride by all CTAs of the grid; f(seg, x, before, cnt).
// pre = the memory's exclusive prefix table (n_seg + 1 entries), in global or in shared memory
template <class F>
__device__ __forceinline__ void for_items(const MemSet &S, int k, const uint64_t *pre, bool in_smem, F f) {
    const uint64_t items = (uint64_t)S.m[k].B.n_seg * S.gx;
    for (uint64_t w = blockIdx.x; w < items; w += gridDim.x) {
        const uint32_t seg = (uint32_t)(w / S.gx), x = (uint32_t)(w % S.gx);
        // the table in global memory was written by another CTA before the grid barrier: read it past L1
        const uint64_t before = in_smem ? pre[seg] : __ldcg(pre + seg), next = in_smem ? pre[seg + 1] : __ldcg(pre + seg + 1);
        f(seg, x, before, next - before);
    }
}

constexpr int kSmallSegs = 32;  // up to this many segments per memory every CTA scans the counts itself (one warp each)

__global__ void __launch_bounds__(kBufThreads, 4) insert_kernel(const MemSet S) {
    __shared__ uint64_t s_pre[NFSP_MAX_INSERT_REQS][kSmallSegs + 1];
    uint64_t *ctrl = S.m[0].scratch;
    uint64_t total[NFSP_MAX_INSERT_REQS], m_all[NFSP_MAX_INSERT_REQS];
    const uint64_t *pre[NFSP_MAX_INSERT_REQS];
    const bool small = S.small != 0;
#pragma unroll
    for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k) total[k] = k < S.n ? *S.m[k].total : 0ull;
    if (small) {  // few segments: every CTA scans the counts itself -- no scan CTA, no grid barrier before the first pass
        const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
        if (warp < (uint32_t)S.n) {
            const Mem &M = S.m[warp];
            unsigned long long c = lane < M.B.n_seg ? (unsigned long long)__ldcg(M.B.counts + lane) : 0ull;
            if (c > M.B.seg_cap) c = M.B.seg_cap;
            unsigned long long incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= (uint32_t)o) incl += up;
            }
            s_pre[warp][lane + 1] = incl;
            if (lane == 0) s_pre[warp][0] = 0ull;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k) {
            pre[k] = s_pre[k];
            m_all[k] = k < S.n ? s_pre[k][S.m[k].B.n_seg] : 0ull;
        }
    } else {
        for (int k = blockIdx.x; k < S.n; k += gridDim.x) scan_counts(S.m[k]);
        grid_sync(ctrl);
#pragma unroll
        for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k) {
            pre[k] = k < S.n ? S.m[k].scratch + kScratchHead : nullptr;
            m_all[k] = k < S.n ? __ldcg(pre[k] + S.m[k].B.n_seg) : 0ull;
        }
    }
    uint64_t res_max = 0;  // records of the largest reservoir batch: the number of stamp / write rounds
#pragma unroll
    for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k)
        if (k < S.n && S.m[k].reservoir) res_max = m_all[k] > res_max ? m_all[k] : res_max;
#pragma unroll
    for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k)
        if (k < S.n && !S.m[k].reservoir)
            for_items(S, k, pre[k], small, [&](uint32_t seg, uint32_t x, uint64_t before, uint64_t cnt) {
                ring_item(S.m[k], total[k], seg, x, S.gx, before, cnt, m_all[k]);
            });
    for (uint64_t lo = 0; lo < res_max; lo += S.chunk) {
#pragma unroll
        for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k)
            if (k < S.n && S.m[k].reservoir)
                for_items(S, k, pre[k], small, [&](uint32_t seg, uint32_t x, uint64_t before, uint64_t cnt) {
                    reservoir_item<false>(S.m[k], total[k], seg, x, S.gx, lo, lo + S.chunk, before, cnt);
                });
        grid_sync(ctrl);
#pragma unroll
        for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k)
            if (k < S.n && S.m[k].reservoir)
                for_items(S, k, pre[k], small, [&](uint32_t seg, uint32_t x, uint64_t before, uint64_t cnt) {
                    reservoir_item<true>(S.m[k], total[k], seg, x, S.gx, lo, lo + S.chunk, before, cnt);
                });
    }
    // commit: total += records of the batch, staged counts cleared for the next rollout.  The totals are read in the
    // kernel's first instructions and the counts before the first pass; with few segments a CTA could still be reading
    // the counts when another one is done (no barrier so far if there is no reservoir), hence one more barrier there.
    if (small && res_max == 0) grid_sync(ctrl);
#pragma unroll
    for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k)
        if (k < S.n && (uint32_t)k % gridDim.x == blockIdx.x) {
            const Mem &M = S.m[k];
            for (uint32_t s = threadIdx.x; s < M.B.n_seg; s += blockDim.x) M.B.counts[s] = 0u;
            if (threadIdx.x == 0) *M.total = total[k] + m_all[k];
        }
}

// ---- K5 ------------------------------------------------------------------------------------------
// Floyd's algorithm (1987) for `batch` distinct positions out of `count`: for i = count-batch .. count-1
// draw t ~ U[0,i]; take t unless already taken, else take i.  One CTA: the draws are computed in
// parallel, the "already taken" scan is a warp-parallel compare over the prefix.
constexpr int kMaxBatch = 1024;

// draw / pick: kMaxBatch words of shared memory each; slot_out[m] (shared or global) = storage slot of sample m, -1
// beyond the records held.  Returns the number of samples (min(count, batch)).  All threads of the CTA call it.
template <class SlotT>
__device__ __forceinline__ int floyd_sample(uint64_t seed, uint64_t call_idx, uint64_t total, uint64_t cap, int is_ring,
                                            int batch, uint64_t *draw, uint64_t *pick, SlotT *slot_out) {
    __shared__ int s_collision;
    const uint64_t count = total < cap ? total : cap;
    const int b = (uint64_t)batch < count ? batch : (int)count;
    const uint64_t lo = count - (uint64_t)b;
    if (threadIdx.x == 0) s_collision = 0;
    for (int m = threadIdx.x; m < b; m += blockDim.x)
        draw[m] = mulhi64(buffer_u64(seed, (uint64_t)m, call_idx, STREAM_SAMPLE), lo + (uint64_t)m + 1u);
    __syncthreads();
    // Floyd: step m takes t = draw[m] unless t was taken before, else lo + m (always new).  Every earlier draw is in the
    // set whether it was taken or replaced, so "taken before" = (some earlier draw equals t) or (t = lo + k for an
    // earlier step k that was replaced).  The first term is b*b/2 independent compares; the second refers to ONE
    // earlier step, k = t - lo < m, so the replaced flags are the least fixpoint of dup[m] |= dup[draw[m] - lo], reached
    // by a few parallel sweeps (flags only turn on, references only point backwards) -- same picks as the sequential
    // algorithm, no sequential scan even when draws collide (a 200 000-record ring and 256 draws: 15 % of the calls).
    __shared__ unsigned char s_dup[kMaxBatch];
    for (int m = threadIdx.x; m < b; m += blockDim.x) {
        const uint64_t t = draw[m];
        bool dup = false;
        for (int k = 0; k < m; ++k) dup |= (draw[k] == t);
        if (dup) s_collision = 1;
        s_dup[m] = dup;
    }
    __syncthreads();
    while (s_collision) {  // uniform: every thread reads the same flag between barriers
        __syncthreads();
        if (threadIdx.x == 0) s_collision = 0;
        __syncthreads();
        for (int m = threadIdx.x; m < b; m += blockDim.x) {
            const uint64_t t = draw[m];
            if (!s_dup[m] && t >= lo && t - lo < (uint64_t)m && s_dup[t - lo]) {
                s_dup[m] = 1;
                s_collision = 1;
            }
        }
        __syncthreads();
    }
    for (int m = threadIdx.x; m < b; m += blockDim.x) pick[m] = s_dup[m] ? lo + (uint64_t)m : draw[m];
    __syncthreads();
    // deque position (oldest first) -> storage slot
    const uint64_t head = (is_ring && total >= cap) ? total % cap : 0;
    for (int m = threadIdx.x; m < batch; m += blockDim.x) {
        int64_t slot = -1;
        if (m < b) slot = is_ring ? (int64_t)((head + pick[m]) % cap) : (int64_t)pick[m];
        slot_out[m] = (SlotT)slot;
    }
    return b;
}

// one output element of a sampled RL / SL row (the dense views of replay_buffer.py:46-59 / ReservoirBuffer.py:33-43)
__device__ __forceinline__ void expand_rl(const uint4 rec, int row, int col, float *__restrict__ s, float *__restrict__ a,
                                          float *__restrict__ r, float *__restrict__ s2, float *__restrict__ t) {
    if (col < 30) s[row * 30 + col] = (float)((rec.x >> col) & 1u);
    else if (col < 60) s2[row * 30 + (col - 30)] = (float)((rec.y >> (col - 30)) & 1u);
    else if (col < 63) a[row * 3 + (col - 60)] = ((rec.w & 0xFFu) == (uint32_t)(col - 60)) ? 1.f : 0.f;
    else if (col == 63) r[row] = __uint_as_float(rec.z);
    else t[row] = (float)((rec.w >> 8) & 0xFFu);
}
__device__ __forceinline__ void expand_sl(const uint4 rec, int row, int col, float *__restrict__ s, float *__restrict__ a) {
    if (col < 30) s[row * 30 + col] = (float)((rec.x >> col) & 1u);
    else a[row * 3 + (col - 30)] = __uint_as_float(col == 30 ? rec.y : (col == 31 ? rec.z : rec.w));
}

// sample_batch of several memories in ONE launch: blockIdx.x = memory.  A CTA draws the positions of its memory, fetches
// its share of the sampled records once (one random 16-byte read per row, all in flight together) and expands them
// into out[m] -- an RL block is s[b][30] a[b][3] r[b] s2[b][30] t[b], an SL block s[b][30] a[b][3] (b = batch).  The
// rows of a memory are split over gridDim.y CTAs; each repeats the (cheap) draw.
// Up to kSmallSampleReqs requests travel in the kernel's parameters as they always have; a larger table (the four memories
// of every run of a batch) in a __grid_constant__ copy of the wide table -- the same draws and rows either way.
constexpr int kSmallSampleReqs = 8;
template <int kReqs>
struct SampleTable {
    const uint4 *mem[kReqs];
    const uint64_t *total[kReqs];
    uint64_t cap[kReqs], seed[kReqs], call_idx[kReqs];
    float *out[kReqs];
    uint4 *rec_out[kReqs];  // packed copies of the sampled slots (ring: 16 bytes, reservoir: 32), or null
    int is_ring[kReqs];
};
struct SampleReqs : SampleTable<kSmallSampleReqs> {};
struct SampleReqsWide : SampleTable<NFSP_MAX_SAMPLE_REQS> {};
template <class Reqs>
__device__ __forceinline__ void sample_gather(const Reqs &R, int batch, int64_t *__restrict__ idx_out, uint32_t *__restrict__ n_out) {
    __shared__ uint64_t draw[kMaxBatch];
    __shared__ uint64_t pick[kMaxBatch];
    __shared__ int64_t slot[kMaxBatch];
    __shared__ uint4 s_rec[kMaxBatch];
    const int m = blockIdx.x;
    const int b = floyd_sample(R.seed[m], R.call_idx[m], *R.total[m], R.cap[m], R.is_ring[m], batch, draw, pick, slot);
    __syncthreads();
    const int per = (batch + (int)gridDim.y - 1) / (int)gridDim.y;
    const int row0 = (int)blockIdx.y * per, row1 = min(batch, row0 + per);
    if (threadIdx.x == 0 && blockIdx.y == 0 && n_out) n_out[m] = (uint32_t)b;
    const uint4 *mem = R.mem[m];
    float *o = R.out[m];
    uint4 *ro = R.rec_out[m];
    const int stride = R.is_ring[m] ? 1 : 2;  // reservoir slots are 32 bytes
    for (int k = row0 + threadIdx.x; k < row1; k += blockDim.x) {
        if (idx_out) idx_out[(int64_t)m * batch + k] = slot[k];
        if (o || ro) {
            const uint4 rec = slot[k] >= 0 ? mem[slot[k] * stride] : make_uint4(0, 0, 0, 0);
            if (o) s_rec[k] = rec;
            if (ro) ro[k * stride] = rec;  // same slot geometry as the memory: the learner kernels read either
        }
    }
    if (!o) return;  // positions only (the learner reads the packed records itself)
    __syncthreads();
    const int rows = max(row1 - row0, 0);
    if (R.is_ring[m]) {
        float *s = o, *a = s + 30 * batch, *r = a + 3 * batch, *s2 = r + batch, *t = s2 + 30 * batch;
        for (int e = threadIdx.x; e < rows * 65; e += blockDim.x) {
            const int row = row0 + e / 65, col = e % 65;
            expand_rl(s_rec[row], row, col, s, a, r, s2, t);
        }
    } else {
        float *s = o, *a = s + 30 * batch;
        for (int e = threadIdx.x; e < rows * 33; e += blockDim.x) {
            const int row = row0 + e / 33, col = e % 33;
            expand_sl(s_rec[row], row, col, s, a);
        }
    }
}
__global__ void __launch_bounds__(kBufThreads)
sample_gather_kernel(const SampleReqs R, int batch, int64_t *__restrict__ idx_out, uint32_t *__restrict__ n_out) {
    sample_gather(R, batch, idx_out, n_out);
}
__global__ void __launch_bounds__(kBufThreads)
sample_gather_wide_kernel(const __grid_constant__ SampleReqsWide R, int batch, int64_t *__restrict__ idx_out, uint32_t *__restrict__ n_out) {
    sample_gather(R, batch, idx_out, n_out);
}

__global__ void __launch_bounds__(kBufThreads)
gather_rl_kernel(const uint4 *__restrict__ ring, const int64_t *__restrict__ idx, int batch, float *__restrict__ s,
                 float *__restrict__ a, float *__restrict__ r, float *__restrict__ s2, float *__restrict__ t) {
    // one thread per output element of the widest rows (30 + 30 + 3 + 1 + 1 = 65 columns)
    const int total = batch * 65;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int row = e / 65, col = e - row * 65;
        const int64_t slot = idx[row];
        expand_rl(slot >= 0 ? ring[slot] : make_uint4(0, 0, 0, 0), row, col, s, a, r, s2, t);
    }
}

__global__ void __launch_bounds__(kBufThreads)
gather_sl_kernel(const uint4 *__restrict__ res, const int64_t *__restrict__ idx, int batch, float *__restrict__ s,
                 float *__restrict__ a) {
    const int total = batch * 33;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int row = e / 33, col = e - row * 33;
        const int64_t slot = idx[row];
        expand_sl(slot >= 0 ? res[2 * slot] : make_uint4(0, 0, 0, 0), row, col, s, a);  // 32-byte slots, the record first
    }
}

}  // namespace nfsp

using namespace nfsp;

// validates the requests and fills the kernel's argument
static int make_memset(const nfsp_insert_req *reqs, int n, int want_kind, MemSet &S, int64_t *seg_cap_max) {
    NFSP_CHECK_ARG(reqs && n >= 1 && n <= NFSP_MAX_INSERT_REQS, "1..%d memories per call", NFSP_MAX_INSERT_REQS);
    *seg_cap_max = 0;
    int64_t rows = 0;
    for (int k = 0; k < NFSP_MAX_INSERT_REQS; ++k) S.m[k] = Mem{};
    for (int k = 0; k < n; ++k) {
        const nfsp_insert_req &r = reqs[k];
        NFSP_CHECK_ARG(r.d_mem && r.d_total && r.cap > 0, "bad memory %d", k);
        NFSP_CHECK_ARG(r.d_recs && r.d_counts && r.d_scratch, "null staged batch or scratch %d", k);
        NFSP_CHECK_ARG(r.n_segments >= 1 && r.n_segments <= 65535 && r.seg_cap >= 0, "bad segment geometry %d", k);
        NFSP_CHECK_ARG(r.reservoir == 0 || r.reservoir == 1, "reservoir must be 0 (ring) or 1 (reservoir)");
        NFSP_CHECK_ARG(want_kind < 0 || r.reservoir == want_kind, "memory %d is of the other kind", k);
        if (r.reservoir) NFSP_CHECK_ARG(r.mode == 0 || r.mode == 1, "mode must be 0 (Algorithm R) or 1 (reference law)");
        S.m[k].data = (uint4 *)r.d_mem;
        S.m[k].cap = (uint64_t)r.cap;
        S.m[k].total = r.d_total;
        S.m[k].scratch = r.d_scratch;
        S.m[k].B = Batch{(const uint4 *)r.d_recs, r.d_counts, (uint32_t)r.n_segments, (uint64_t)r.seg_cap};
        S.m[k].seed = r.seed;
        S.m[k].mode = r.mode;
        S.m[k].reservoir = r.reservoir;
        if (r.seg_cap > *seg_cap_max) *seg_cap_max = r.seg_cap;
        rows += r.n_segments;
    }
    S.n = n;
    // work items per segment: about 8 CTAs' worth per SM in total, never more than a segment has 256-record slices
    int64_t g = (*seg_cap_max + kBufThreads - 1) / kBufThreads;
    const int64_t lim = rows >= 148 * 8 ? 1 : (148 * 8 + rows - 1) / rows;
    if (g > lim) g = lim;
    if (g < 1) g = 1;
    S.gx = (uint32_t)g;
    S.small = 1;
    for (int k = 0; k < n; ++k)
        if (reqs[k].n_segments > 32) S.small = 0;
    S.chunk = kResChunk;
#ifdef NFSP_TUNING_HOOKS  // profiles/run_buffers.py with a library built with -DNFSP_TUNING_HOOKS
    if (const char *e = getenv("NFSP_RES_CHUNK")) {
        const long long v = atoll(e);
        if (v >= 1024) S.chunk = (uint64_t)v;
    }
#endif
    return NFSP_OK;
}

// one cooperative launch: every CTA must be resident for the grid barriers
static int launch_insert(MemSet &S, cudaStream_t st) {
    int dev = 0, sms = 0, per_sm = 0;
    NFSP_CUDA(cudaGetDevice(&dev));
    NFSP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    NFSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, insert_kernel, kBufThreads, 0));
    if (per_sm < 1) return set_error(NFSP_E_CUDA, "insert_kernel does not fit an SM");
    if (per_sm > 8) per_sm = 8;
    int64_t items = 0;
    for (int k = 0; k < S.n; ++k) items += (int64_t)S.m[k].B.n_seg * S.gx;
    int64_t grid = (int64_t)sms * per_sm;
    if (items < grid) grid = items;
    if (grid < S.n) grid = S.n;
    void *args[] = {(void *)&S};
    NFSP_CUDA(cudaLaunchCooperativeKernel((const void *)insert_kernel, dim3((unsigned)grid), dim3(kBufThreads), args, 0, st));
    return NFSP_OK;
}

extern "C" int nfsp_insert_multi(const nfsp_insert_req *reqs, int n, void *stream) {
    MemSet S;
    int64_t seg_cap;
    const int rc = make_memset(reqs, n, -1, S, &seg_cap);
    if (rc != NFSP_OK) return rc;
    if (seg_cap == 0) return NFSP_OK;
    return launch_insert(S, (cudaStream_t)stream);
}

extern "C" int nfsp_ring_insert_multi(const nfsp_insert_req *reqs, int n, void *stream) {
    MemSet S;
    int64_t seg_cap;
    const int rc = make_memset(reqs, n, 0, S, &seg_cap);
    if (rc != NFSP_OK) return rc;
    if (seg_cap == 0) return NFSP_OK;
    return launch_insert(S, (cudaStream_t)stream);
}

extern "C" int nfsp_reservoir_insert_multi(const nfsp_insert_req *reqs, int n, void *stream) {
    MemSet S;
    int64_t seg_cap;
    const int rc = make_memset(reqs, n, 1, S, &seg_cap);
    if (rc != NFSP_OK) return rc;
    if (seg_cap == 0) return NFSP_OK;
    return launch_insert(S, (cudaStream_t)stream);
}

extern "C" int nfsp_ring_insert(void *d_ring, int64_t cap, uint64_t *d_total, const void *d_recs, uint32_t *d_counts,
                                int n_segments, int64_t seg_cap, uint64_t *d_scratch, void *stream) {
    nfsp_insert_req r{};
    r.d_mem = d_ring; r.cap = cap; r.d_total = d_total; r.d_recs = d_recs; r.d_counts = d_counts;
    r.n_segments = n_segments; r.seg_cap = seg_cap; r.d_scratch = d_scratch;
    return nfsp_ring_insert_multi(&r, 1, stream);
}

extern "C" int nfsp_reservoir_insert(void *d_res, int64_t cap, uint64_t *d_total, const void *d_recs, uint32_t *d_counts,
                                     int n_segments, int64_t seg_cap, uint64_t seed, int mode, uint64_t *d_scratch,
                                     void *stream) {
    nfsp_insert_req r{};
    r.d_mem = d_res; r.cap = cap; r.d_total = d_total; r.d_recs = d_recs; r.d_counts = d_counts;
    r.n_segments = n_segments; r.seg_cap = seg_cap; r.seed = seed; r.mode = mode; r.d_scratch = d_scratch; r.reservoir = 1;
    return nfsp_reservoir_insert_multi(&r, 1, stream);
}

extern "C" int nfsp_sample_indices(uint64_t seed, uint64_t call_idx, const uint64_t *d_total, int64_t cap,
                                   int is_ring, int batch, int64_t *d_idx, uint32_t *d_n_out, void *stream) {
    nfsp_sample_req r{};  // positions only: no memory is read
    r.d_total = d_total; r.cap = cap; r.seed = seed; r.call_idx = call_idx; r.is_ring = is_ring;
    return nfsp_sample_minibatches(&r, 1, batch, d_idx, d_n_out, stream);
}

template <int kReqs>
static int fill_sample_table(const nfsp_sample_req *reqs, int n_reqs, const int64_t *d_idx, SampleTable<kReqs> &R) {
    for (int m = 0; m < n_reqs; ++m) {
        const bool reads_mem = reqs[m].d_out || reqs[m].d_rec_out;
        NFSP_CHECK_ARG((reqs[m].d_mem || !reads_mem) && reqs[m].d_total && reqs[m].cap > 0, "bad request %d", m);
        NFSP_CHECK_ARG(reqs[m].d_out || reqs[m].d_rec_out || d_idx, "request %d has neither an output block nor an index array", m);
        R.mem[m] = (const uint4 *)reqs[m].d_mem;
        R.total[m] = reqs[m].d_total;
        R.cap[m] = (uint64_t)reqs[m].cap;
        R.seed[m] = reqs[m].seed;
        R.call_idx[m] = reqs[m].call_idx;
        R.out[m] = reqs[m].d_out;
        R.rec_out[m] = (uint4 *)reqs[m].d_rec_out;
        R.is_ring[m] = reqs[m].is_ring;
    }
    return NFSP_OK;
}

extern "C" int nfsp_sample_minibatches(const nfsp_sample_req *reqs, int n_reqs, int batch, int64_t *d_idx, uint32_t *d_n_out,
                                       void *stream) {
    NFSP_CHECK_ARG(reqs && n_reqs >= 1 && n_reqs <= NFSP_MAX_SAMPLE_REQS, "1..%d requests", NFSP_MAX_SAMPLE_REQS);
    NFSP_CHECK_ARG(batch >= 1 && batch <= kMaxBatch, "batch must be in [1,%d]", kMaxBatch);
    const dim3 grid((unsigned)n_reqs, 8u, 1u);
    if (n_reqs <= kSmallSampleReqs) {
        SampleReqs R;
        const int rc = fill_sample_table(reqs, n_reqs, d_idx, R);
        if (rc != NFSP_OK) return rc;
        sample_gather_kernel<<<grid, kBufThreads, 0, (cudaStream_t)stream>>>(R, batch, d_idx, d_n_out);
    } else {
        SampleReqsWide R;
        const int rc = fill_sample_table(reqs, n_reqs, d_idx, R);
        if (rc != NFSP_OK) return rc;
        sample_gather_wide_kernel<<<grid, kBufThreads, 0, (cudaStream_t)stream>>>(R, batch, d_idx, d_n_out);
    }
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

extern "C" int nfsp_gather_rl(const void *d_ring, const int64_t *d_idx, int batch, float *d_s, float *d_a, float *d_r,
                              float *d_s2, float *d_t, void *stream) {
    NFSP_CHECK_ARG(d_ring && d_idx && d_s && d_a && d_r && d_s2 && d_t && batch >= 1, "bad arguments");
    gather_rl_kernel<<<(batch * 65 + kBufThreads - 1) / kBufThreads, kBufThreads, 0, (cudaStream_t)stream>>>(
        (const uint4 *)d_ring, d_idx, batch, d_s, d_a, d_r, d_s2, d_t);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

extern "C" int nfsp_gather_sl(const void *d_res, const int64_t *d_idx, int batch, float *d_s, float *d_a,
                              void *stream) {
    NFSP_CHECK_ARG(d_res && d_idx && d_s && d_a && batch >= 1, "bad arguments");
    gather_sl_kernel<<<(batch * 33 + kBufThreads - 1) / kBufThreads, kBufThreads, 0, (cudaStream_t)stream>>>(
        (const uint4 *)d_res, d_idx, batch, d_s, d_a);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}
