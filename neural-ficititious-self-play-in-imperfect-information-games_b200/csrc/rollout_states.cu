// K2, variant 6: the fused rollout over a table of the nets' outputs on every decision state.
//
// Under main.train's turn order (the precondition of the factorised first layer, rollout_tables.cuh) the observation a
// net sees at a decision is one of 702 values: the actor's card, the dealer and the betting sequence so far in round 0
// (54), or card, public card, dealer, the finished round-0 sequence and the round-1 sequence so far (648).  A net is a
// pure function of the observation, so its three outputs on all of them -- computed by states_pack_kernel from the SAME
// table image and with the same operations as variant 1 (two rows added, relu, FFMA2 second layer, head; the 16
// hidden-unit quads summed in four interleaved groups) every time the weights change -- stand for the 8.4 M forwards
// of a 2^20-game x 8-step launch.  A decision then costs ONE 16-byte shared-memory read instead of variant 1's 80.
//
// What is left is the game logic, Philox and the record append, and the game logic runs on the state machine of the
// env-only kernel (nfsp_fsm.cuh, the rollout image): a step is two 16-byte reads of the entry (row, raw action) whose
// words are used as loaded -- no field extraction, no index formula for the state table (each player carries its
// address, moved by the entry).  The records, game words and counters are those of variant 1 run on the same score
// vectors; the score vectors differ from variant 1's only by the summation order of a lane's rotation (held to 1e-5 of
// the CPU restatement in tests/test_gpu_act.py and tests/test_gpu_baseline_sizes.py).  The append is this kernel's own:
// warp-private buffers in shared memory (below).
#include "nfsp_fsm.cuh"
#include "rollout_fast.cuh"
#include "rollout_tables.cuh"
#include "ptx_helpers.cuh"

namespace nfsp {

// Table slot of a decision state: x * 18 + sigma, x = ((card * 3 + public card) * 2 + dealer) * 4 + finished round-0
// sequence, sigma = 9 * round + sequence id.  One formula for both rounds, no branch in the step loop: round 0 does not see
// the public card and has no finished sequence yet (f = 0), so its 54 states are stored once per public card; slots with
// round 0 and f != 0 are never read.  702 distinct states in 72 * 18 = 1 296 slots per net.
constexpr int kNetStates = 72 * 18;
constexpr int kStateQuads = 4 * kNetStates;      // one float4 {o0, o1, o2, action word} per net and slot
constexpr int kStateBytes = kStateQuads * 16;    // 82 944
static_assert(kStateBytes % 16 == 0, "bulk copies move multiples of 16 bytes");
static_assert(kNetStates == fsm::kNetSlots, "the rollout image addresses this table");

// action word of a score vector: np.argmax (first maximum) * the entry size (the entry's offset in its row) | the
// non-zero flag (np.average != 0, agent.py:134) at its bit in the P word
__device__ __forceinline__ uint32_t score_word(float v0, float v1, float v2) {
    const uint32_t an = score_action(v0, v1, v2);
    return (an & 3u) * (uint32_t)fsm::kEntryBytes | (an >> 2) << 15;
}
constexpr uint32_t kWordEntry = 0x60u, kWordNz = 1u << 15;

// table slot -> rows of the factorised first layer (the inverse of the index the rollout computes)
__device__ __forceinline__ void state_rows(int s, uint32_t &xrow, uint32_t &yrow) {
    const uint32_t sg = (uint32_t)s % 18u, x = (uint32_t)s / 18u, dl = (x >> 2) & 1u;
    xrow = sg >= 9u ? 3u + x : x / 24u;  // round 0: the private card alone
    yrow = 75u + dl * 18u + sg;
}

// One table slot per FOUR lanes: lane j of a quad takes hidden-unit quads j, j + 4, j + 8, j + 12 of mlp_forward_tables'
// loop (two table rows added, relu, FFMA2 second layer), the three partial sums are combined with two shuffles, lane 0
// applies the head.  All 20 loads of a lane are in flight at once: the launch is ~3 us on the step path.
__device__ __forceinline__ void states_pack(const float *__restrict__ tab, float4 *__restrict__ states) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x, e = t >> 2, j = t & 3;
    const bool valid = e < kStateQuads;  // the grid is a whole number of warps: every lane reaches the shuffles
    uint32_t xrow, yrow;
    state_rows(valid ? e % kNetStates : 0, xrow, yrow);
    const uint32_t net = valid ? (uint32_t)(e / kNetStates) : 0u;
    const float4 *T = reinterpret_cast<const float4 *>(tab);
    const float4 *xr = T + (net * kNetRows + xrow) * kRowQuads, *yr = T + (net * kNetRows + yrow) * kRowQuads;
    const float4 *wr = T + kTabRows * kRowQuads + net * (3 * kRowQuads);
    Layer2Acc acc;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int q = j + 4 * k;
        acc.quad_sum(xr[q], yr[q], wr[q], wr[kRowQuads + q], wr[2 * kRowQuads + q]);
    }
    float s0 = hsum2(acc.z0), s1 = hsum2(acc.z1), s2 = hsum2(acc.z2);
#pragma unroll
    for (int o = 1; o < 4; o <<= 1) {
        s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, o);
        s1 += __shfl_xor_sync(0xFFFFFFFFu, s1, o);
        s2 += __shfl_xor_sync(0xFFFFFFFFu, s2, o);
    }
    if (valid && j == 0) {
        float o0, o1, o2;
        Layer2Acc::head_of_sums(s0, s1, s2, reinterpret_cast<const float4 *>(tab + kTabFloats + kTabW2Floats)[net], net & 1u, o0, o1, o2);
        states[e] = make_float4(o0, o1, o2, __uint_as_float(score_word(o0, o1, o2)));
    }
}
// the tables of 1..NFSP_MAX_RUNS handles in one launch: blockIdx.y = handle
struct StatesRuns {
    const float *tab[NFSP_MAX_RUNS];
    float4 *states[NFSP_MAX_RUNS];
};
__global__ void states_pack_kernel(const __grid_constant__ StatesRuns P) { states_pack(P.tab[blockIdx.y], P.states[blockIdx.y]); }

// 1 024 threads per CTA for launches that keep every warp busy with several blocks of games; 512 (16 warps, 90 registers)
// when the launch has no more blocks than that gives warps -- a warp then plays one block, and what counts is the latency
// of its steps, which fewer warps per SM shorten (65 536 games: kernel 24.6 -> 21.3 us)
constexpr int kStatesThreads = 1024, kStatesThreadsSmall = 512;

// ---- warp-private record buffers -----------------------------------------------------------------
// Variant 1 claims its slots with four global atomics per warp and step.  That is one round trip per step on every
// warp's critical path, and with the direct ring append every one of the launch's 262 144 warp-steps hits the SAME two
// words (the rings' totals): same-address atomics retire at ~1.4 ns each, 0.37 ms per launch -- invisible beside variant
// 1's 0.37 ms of shared-memory traffic, the bound of this kernel once the forward is a table read.  Here a warp collects
// its records in shared memory (beside the table and the image) and claims slots for a whole buffer at a time: one
// atomic and one coalesced copy (512 B per warp instruction) per ~100 records.  100 RL records is what the 227 KB of a
// CTA leave at 32 warps.
constexpr int kBufRL = 100, kBufSL = 32;                 // records per player and warp; >= a step's worst case (64, 32)
constexpr int kWarpBufQuads = 2 * kBufRL + 2 * kBufSL;   // 264 uint4 = 4 224 B per warp
constexpr int kImageQuads = fsm::kRImageBytes / 16;
constexpr int states_smem_bytes(int threads) { return kStateBytes + fsm::kRImageBytes + (threads / 32) * kWarpBufQuads * 16; }
static_assert(fsm::kRImageBytes % 16 == 0, "the warps' buffers follow the image 16-byte aligned");
static_assert(kBufRL >= 64 && kBufSL >= 32, "a buffer must take the records of one step");

// quad offsets of the four lists in a warp's buffer: RL of player 0 / 1, SL of player 0 / 1
constexpr uint32_t kOffRL1 = kBufRL, kOffSL0 = 2 * kBufRL, kOffSL1 = 2 * kBufRL + kBufSL;

struct WarpBuf {
    uint4 *b;            // this warp's kWarpBufQuads of shared memory
    uint32_t cnt = 0u;   // records held, one byte per list: rl0 | rl1 << 8 | sl0 << 16 | sl1 << 24 (warp-uniform)
};

// inclusive warp scan of four byte counters (no byte exceeds 255); the shuffle's own predicate says whether a lane has a
// source, so a step is SHFL + a predicated add
__device__ __forceinline__ uint32_t warp_scan_bytes_p(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
        asm volatile("{ .reg .pred p; .reg .u32 r; shfl.sync.up.b32 r|p, %0, %1, 0, 0xffffffff; @p add.u32 %0, %0, r; }" : "+r"(v) : "r"(o));
    return v;
}

// copies the n buffered records of one list to base, base + 1, ... of its destination (coalesced: 512 B per warp store)
template <bool kRing, int kCap>
__device__ __forceinline__ void buf_copy(const uint4 *src, uint32_t n, uint4 *dst, uint32_t base, uint32_t cap, int &drop) {
    const uint32_t lane = threadIdx.x & 31u;
#pragma unroll
    for (int it = 0; it < (kCap + 31) / 32; ++it) {
        const uint32_t k = lane + 32u * it;
        if (k < n) {
            uint32_t off = base + k;
            if (kRing) {
                off = off < cap ? off : off - cap;  // a launch never laps the ring
                dst[off] = src[k];
            } else if (off < cap) {
                dst[off] = src[k];
            } else {
                ++drop;
            }
        }
    }
}

// moves the lists named in `which` (bit l = list l; warp-uniform) to their destinations: the claims of all lists go out
// together (lanes 0-3, one round trip), then one coalesced copy per list
template <bool kDirect>
__device__ __forceinline__ void buf_flush(WarpBuf &B, const RolloutArgs &A, const WarpStage &W, FastCounters &c, uint32_t which) {
    __syncwarp();
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t base = 0u;
    if (lane < 4u) {
        const uint32_t n = (B.cnt >> (8u * lane)) & 0xFFu;
        if (n && ((which >> lane) & 1u)) {
            if (kDirect && lane < 2u) base = ring_slot(atomicAdd(A.ring_total[lane], (unsigned long long)n), A.ring_cap, A.ring_magic);
            else base = atomicAdd(W.cnt + lane * W.n_seg, n);
        }
    }
    const uint32_t b0 = __shfl_sync(0xFFFFFFFFu, base, 0), b1 = __shfl_sync(0xFFFFFFFFu, base, 1);
    const uint32_t b2 = __shfl_sync(0xFFFFFFFFu, base, 2), b3 = __shfl_sync(0xFFFFFFFFu, base, 3);
    int drop = 0;
    if (which & 1u) buf_copy<kDirect, kBufRL>(B.b, B.cnt & 0xFFu, W.rl0, b0, W.cap_rl, drop);
    if (which & 2u) buf_copy<kDirect, kBufRL>(B.b + kOffRL1, (B.cnt >> 8) & 0xFFu, W.rl1, b1, W.cap_rl, drop);
    if (which & 4u) buf_copy<false, kBufSL>(B.b + kOffSL0, (B.cnt >> 16) & 0xFFu, W.sl0, b2, W.cap_sl, drop);
    if (which & 8u) buf_copy<false, kBufSL>(B.b + kOffSL1, B.cnt >> 24, W.sl1, b3, W.cap_sl, drop);
    c.wide.drop += drop;
    B.cnt &= ~(((which & 1u) ? 0xFFu : 0u) | ((which & 2u) ? 0xFF00u : 0u) | ((which & 4u) ? 0xFF0000u : 0u) | ((which & 8u) ? 0xFF000000u : 0u));
    __syncwarp();
}

// a step's records into the warp's buffers (what warp_append does with global atomics): the actor q's RL records A (the
// transition it remembered before acting) and B (its terminal observation), the other player's RL record C and the
// actor's SL record S.  All lanes call it.
template <bool kDirect>
__device__ __forceinline__ void buf_append(WarpBuf &B, const RolloutArgs &A, const WarpStage &W, FastCounters &c, uint32_t q,
                                           bool vA, bool vB, bool vC, bool vS, const uint4 &recA, const uint4 &recB,
                                           const uint4 &recC, const uint4 &recS) {
    // actor-relative counts: own ring | other ring << 8 | own reservoir << 16; swapping the bytes of each half makes them
    // absolute (rl0 | rl1 << 8 | sl0 << 16 | sl1 << 24) for player 1
    const uint32_t rel = ((uint32_t)vA + (uint32_t)vB) | (uint32_t)vC << 8 | (uint32_t)vS << 16;
    const uint32_t mine = q ? __byte_perm(rel, 0u, 0x2301u) : rel;
    const uint32_t incl = warp_scan_bytes_p(mine);
    const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
    // a list that cannot take this step's records is flushed first (warp-uniform, rare): byte > cap <=> bit 7 of
    // byte + 127 - cap (no byte carries: <= 100 + 64 and <= 32 + 32)
    constexpr uint32_t kOverRL = 127u - (uint32_t)kBufRL, kOverSL = 127u - (uint32_t)kBufSL;
    const uint32_t over = (B.cnt + tot + (kOverRL | kOverRL << 8 | kOverSL << 16 | kOverSL << 24)) & 0x80808080u;
    if (over) {
        uint32_t which = ((over >> 7) & 1u) | ((over >> 14) & 2u) | ((over >> 21) & 4u) | ((over >> 28) & 8u);
        if (which & 3u) which |= 3u;  // the two rings fill at the same pace: claim for both in one round trip
        buf_flush<kDirect>(B, A, W, c, which);
    }
    const uint32_t pos = B.cnt + (incl - mine);                       // absolute positions, bytewise
    const uint32_t prel = q ? __byte_perm(pos, 0u, 0x2301u) : pos;    // own ring | other ring | own reservoir
    uint32_t own = q * kOffRL1 + (prel & 0xFFu);
    if (vA) B.b[own++] = recA;
    if (vB) B.b[own] = recB;
    if (vC) B.b[(q ^ 1u) * kOffRL1 + ((prel >> 8) & 0xFFu)] = recC;
    if (vS) B.b[kOffSL0 + q * (uint32_t)kBufSL + ((prel >> 16) & 0xFFu)] = recS;
    B.cnt += tot;
}

// Which of the CTAs that serve A's games this CTA is: CTA c of n owns the blocks of 32 games c, c + n, c + 2 n, ... (every
// SM gets its share however few games there are) and its warps take them dynamically.  A launch of one run: the grid.
struct WholeGrid {
    __device__ __forceinline__ uint32_t cta() const { return blockIdx.x; }
    __device__ __forceinline__ uint32_t ctas() const { return gridDim.x; }
};
// one of several runs in a launch: a contiguous range of the grid
struct RunRange {
    uint32_t c, n;
    __device__ __forceinline__ uint32_t cta() const { return c; }
    __device__ __forceinline__ uint32_t ctas() const { return n; }
};

template <bool kDebug, bool kDirect, int kThreads, class Grid>
__device__ __forceinline__ void rollout_states_cta(const RolloutArgs &A, const Grid &G) {
    extern __shared__ __align__(128) float4 s_tab[];  // kStateQuads, the rollout image, then the warps' record buffers
    __shared__ unsigned long long s_stats[NFSP_STATS_FIELDS];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ uint32_t s_next;  // blocks of games this CTA has handed to its warps
    if (threadIdx.x < NFSP_STATS_FIELDS) s_stats[threadIdx.x] = 0ull;
    const uint32_t sbase = smem_u32(s_tab), ibase = sbase + (uint32_t)kStateBytes;
    {
        const uint32_t *img = reinterpret_cast<const uint32_t *>(A.pack) + 4 * kStateQuads;
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_tab + kStateQuads);
        for (int w = threadIdx.x; w < fsm::kRImageWords; w += kThreads) dst[w] = img[w] + (fsm::is_rollout_address(w) ? sbase : 0u);
    }
    const uint32_t bar = smem_u32(&s_bar);
    if (threadIdx.x == 0) {
        s_next = 0u;
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // the state table comes in as two bulk async copies, completion on an mbarrier
        mbar_expect_tx(bar, kStateBytes);
        constexpr uint32_t kChunk = 32768;
        for (uint32_t off = 0; off < (uint32_t)kStateBytes; off += kChunk) {
            const uint32_t len = (uint32_t)kStateBytes - off < kChunk ? (uint32_t)kStateBytes - off : kChunk;
            bulk_g2s(sbase + off, reinterpret_cast<const uint8_t *>(A.pack) + off, len, bar);
        }
    }
    bool image_ready = false;
    const uint32_t dl_sum = 2u * (ibase + (uint32_t)fsm::kRDealOff) + (uint32_t)fsm::kRDealHalf;
    const uint32_t rew_base = ibase + (uint32_t)fsm::kRRewardOff;

    FastCounters c;
    const int64_t plane = (int64_t)A.n_steps * A.n;
    const uint32_t lane = threadIdx.x & 31u;
    WarpBuf B;
    // the warp's offset goes through a shuffle so that it lives in a register: left as arithmetic on threadIdx.x, it was
    // recomputed at each of the step's four buffer stores (16 instructions per warp-step in ncu's source view)
    B.b = reinterpret_cast<uint4 *>(s_tab) + kStateQuads + kImageQuads + __shfl_sync(0xFFFFFFFFu, (threadIdx.x >> 5) * (uint32_t)kWarpBufQuads, 0);
    WarpStage W;
    W.init(A, 0u, kDirect);
    const int64_t n_blocks = (A.n + 31) >> 5;  // CTA c owns blocks c, c + grid, ...; its warps take them dynamically
    for (;;) {
        uint32_t blk = 0;
        if (lane == 0) blk = G.cta() + G.ctas() * atomicAdd(&s_next, 1u);
        blk = __shfl_sync(0xFFFFFFFFu, blk, 0);
        if ((int64_t)blk >= n_blocks) break;
        const int64_t base = (int64_t)blk << 5;
        const int64_t i = base + lane;
        const bool live = i < A.n;
        const uint64_t game = A.game0 + (uint64_t)i;
        W.init(A, (uint32_t)(base >> 5) & (A.n_seg - 1u), kDirect);
        fsm::RolloutGame g;
        g.unpack(live ? A.state[i] : 0ull, ibase, sbase);
        if (!image_ready) {  // the table's copy ran beside the set-up and the first loads of the game words
            mbar_wait(bar, 0);
            image_ready = true;
        }
        for (int t = 0; t < A.n_steps; ++t) {
            const uint64_t step = A.step0 + (uint64_t)t;
            const Philox4 x = game_block(A.keys, game, step, STREAM_STEP);
            uint32_t started = 0u;
            if (g.HX & fsm::kHxOver) {  // newenv.py:76-114 + main.py:28-45: the other player deals
                g.dl = dl_sum - g.dl;
                const uint4 D = fsm::lds128(g.dl + __umulhi(x.y, 120u) * 16u);
                uint32_t pa = g.dl + (uint32_t)fsm::kPolOff;
                if (x.z < A.eta_u32) pa += 16u;
                if (x.w < A.eta_u32) pa += 32u;
                const uint4 P = fsm::lds128(pa);
                g.PA = D.x | P.x;
                g.PO = D.y | P.y;
                g.FA = D.z + P.z;
                g.FO = D.w + P.w;
                g.SA = 0u;
                g.SO = 0u;
                g.tix = g.dl - (uint32_t)fsm::kRDealOff;
                g.HX = fsm::kCm0;
                started = 1u;
                c.wide.hands += live;
            }
            // agent.py:130-141: the observation, the transition to remember, the policy of the hand, the epsilon branch
            const uint32_t q = (g.PA >> 23) & 1u;
            const uint32_t obs = g.HX & (g.PA | 0x00FFFFFFu);
            const bool vA = (g.PA & kWordNz) != 0u, pol = (g.PA & (1u << 12)) != 0u;
            const uint4 recA = make_uint4(g.SA, obs, 0u, ((g.PA >> 13) & 3u) | (q << 16));
            const uint4 o = fsm::lds128(g.FA);
            float v0 = __uint_as_float(o.x), v1 = __uint_as_float(o.y), v2 = __uint_as_float(o.z);
            uint32_t aw = o.w;
            if (pol && x.x < (q ? A.eps1_u32 : A.eps_u32)) {  // np.random.rand(1,1,3): rare, so it has its own Philox block
                const Philox4 y = game_block(A.keys, game, step, STREAM_VECTOR);
                v0 = (float)(y.x >> 8) * (1.0f / 16777216.0f);
                v1 = (float)(y.y >> 8) * (1.0f / 16777216.0f);
                v2 = (float)(y.z >> 8) * (1.0f / 16777216.0f);
                aw = score_word(v0, v1, v2);
            }
            const int64_t at = (int64_t)t * A.n + i;
            if (kDebug && live) {
                if (A.vec) { A.vec[3 * at] = v0; A.vec[3 * at + 1] = v1; A.vec[3 * at + 2] = v2; }
                if (A.forced) { v0 = A.forced[3 * at]; v1 = A.forced[3 * at + 1]; v2 = A.forced[3 * at + 2]; }
                aw = score_word(v0, v1, v2);
            }
            // newenv.py:192-349: the entry (row, raw action)
            const uint32_t ea = g.tix + (aw & kWordEntry);
            const uint4 E = fsm::lds128(ea);        // hc, pa, pm, nx
            const uint4 M = fsm::lds128(ea + 16u);  // ds, mx, rm, inc
            g.PA = ((g.PA & ~fsm::kPClear) | (aw & kWordNz)) + E.y;
            g.HX = (g.HX & 0xFFFFFFu) | E.x;
            c.small += live ? M.w : 0u;
            // main.py:55-67: at the end of the hand both players observe the terminal state once (no swap happens then)
            const bool term = (g.HX & fsm::kHxOver) != 0u;
            const uint32_t rw = fsm::lds32(rew_base + (M.z & ((g.PA & 0xFFu) | (g.PO & 0xF00u))));  // 0 while the hand is live
            const int ra = (int)(int8_t)(rw & 0xFFu), ro = (int)(int8_t)((rw >> 8) & 0xFFu);
            c.wide.rew0 += live ? (q ? ro : ra) : 0;
            c.wide.rew1 += live ? (q ? ra : ro) : 0;
            const float fa = 0.5f * (float)ra;
            const uint4 recB = make_uint4(obs, g.HX & (g.PA | 0x00FFFFFFu), __float_as_uint(fa), M.y & 0x10103u);
            const uint4 recC = make_uint4(g.SO, g.HX & (g.PO | 0x00FFFFFFu), __float_as_uint(0.5f * (float)ro),
                                          ((g.PO >> 13) & 3u) | ((M.y & 0x10100u) ^ 0x10000u));
            const bool vB = term && (aw & kWordNz) && live, vC = term && (g.PO & kWordNz) && live;
            if (kDebug && live && A.trace) {
                const uint32_t P0 = q ? g.PO : g.PA, P1 = q ? g.PA : g.PO;
                const uint32_t d = g.dl != ibase + (uint32_t)fsm::kRDealOff ? 1u : 0u;
                A.trace[at] = g.HX & (g.PA | 0xC0FFFFFFu);  // observation of the actor | hand over << 30 | actor << 31
                A.trace[plane + at] = __float_as_uint(fa);
                A.trace[2 * plane + at] = (M.y & 0x101Fu) | (d << 5) | (((P0 >> 19) & 3u) << 6) | (((P1 >> 19) & 3u) << 8) |
                                          (((P0 >> 21) & 3u) << 10) | (((P0 >> 2) & 15u) << 13) | (((P1 >> 2) & 15u) << 17) |
                                          (started << 21) | (((P0 >> 12) & 1u) << 22) | (((P1 >> 12) & 1u) << 23);
            }
            // the turn passes: swap the per-player registers
            const uint32_t pm = E.z, pa = g.PA, sa = obs, fa_ = g.FA + M.x, fo = g.FO + M.x;
            g.PA = (g.PO & pm) | (pa & ~pm);
            g.PO = (pa & pm) | (g.PO & ~pm);
            g.SA = (g.SO & pm) | (sa & ~pm);
            g.SO = (sa & pm) | (g.SO & ~pm);
            g.FA = (fo & pm) | (fa_ & ~pm);
            g.FO = (fa_ & pm) | (fo & ~pm);
            g.tix = E.w;
            buf_append<kDirect>(B, A, W, c, q, vA && live, vB, vC, pol && live, recA, recB, recC,
                                make_uint4(obs, __float_as_uint(v0), __float_as_uint(v1), __float_as_uint(v2)));
            if ((t & 15) == 15) c.spill();
        }
        c.spill();
        if (live) A.state[i] = g.pack(ibase);
        c.wide.trans += live ? A.n_steps : 0;
        // a block's staged records belong to the block's segment; the rings have no segments, their records stay buffered
        buf_flush<kDirect>(B, A, W, c, kDirect ? 12u : 15u);
    }
    if (kDirect) buf_flush<true>(B, A, W, c, 3u);
    if (!image_ready) mbar_wait(bar, 0);  // the copy into this CTA's shared memory must land before the CTA exits
    c.spill();
    if (A.stats) c.wide.commit(s_stats, A.stats);
}

template <bool kDebug, bool kDirect, int kThreads>
__global__ void __launch_bounds__(kThreads, 1)
rollout_states_kernel(const RolloutArgs A) {
    rollout_states_cta<kDebug, kDirect, kThreads>(A, WholeGrid{});
}

// ---- independent runs in one launch (nfsp_rollout_runs) -------------------------------------------
// Runs of the same shape (game count, record mode) each get the same number of CTAs, in contiguous ranges of the grid:
// CTA b serves run b / ctas_per_run as CTA b % ctas_per_run of ctas_per_run, with that run's state table, keys,
// thresholds, game words, records and counters -- exactly what the run's own launch on ctas_per_run CTAs would do.
// The run dimension is a compile-time bound on the argument table, which lives in the parameter space (~10 KB); a CTA
// copies its run's entry to shared memory first (fewer registers than indexing the parameter space at every use).
template <int kRuns>
struct RolloutRuns {
    RolloutArgs run[kRuns];
    uint32_t ctas_per_run;
};

template <bool kDebug, bool kDirect, int kThreads, int kRuns>
__global__ void __launch_bounds__(kThreads, 1)
rollout_states_kernel(const __grid_constant__ RolloutRuns<kRuns> R) {
    static_assert(!kDebug, "runs have no debug outputs");
    static_assert(sizeof(RolloutArgs) % 4 == 0, "copied in words");
    __shared__ __align__(16) RolloutArgs s_args;  // the run's arguments, read by the steps from shared memory
    const uint32_t r = blockIdx.x / R.ctas_per_run;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&R.run[r]);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&s_args);
        for (int w = threadIdx.x; w < (int)(sizeof(RolloutArgs) / 4); w += kThreads) dst[w] = src[w];
    }
    __syncthreads();
    rollout_states_cta<false, kDirect, kThreads>(s_args, RunRange{blockIdx.x - r * R.ctas_per_run, R.ctas_per_run});
}

}  // namespace nfsp

using namespace nfsp;

// the state table, then the rollout image (uploaded once, nfsp_states_upload_image)
int nfsp_states_floats() { return kStateQuads * 4 + fsm::kRImageWords; }

static void build_states_image(uint32_t *img) { fsm::build_rollout_image(img, (uint32_t)kStateBytes); }

int nfsp_states_upload_image(float *d_states) {
    static uint32_t image[fsm::kRImageWords];
    static const bool built = (build_states_image(image), true);
    (void)built;
    NFSP_CUDA(cudaMemcpy(d_states + 4 * kStateQuads, image, sizeof(image), cudaMemcpyHostToDevice));
    return NFSP_OK;
}

// the rollout image for inspection on the host (addresses: byte offsets from the state table, which it follows)
extern "C" int nfsp_rollout_image(uint32_t *out, int capacity_words) {
    if (out && capacity_words >= fsm::kRImageWords) build_states_image(out);
    return fsm::kRImageWords;
}

template <int kThreads>
static int configure_states() {
    constexpr int kBytes = states_smem_bytes(kThreads);
    NFSP_CUDA(cudaFuncSetAttribute(rollout_states_kernel<true, true, kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBytes));
    NFSP_CUDA(cudaFuncSetAttribute(rollout_states_kernel<true, false, kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBytes));
    NFSP_CUDA(cudaFuncSetAttribute(rollout_states_kernel<false, true, kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBytes));
    NFSP_CUDA(cudaFuncSetAttribute(rollout_states_kernel<false, false, kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBytes));
    return NFSP_OK;
}

int nfsp_rollout_states_configure() {
    const int rc = configure_states<kStatesThreads>();
    return rc != NFSP_OK ? rc : configure_states<kStatesThreadsSmall>();
}

template <int kThreads>
static int launch_states(const RolloutArgs &A, int grid, bool debug, bool direct, cudaStream_t st) {
    constexpr int kBytes = states_smem_bytes(kThreads);
    if (debug && direct) rollout_states_kernel<true, true, kThreads><<<grid, kThreads, kBytes, st>>>(A);
    else if (debug) rollout_states_kernel<true, false, kThreads><<<grid, kThreads, kBytes, st>>>(A);
    else if (direct) rollout_states_kernel<false, true, kThreads><<<grid, kThreads, kBytes, st>>>(A);
    else rollout_states_kernel<false, false, kThreads><<<grid, kThreads, kBytes, st>>>(A);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

int nfsp_states_pack(const nfsp_env_t *h, const float *const *tab, int n, cudaStream_t st) {
    StatesRuns P;
    for (int r = 0; r < n; ++r) {
        P.tab[r] = tab[r];
        P.states[r] = reinterpret_cast<float4 *>(h[r]->d_states);
    }
    states_pack_kernel<<<dim3((4 * kStateQuads + 127) / 128, (unsigned)n), 128, 0, st>>>(P);
    NFSP_LAUNCH_CHECK();
    for (int r = 0; r < n; ++r) h[r]->st_dirty = false;
    return NFSP_OK;
}

template <bool kDirect, int kThreads>
static int launch_states_runs(const RolloutArgs *A, int n_runs, int ctas_per_run, cudaStream_t st) {
    constexpr int kBytes = states_smem_bytes(kThreads);
    using Kernel = void (*)(RolloutRuns<NFSP_MAX_RUNS>);
    const Kernel k = rollout_states_kernel<false, kDirect, kThreads, NFSP_MAX_RUNS>;
    // per call: the attribute belongs to the current device's context
    NFSP_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kBytes));
    RolloutRuns<NFSP_MAX_RUNS> R;
    for (int r = 0; r < n_runs; ++r) R.run[r] = A[r];
    R.ctas_per_run = (uint32_t)ctas_per_run;
    k<<<n_runs * ctas_per_run, kThreads, kBytes, st>>>(R);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

// n_runs runs of h->n games each, of one record mode (A[r].ring[0] != null for all or none); sms = SMs the grid may use.
// Always 512 threads per CTA: a run's arguments are no longer constant-bank operands (the 20 Philox round keys alone), and
// at 1 024 threads' 64 registers that spilled; at 512 the kernel holds them without spills (ptxas log).
int nfsp_rollout_states_runs_launch(nfsp_env_t h, const RolloutArgs *A, int n_runs, int sms, cudaStream_t st) {
    const int ctas = grid_for(h->n, 32, sms / n_runs, 1);  // at least one block of 32 games per CTA
    return A[0].ring[0] != nullptr ? launch_states_runs<true, kStatesThreadsSmall>(A, n_runs, ctas, st)
                                   : launch_states_runs<false, kStatesThreadsSmall>(A, n_runs, ctas, st);
}

int nfsp_rollout_states_launch(nfsp_env_t h, const RolloutArgs &A, const nfsp_rollout_io *io, bool debug, cudaStream_t st) {
    const bool direct = A.ring[0] != nullptr;
    const int sms = h->sm_count - io->reserve_sms;
    const int grid = grid_for(h->n, 32, sms, 1);  // at least one block of 32 games per CTA
    const int64_t blocks = (h->n + 31) / 32;
    if (blocks <= (int64_t)sms * (kStatesThreadsSmall / 32)) return launch_states<kStatesThreadsSmall>(A, grid, debug, direct, st);
    return launch_states<kStatesThreads>(A, grid, debug, direct, st);
}
