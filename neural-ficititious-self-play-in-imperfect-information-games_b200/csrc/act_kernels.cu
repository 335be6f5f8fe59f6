// K2 (CUDA-core variant): NFSP acting fused with the env step.
//
// One thread per game.  Per step a game does exactly one Agent.play decision (agent.py:130-156):
// observation -> one of four 30-64-3 MLPs (player x {average, best-response}) -> eta-mixed /
// epsilon-greedy score vector -> argmax -> newenv step, and emits the RL / SL memory records of
// agent.py:134-136,151 and the terminal observations of main.py:55-67.  The observation is a
// 30-bit mask that never leaves registers; because it is binary and sparse (<= 9 bits set) the
// first layer is a SUM OF WEIGHT ROWS read from shared memory as float4s instead of a dense 30x64
// product: <= 9 rows for arbitrary masks (act_forward_kernel), 3 precombined rows in the rollout.
#include "mlp_math.cuh"
#include "ptx_helpers.cuh"
#include "rollout_fast.cuh"
#include "rollout_tables.cuh"

namespace nfsp {

constexpr int kActThreads = 128;   // act_forward_kernel (generic observation masks)
constexpr int kRollThreads = 1024;  // rollout_kernel: one CTA per SM
// packed weight image (floats) of the generic forward: W1 rows as [128 rows = net*32 + input][24 quads][4], where
// input 30 is the bias b1 and a row is its 16 quads of hidden units followed by a copy of the first 8 (so a thread can
// read from quad rot = index & 7 with immediate offsets and the 8 threads of a quarter-warp never share a bank
// group, see the rollout tables below); then W2 as [4 nets][3 outputs][24 quads][4]; then b2 as [4 nets][4].
constexpr int kFwdRowQuads = 24;
constexpr int kW1Floats = 128 * kFwdRowQuads * 4;
constexpr int kW2Floats = 4 * 3 * kFwdRowQuads * 4;
constexpr int kPackFloats = kW1Floats + kW2Floats + kB2Floats;

// element e of the batched forward's weight image
__device__ __forceinline__ float pack_weights_value(const float *__restrict__ w, int e) {
    {
        float v = 0.f;
        if (e < kW1Floats) {
            const int c = e & 3, pos = (e >> 2) % kFwdRowQuads, row = (e >> 2) / kFwdRowQuads;
            const int net = row >> 5, i = row & 31, j = (pos & 15) * 4 + c;
            const float *wn = w + net * NFSP_NET_PARAMS;
            if (i < 30) v = wn[i * 64 + j];
            else if (i == 30) v = wn[1920 + j];
        } else if (e < kW1Floats + kW2Floats) {
            const int f = e - kW1Floats, x = f & 3, pos = (f >> 2) % kFwdRowQuads, c = ((f >> 2) / kFwdRowQuads) % 3;
            const int net = (f >> 2) / (3 * kFwdRowQuads);
            v = w[net * NFSP_NET_PARAMS + 1984 + ((pos & 15) * 4 + x) * 3 + c];
        } else {
            const int f = e - kW1Floats - kW2Floats, c = f & 3, net = f >> 2;
            if (c < 3) v = w[net * NFSP_NET_PARAMS + 2176 + c];
        }
        return v;
    }
}

static_assert((kPackFloats + kTabImageFloats + 4 * NFSP_NET_PARAMS) % 4 == 0, "the state table behind the images must be 16-byte aligned (bulk copy)");
// both images in one launch: pack = [batched-forward image (kPackFloats) | rollout table image (kTabImageFloats)] + a plain copy of the four nets (what the tensor-core variants' images are built from, on demand)
__device__ __forceinline__ void pack_images(const float *__restrict__ w, float *__restrict__ pack) {
    constexpr int kImages = kPackFloats + kTabImageFloats;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kImages + 4 * NFSP_NET_PARAMS; e += gridDim.x * blockDim.x)
        pack[e] = e < kPackFloats ? pack_weights_value(w, e) : (e < kImages ? pack_tables_value(w, e - kPackFloats) : w[e - kImages]);
}
// the images of 1..NFSP_MAX_RUNS handles in one launch: blockIdx.y = handle
struct ImageRuns {
    const float *w[NFSP_MAX_RUNS];
    float *pack[NFSP_MAX_RUNS];
};
__global__ void pack_images_kernel(const __grid_constant__ ImageRuns P) { pack_images(P.w[blockIdx.y], P.pack[blockIdx.y]); }

// forward of one net on one observation mask; sw = packed image in shared memory.  The first layer is the sum of the
// <= 10 weight rows of the set input bits (+ the bias row), accumulated in the thread's ROTATED quad order.
__device__ __forceinline__ void mlp_forward(const float *__restrict__ sw, uint32_t obs, int net, uint32_t rot, float out[3]) {
    const float4 *w1 = reinterpret_cast<const float4 *>(sw) + rot;
    float4 h[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) h[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t bits = (obs & 0x3FFFFFFFu) | (1u << 30);  // input 30 = constant 1 -> adds the bias row last
    while (bits) {
        const int i = __ffs(bits) - 1;
        bits &= bits - 1u;
        const float4 *r = w1 + (net * 32 + i) * kFwdRowQuads;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const float4 v = r[q];
            h[q].x += v.x; h[q].y += v.y; h[q].z += v.z; h[q].w += v.w;
        }
    }
    const float4 *w2 = reinterpret_cast<const float4 *>(sw + kW1Floats) + net * (3 * kFwdRowQuads) + rot;
    Layer2Acc acc;
#pragma unroll
    for (int q = 0; q < 16; ++q)  // Dense(64, relu) then Dense(3), agent.py:102-103,111-112
        acc.quad(h[q].x, h[q].y, h[q].z, h[q].w, w2[q], w2[kFwdRowQuads + q], w2[2 * kFwdRowQuads + q]);
    acc.head(reinterpret_cast<const float4 *>(sw + kW1Floats + kW2Floats)[net], net & 1, out[0], out[1], out[2]);
}

__device__ __forceinline__ void load_pack(float *sw, const float *__restrict__ pack) {
    const float4 *src = reinterpret_cast<const float4 *>(pack);
    float4 *dst = reinterpret_cast<float4 *>(sw);
    for (int e = threadIdx.x; e < kPackFloats / 4; e += blockDim.x) dst[e] = src[e];
    __syncthreads();
}

__global__ void __launch_bounds__(kActThreads)
act_forward_kernel(const float *__restrict__ pack, const uint32_t *__restrict__ obs, const int8_t *__restrict__ net,
                   int64_t n, float *__restrict__ out) {
    extern __shared__ __align__(16) float sw[];  // kPackFloats
    load_pack(sw, pack);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float v[3];
        mlp_forward(sw, obs[i], (int)(net[i] & 3), (uint32_t)i & 7u, v);
        out[3 * i] = v[0]; out[3 * i + 1] = v[1]; out[3 * i + 2] = v[2];
    }
}

// One persistent CTA per SM (the table image fills most of its shared memory); a warp owns 32 consecutive
// games for the launch's steps, the games' state lives in registers in the actor-relative form of
// nfsp_fast.cuh and goes back to HBM as the packed word.
template <bool kDebug, bool kDirect>
__global__ void __launch_bounds__(kRollThreads, 1)
rollout_kernel(const RolloutArgs A) {
    extern __shared__ __align__(128) float sw[];  // table image, kTabImageBytes
    __shared__ unsigned long long s_stats[NFSP_STATS_FIELDS];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ FastLuts s_lut;
    __shared__ uint32_t s_next;  // blocks of games this CTA has handed to its warps
    if (threadIdx.x < NFSP_STATS_FIELDS) s_stats[threadIdx.x] = 0ull;
    s_lut.fill();
    const uint32_t bar = smem_u32(&s_bar);
    if (threadIdx.x == 0) {
        s_next = 0u;
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // the table image comes in as bulk async copies (TMA unit), completion on an mbarrier
        mbar_expect_tx(bar, kTabImageBytes);
        constexpr uint32_t kChunk = 32768;
        for (uint32_t off = 0; off < (uint32_t)kTabImageBytes; off += kChunk) {
            const uint32_t len = (uint32_t)kTabImageBytes - off < kChunk ? (uint32_t)kTabImageBytes - off : kChunk;
            bulk_g2s(smem_u32(sw) + off, reinterpret_cast<const uint8_t *>(A.pack) + off, len, bar);
        }
    }
    bool image_ready = false;  // waited for just before the first MLP evaluation: the copy overlaps the first step's game logic

    FastCounters c;
    const int64_t plane = (int64_t)A.n_steps * A.n;
    const uint32_t lane = threadIdx.x & 31u;
    // blocks of 32 consecutive games: CTA c owns blocks c, c + grid, c + 2 grid, ... (every SM gets its share however
    // few games there are -- with one global counter the first CTAs to start took all 2 048 blocks of a 64k-game
    // launch and 84 SMs idled), and its warps take them dynamically through a shared-memory counter, which keeps the
    // 32 warps busy to the end (a static split over the warps leaves 8% of the last pass idle)
    const int64_t n_blocks = (A.n + 31) >> 5;
    for (;;) {
        uint32_t blk = 0;
        if (lane == 0) blk = blockIdx.x + gridDim.x * atomicAdd(&s_next, 1u);
        blk = __shfl_sync(0xFFFFFFFFu, blk, 0);
        if ((int64_t)blk >= n_blocks) break;
        const int64_t base = (int64_t)blk << 5;
        const int64_t i = base + lane;
        const bool live = i < A.n;
        const uint64_t game = A.game0 + (uint64_t)i;
        const uint32_t rot = (uint32_t)game & 7u;
        WarpStage W;
        W.init(A, (uint32_t)(base >> 5) & (A.n_seg - 1u), kDirect);
        NfspFast g;
        g.unpack(live ? A.state[i] : 0ull);
        for (int t = 0; t < A.n_steps; ++t) {
            FastDecision d;
            fast_begin(g, s_lut, A, game, A.step0 + (uint64_t)t, live, d, c);
            const uint32_t sg = g.sigma(), dl = g.dealer(), ca = (g.PA >> 11) & 3u;
            const uint32_t xrow = sg >= 9u ? 3u + ((((ca * 3u + g.pub()) * 2u + dl) << 2) | g.fin0()) : ca;
            const uint32_t yrow = 75u + dl * 18u + sg;
            float v0, v1, v2;
            if (!image_ready) {
                mbar_wait(bar, 0);
                image_ready = true;
            }
            mlp_forward_tables(sw, xrow, yrow, g.p() * 2u + (uint32_t)d.pol, rot, v0, v1, v2);
            if (d.random) { v0 = d.r0; v1 = d.r1; v2 = d.r2; }
            fast_finish<kDebug, kDirect>(g, s_lut, A, W, d, v0, v1, v2, live, (int64_t)t * A.n + i, plane, c);
            if ((t & 15) == 15) c.spill();
        }
        c.spill();  // the 5-bit counters must not run on into the warp's next block of games
        if (live) A.state[i] = g.pack();
        c.wide.trans += live ? A.n_steps : 0;
    }
    if (!image_ready) mbar_wait(bar, 0);  // no block came this way: the copy into this CTA's shared memory must still land
    c.spill();
    if (A.stats) c.wide.commit(s_stats, A.stats);
}

}  // namespace nfsp

using namespace nfsp;

// nfsp_act_set_weights of n handles whose buffers exist: handle r's images from w[r], then the default rollout's table of
// the nets' outputs per decision state from the table image just built -- one launch each, whatever n.  The tensor-core
// variants' images follow lazily (nfsp_ensure_tc_images).
static int rebuild_images(const nfsp_env_t *h, const float *const *w, int n, cudaStream_t st) {
    ImageRuns P;
    const float *tab[NFSP_MAX_RUNS];
    for (int r = 0; r < n; ++r) {
        P.w[r] = w[r];
        P.pack[r] = h[r]->d_wpack;
        tab[r] = h[r]->d_wpack + kPackFloats;
    }
    pack_images_kernel<<<dim3((kPackFloats + kTabImageFloats + 4 * NFSP_NET_PARAMS + 255) / 256, (unsigned)n), 256, 0, st>>>(P);
    NFSP_LAUNCH_CHECK();
    for (int r = 0; r < n; ++r) {
        h[r]->tc_dirty = h[r]->tq_dirty = h[r]->st_dirty = true;
        h[r]->has_weights = true;
    }
    return nfsp_states_pack(h, tab, n, st);  // clears st_dirty
}

// the state table alone, when it is older than the table image
static int states_ensure(nfsp_env_t h, cudaStream_t st) {
    if (!h->st_dirty) return NFSP_OK;
    const float *tab = h->d_wpack + kPackFloats;
    return nfsp_states_pack(&h, &tab, 1, st);
}

extern "C" int nfsp_act_set_weights(nfsp_env_t h, const float *d_weights, void *stream) {
    NFSP_CHECK_ARG(h != nullptr && d_weights != nullptr, "null argument");
    NFSP_CHECK_ARG(h->rules == NFSP_RULES_NFSP, "acting nets need NFSP rules");
    DeviceGuard guard(h->device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", h->device);
    if (!h->d_wpack) {
        NFSP_CUDA(cudaMalloc(&h->d_wpack, sizeof(float) * (kPackFloats + kTabImageFloats + 4 * NFSP_NET_PARAMS + nfsp_states_floats())));
        h->d_wcopy = h->d_wpack + kPackFloats + kTabImageFloats;
        h->d_states = h->d_wpack + kPackFloats + kTabImageFloats + 4 * NFSP_NET_PARAMS;
        NFSP_CUDA(cudaMalloc(&h->d_work, sizeof(uint32_t)));
        NFSP_CUDA(cudaFuncSetAttribute(act_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kPackFloats * sizeof(float))));
        NFSP_CUDA(cudaFuncSetAttribute(rollout_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabImageBytes));
        NFSP_CUDA(cudaFuncSetAttribute(rollout_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabImageBytes));
        NFSP_CUDA(cudaFuncSetAttribute(rollout_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabImageBytes));
        NFSP_CUDA(cudaFuncSetAttribute(rollout_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabImageBytes));
        int rc = nfsp_rollout_sorted_configure();
        if (rc != NFSP_OK) return rc;
        rc = nfsp_rollout_pairs_configure();
        if (rc != NFSP_OK) return rc;
        rc = nfsp_rollout_states_configure();
        if (rc != NFSP_OK) return rc;
        rc = nfsp_states_upload_image(h->d_states);
        if (rc != NFSP_OK) return rc;
    }
    return rebuild_images(&h, &d_weights, 1, (cudaStream_t)stream);
}

int nfsp_ensure_tc_images(nfsp_env_t h, bool tq, cudaStream_t st) {
    if (h->tc_dirty) {
        const int rc = nfsp_pack_tc_image(h, h->d_wcopy, st);
        if (rc != NFSP_OK) return rc;
        h->tc_dirty = false;
    }
    if (tq && h->tq_dirty) {
        const int rc = nfsp_tq_set_weights(h, h->d_wcopy, st);
        if (rc != NFSP_OK) return rc;
        h->tq_dirty = false;
    }
    return NFSP_OK;
}

extern "C" int nfsp_act_set_weights_from_host(nfsp_env_t h, const float *h_weights, float *d_weights, void *stream) {
    NFSP_CHECK_ARG(h != nullptr && h_weights != nullptr && d_weights != nullptr, "null argument");
    DeviceGuard guard(h->device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", h->device);
    NFSP_CUDA(cudaMemcpyAsync(d_weights, h_weights, sizeof(float) * 4 * NFSP_NET_PARAMS, cudaMemcpyHostToDevice,
                              (cudaStream_t)stream));
    return nfsp_act_set_weights(h, d_weights, stream);
}

extern "C" int nfsp_act_forward(nfsp_env_t h, const uint32_t *d_obs, const int8_t *d_net, int64_t n, float *d_out,
                                void *stream) {
    NFSP_CHECK_ARG(h != nullptr && d_obs && d_net && d_out && n >= 0, "bad arguments");
    if (!h->has_weights) return set_error(NFSP_E_STATE, "nfsp_act_set_weights has not been called");
    if (n == 0) return NFSP_OK;
    DeviceGuard guard(h->device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", h->device);
    const int grid = grid_for(n, kActThreads, h->sm_count, 4);
    act_forward_kernel<<<grid, kActThreads, kPackFloats * sizeof(float), (cudaStream_t)stream>>>(h->d_wpack, d_obs, d_net, n, d_out);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

int nfsp_rollout_direct_args(const nfsp_rollout_io *io, RolloutArgs &A, bool *direct) {
    for (int q = 0; q < 2; ++q) { A.ring[q] = nullptr; A.ring_total[q] = nullptr; }
    A.ring_cap = 0u;
    A.ring_magic = 0ull;
    *direct = io->d_ring[0] != nullptr || io->d_ring[1] != nullptr;
    if (!*direct) return NFSP_OK;
    NFSP_CHECK_ARG(io->d_ring[0] && io->d_ring[1] && io->d_ring_total[0] && io->d_ring_total[1],
                   "the direct ring append needs both rings and their totals");
    NFSP_CHECK_ARG(io->ring_cap > 1 && io->ring_cap < ((int64_t)1 << 32), "ring capacity out of range");
    NFSP_CHECK_ARG(2 * A.n * (int64_t)A.n_steps <= io->ring_cap,
                   "direct ring append needs 2 * n * n_steps <= ring capacity (a launch must not lap the ring)");
    for (int q = 0; q < 2; ++q) {
        A.ring[q] = (uint4 *)io->d_ring[q];
        A.ring_total[q] = (unsigned long long *)io->d_ring_total[q];
    }
    A.ring_cap = (uint32_t)io->ring_cap;
    A.ring_magic = ~0ull / (uint64_t)io->ring_cap;
    return NFSP_OK;
}

// validates the arguments of a rollout of handle h and fills A (nothing is launched): the variant to run (0 resolved),
// whether the call has debug outputs, whether it appends to the rings directly
static int rollout_args(nfsp_env_t h, int n_steps, double eta, double epsilon, const nfsp_rollout_io *io, RolloutArgs &A,
                        int *variant_out, bool *debug_out, bool *direct_out) {
    NFSP_CHECK_ARG(h != nullptr && io != nullptr, "null argument");
    NFSP_CHECK_ARG(h->rules == NFSP_RULES_NFSP, "rollout needs NFSP rules");
    NFSP_CHECK_ARG(n_steps >= 1 && n_steps <= 4096, "n_steps must be in [1,4096]");
    NFSP_CHECK_ARG(io->d_rl[0] && io->d_rl[1] && io->d_sl[0] && io->d_sl[1] && io->d_counts, "missing staging arrays");
    NFSP_CHECK_ARG(io->cap_rl > 0 && io->cap_sl > 0 && io->cap_rl < ((int64_t)1 << 32) && io->cap_sl < ((int64_t)1 << 32),
                   "staging capacity out of range");
    NFSP_CHECK_ARG(io->n_segments >= 1 && io->n_segments <= 65536 && (io->n_segments & (io->n_segments - 1)) == 0,
                   "n_segments must be a power of two in [1,65536]");
    if (!h->has_weights) return set_error(NFSP_E_STATE, "nfsp_act_set_weights has not been called");
    A.keys = philox_keys(h->seed);
    A.state = h->d_state; A.n = h->n; A.seed = h->seed; A.game0 = h->game0; A.step0 = h->step; A.n_steps = n_steps;
    A.eta_u32 = frac_u32(eta); A.eps_u32 = frac_u32(epsilon);
    A.eps1_u32 = io->epsilon_per_player ? frac_u32(io->epsilon_p1) : A.eps_u32;
    A.pack = h->d_wpack + kPackFloats;
    for (int q = 0; q < 2; ++q) { A.rl[q] = (uint4 *)io->d_rl[q]; A.sl[q] = (uint4 *)io->d_sl[q]; }
    A.cap_rl = io->cap_rl; A.cap_sl = io->cap_sl; A.n_seg = (uint32_t)io->n_segments; A.counts = io->d_counts;
    A.work = h->d_work;
    A.stats = (unsigned long long *)io->d_stats; A.trace = io->d_trace; A.vec = io->d_vec; A.forced = io->d_forced_vec;
    const bool debug = io->d_trace || io->d_vec || io->d_forced_vec;
    NFSP_CHECK_ARG(io->variant >= 0 && io->variant <= 6,
                   "variant must be 0 (default), 1 (CUDA cores), 2 (tcgen05, one tile per group), 3 (tcgen05, warp-specialised), "
                   "4 (CUDA cores, net-sorted groups), 5 (CUDA cores, two games per lane) or 6 (table of the nets' outputs per decision state)");
    const int variant = io->variant == 0 ? NFSP_ROLLOUT_DEFAULT_VARIANT : io->variant;
    NFSP_CHECK_ARG(io->reserve_sms >= 0 && io->reserve_sms < h->sm_count, "reserve_sms must be in [0, %d)", h->sm_count);
    bool direct = false;
    {
        const int rc = nfsp_rollout_direct_args(io, A, &direct);
        if (rc != NFSP_OK) return rc;
    }
    NFSP_CHECK_ARG(!direct || variant == 1 || variant >= 4, "the direct ring append (d_ring) exists in variants 1, 4, 5 and 6 only");
    *variant_out = variant;
    *debug_out = debug;
    *direct_out = direct;
    return NFSP_OK;
}

extern "C" int nfsp_rollout(nfsp_env_t h, int n_steps, double eta, double epsilon, const nfsp_rollout_io *io,
                            void *stream) {
    RolloutArgs A;
    int variant = 0;
    bool debug = false, direct = false;
    {
        const int rc = rollout_args(h, n_steps, eta, epsilon, io, A, &variant, &debug, &direct);
        if (rc != NFSP_OK) return rc;
    }
    DeviceGuard guard(h->device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", h->device);
    if (variant == 6) {
        int rc = states_ensure(h, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        A.pack = h->d_states;
        rc = nfsp_rollout_states_launch(h, A, io, debug, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        h->step += (uint64_t)n_steps;
        return NFSP_OK;
    }
    if (variant == 5) {
        const int rc = nfsp_rollout_pairs_launch(h, A, io, debug, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        h->step += (uint64_t)n_steps;
        return NFSP_OK;
    }
    if (variant == 4) {
        const int rc = nfsp_rollout_sorted_launch(h, A, io, debug, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        h->step += (uint64_t)n_steps;
        return NFSP_OK;
    }
    if (variant == 2 || variant == 3) {
        const int rc = nfsp_ensure_tc_images(h, variant == 3, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
    }
    if (variant == 3) {
        const int rc = nfsp_rollout_tq_launch(h, A, debug, io->reserve_sms, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        h->step += (uint64_t)n_steps;
        return NFSP_OK;
    }
    if (variant == 2) {
        const int rc = nfsp_rollout_tc_launch(h, A, debug, (cudaStream_t)stream);
        if (rc != NFSP_OK) return rc;
        h->step += (uint64_t)n_steps;
        return NFSP_OK;
    }
    const int grid = grid_for(h->n, 32, h->sm_count - io->reserve_sms, 1);  // at least one block of 32 games per CTA
    if (debug && direct) rollout_kernel<true, true><<<grid, kRollThreads, kTabImageBytes, (cudaStream_t)stream>>>(A);
    else if (debug) rollout_kernel<true, false><<<grid, kRollThreads, kTabImageBytes, (cudaStream_t)stream>>>(A);
    else if (direct) rollout_kernel<false, true><<<grid, kRollThreads, kTabImageBytes, (cudaStream_t)stream>>>(A);
    else rollout_kernel<false, false><<<grid, kRollThreads, kTabImageBytes, (cudaStream_t)stream>>>(A);
    NFSP_LAUNCH_CHECK();
    h->step += (uint64_t)n_steps;
    return NFSP_OK;
}

extern "C" int nfsp_rollout_with_weights(nfsp_env_t h, const float *h_weights, float *d_weights, int n_steps, double eta,
                                         double epsilon, const nfsp_rollout_io *io, void *stream) {
    const int rc = h_weights ? nfsp_act_set_weights_from_host(h, h_weights, d_weights, stream) : nfsp_act_set_weights(h, d_weights, stream);
    if (rc != NFSP_OK) return rc;
    return nfsp_rollout(h, n_steps, eta, epsilon, io, stream);
}

extern "C" int nfsp_rollout_runs(const nfsp_env_t *h, int n_runs, int n_steps, const double *eta, const double *epsilon,
                                 const nfsp_rollout_io *io, float *const *d_weights, void *stream) {
    NFSP_CHECK_ARG(h != nullptr && eta != nullptr && epsilon != nullptr && io != nullptr, "null argument");
    NFSP_CHECK_ARG(n_runs >= 1 && n_runs <= NFSP_MAX_RUNS, "n_runs must be in [1, %d]", NFSP_MAX_RUNS);
    RolloutArgs A[NFSP_MAX_RUNS];
    for (int r = 0; r < n_runs; ++r) {
        NFSP_CHECK_ARG(h[r] != nullptr, "null handle of run %d", r);
        for (int q = 0; q < r; ++q) NFSP_CHECK_ARG(h[q] != h[r], "runs %d and %d share a handle", q, r);
        NFSP_CHECK_ARG(io[r].variant == 0 || io[r].variant == 6, "runs play variant 6 (run %d asks for %d)", r, io[r].variant);
        NFSP_CHECK_ARG(!io[r].d_trace && !io[r].d_vec && !io[r].d_forced_vec, "runs have no debug outputs (run %d)", r);
        NFSP_CHECK_ARG(!d_weights || d_weights[r], "null weights of run %d", r);
        int variant = 0;
        bool debug = false, direct = false;
        const int rc = rollout_args(h[r], n_steps, eta[r], epsilon[r], &io[r], A[r], &variant, &debug, &direct);
        if (rc != NFSP_OK) return rc;
        A[r].pack = h[r]->d_states;
        // the shape every run shares: one thread count and one CTA count per run for the whole launch
        NFSP_CHECK_ARG(h[r]->device == h[0]->device, "run %d is on device %d, run 0 on %d", r, h[r]->device, h[0]->device);
        NFSP_CHECK_ARG(h[r]->n == h[0]->n, "run %d has %lld games, run 0 %lld", r, (long long)h[r]->n, (long long)h[0]->n);
        NFSP_CHECK_ARG((A[r].ring[0] != nullptr) == (A[0].ring[0] != nullptr), "runs 0 and %d differ in the record mode (direct rings)", r);
        NFSP_CHECK_ARG(io[r].n_segments == io[0].n_segments, "runs 0 and %d differ in n_segments", r);
        NFSP_CHECK_ARG(io[r].ring_cap == io[0].ring_cap, "runs 0 and %d differ in ring_cap", r);
        NFSP_CHECK_ARG(io[r].reserve_sms == io[0].reserve_sms, "runs 0 and %d differ in reserve_sms", r);
    }
    const int sms = h[0]->sm_count - io[0].reserve_sms;
    NFSP_CHECK_ARG(n_runs <= sms, "%d runs need as many SMs (%d free)", n_runs, sms);
    DeviceGuard guard(h[0]->device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", h[0]->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (d_weights) {  // nfsp_act_set_weights of every run
        const int rc = rebuild_images(h, d_weights, n_runs, st);
        if (rc != NFSP_OK) return rc;
    }
    for (int r = 0; r < n_runs; ++r) {
        const int rc = states_ensure(h[r], st);
        if (rc != NFSP_OK) return rc;
    }
    const int rc = nfsp_rollout_states_runs_launch(h[0], A, n_runs, sms, st);
    if (rc != NFSP_OK) return rc;
    for (int r = 0; r < n_runs; ++r) h[r]->step += (uint64_t)n_steps;
    return NFSP_OK;
}
