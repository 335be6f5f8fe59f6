// Learner half of agent.Agent (agent.py:209-273), SURVEY 8 f-1: one launch computes the minibatch
// gradients of all four acting nets (player x {average policy, best response}) straight from the
// packed records of the memories, into ONE flat fp32 buffer that the host all-reduces over GPUs
// (NCCL) together with the exploitability statistics; a second kernel applies the SGD step.
//
//   best response (agent.py:90-107, 209-253): Q = relu(W2^T relu(W1^T s + b1) + b2), Huber loss on the
//     taken action against r + gamma * (1 - t) * max_a' Q_target(s2), mean over the 3 outputs and the rows;
//   average policy (agent.py:109-116, 255-264): softmax head, categorical cross-entropy against the stored
//     score vector a (Keras semantics: the target is used as is, not renormalised).
// One CTA per net, kRowGroups groups of 64 threads, one thread per hidden unit and group: the thread keeps its column
// of W1, its row of W2 and the matching gradient accumulators in registers; the 64-wide reductions of layer 2 go
// through shuffles and a 64-thread named barrier.  The groups take the minibatch rows round-robin (the kernel is
// latency-bound: three dependent reductions per row) and their partial gradients are summed in a fixed order.
#include <cstring>

#include "common.cuh"

namespace nfsp {

constexpr int kRowGroups = 4;
constexpr int kLearnThreads = 64 * kRowGroups;
constexpr int kGradFloats = 4 * NFSP_NET_PARAMS;

struct LearnerArgs {
    const float *w;          // [4][2179] acting nets, index player*2 + policy
    const float *w_target;   // [2][2179] target best-response nets (agent.py:71-72)
    const uint4 *rl[2];      // rings (M_RL) of the two players
    const int64_t *rl_idx[2];
    const uint4 *sl[2];      // reservoirs (M_SL)
    const int64_t *sl_idx[2];
    int row0, rows;          // minibatch = sampled rows [row0, row0 + rows)
    float gamma;
    int net_mask;            // bit k set = net k takes part (memory large enough, agent.py:215,259)
    int terminal_bootstraps; // reference quirk agent.py:227: `t is True` never holds, terminals bootstrap too
    int others_to_target;    // the two outputs not taken regress to the target net's predictions (agent.py:220,243)
    float *grad;             // [4][2179] mean gradients (+= nothing: overwritten)
    float *stats;            // [NFSP_LEARNER_STATS]
};

struct NetRegs {
    float w1[30], b1, w2[3];
    __device__ __forceinline__ void load(const float *w, int j) {
#pragma unroll
        for (int i = 0; i < 30; ++i) w1[i] = w[i * 64 + j];
        b1 = w[1920 + j];
#pragma unroll
        for (int c = 0; c < 3; ++c) w2[c] = w[1984 + j * 3 + c];
    }
    __device__ __forceinline__ float hidden(uint32_t obs) const {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 30; ++i) acc += ((obs >> i) & 1u) ? w1[i] : 0.f;
        return fmaxf(acc + b1, 0.f);
    }
};

// sum over the 64 threads of a group (2 warps); every thread of the group gets the 3 totals
__device__ __forceinline__ void group_sync(int group) { asm volatile("bar.sync %0, 64;" ::"r"(1 + group) : "memory"); }
__device__ __forceinline__ void cta_sum3(float &a, float &b, float &c, float (*red)[2][4], int slot, int group) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
        c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    }
    const int warp = (threadIdx.x >> 5) & 1;
    if ((threadIdx.x & 31) == 0) { red[slot][warp][0] = a; red[slot][warp][1] = b; red[slot][warp][2] = c; }
    group_sync(group);
    a = red[slot][0][0] + red[slot][1][0];
    b = red[slot][0][1] + red[slot][1][1];
    c = red[slot][0][2] + red[slot][1][2];
}

// the same for nine values at once: the three forward passes of a best-response row (online Q(s), target Q(s2), target
// Q(s)) do not depend on each other, so they share one round of shuffles and ONE barrier instead of three
__device__ __forceinline__ void cta_sum9(float (&v)[9], float (*red)[2][4], int group) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 9; ++k) v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o);
    }
    const int warp = (threadIdx.x >> 5) & 1;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 9; ++k) red[k / 3][warp][k % 3] = v[k];
    }
    group_sync(group);
#pragma unroll
    for (int k = 0; k < 9; ++k) v[k] = red[k / 3][0][k % 3] + red[k / 3][1][k % 3];
}

// Per-thread state of one net: the thread's column of W1, its row of W2, the output biases, and -- for a best-response
// net -- the same of the target net.
struct NetState {
    NetRegs W, T;
    float b2[3], t2[3];
    __device__ __forceinline__ void load(const LearnerArgs &A, int net, int j) {
        const float *w = A.w + net * NFSP_NET_PARAMS;
        W.load(w, j);
        b2[0] = w[2176]; b2[1] = w[2177]; b2[2] = w[2178];
        t2[0] = t2[1] = t2[2] = 0.f;
        if (net & 1) {
            const float *wt = A.w_target + (net >> 1) * NFSP_NET_PARAMS;
            T.load(wt, j);
            t2[0] = wt[2176]; t2[1] = wt[2177]; t2[2] = wt[2178];
        }
    }
};

// One SGD step's sums over the rows [row0, row0 + rows) for net `net`: every group takes its rows round-robin, the
// groups' partial sums meet in shared memory and are added in group order (deterministic).  On return (after a CTA
// barrier) part[0][i][j] holds, for hidden unit j, the summed gradients of W1 rows i = 0..29, b1 (30), W2 (31..33) and
// part[0][34][0..4] those of b2, the loss sum and the exploitability-proxy sum.
// s_rec: the net's sampled records of rows [s_base, s_base + kMaxFitRows) prefetched into shared memory (the two
// dependent global reads per row -- index, then record -- were most of a row's latency), or nullptr.
constexpr int kMaxFitRows = NFSP_FIT_ROWS_MAX_MINIBATCH;
__device__ __forceinline__ void prefetch_rows(const LearnerArgs &A, int net, int base, int rows, uint4 *s_rec) {
    const int player = net >> 1;
    const uint4 *mem = (net & 1) ? A.rl[player] : A.sl[player];
    const int64_t *idx = (net & 1) ? A.rl_idx[player] : A.sl_idx[player];
    const int stride = (net & 1) ? 1 : 2;  // a reservoir slot is 32 bytes, the record first (buffer_kernels.cu)
    for (int r = threadIdx.x; r < rows; r += blockDim.x) s_rec[r] = mem[idx[base + r] * stride];
    __syncthreads();
}
// Huber loss (agent.py:91-99) of the best-response net on one row, averaged over the three outputs as Keras does, and its
// derivative w.r.t. the pre-activations z.  The taken action regresses to the TD target; the other two outputs have zero
// error by default, or -- `others_to_target`, what agent.py:220-243 does with `target = target_br_model.predict(s_batch)`
// -- regress to the target net's own predictions qt on s.
__device__ __forceinline__ float br_loss(float z0, float z1, float z2, float qt0, float qt1, float qt2, uint32_t a, float td,
                                         int others_to_target, float &dz0, float &dz1, float &dz2) {
    const float z[3] = {z0, z1, z2}, qt[3] = {qt0, qt1, qt2};
    float dz[3], loss = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const bool taken = (uint32_t)c == a;
        const float err = (taken ? td : qt[c]) - fmaxf(z[c], 0.f);
        const float ae = fabsf(err);
        const bool on = taken || others_to_target;
        loss += on ? (ae > 1.f ? ae - 0.5f : 0.5f * err * err) * (1.0f / 3.0f) : 0.f;
        dz[c] = on ? -(ae > 1.f ? copysignf(1.f, err) : err) * (1.0f / 3.0f) * (z[c] > 0.f ? 1.f : 0.f) : 0.f;
    }
    dz0 = dz[0]; dz1 = dz[1]; dz2 = dz[2];
    return loss;
}

__device__ __forceinline__ void step_sums(const LearnerArgs &A, const NetState &N, int net, int row0, int rows,
                                          float (*red_all)[4][2][4], float (*part)[40][64], const uint4 *s_rec, int s_base) {
    const int player = net >> 1, is_br = net & 1, group = threadIdx.x >> 6, j = threadIdx.x & 63;
    float (*red)[2][4] = red_all[group];
    const NetRegs &W = N.W, &T = N.T;
    const float b2_0 = N.b2[0], b2_1 = N.b2[1], b2_2 = N.b2[2], t2_0 = N.t2[0], t2_1 = N.t2[1], t2_2 = N.t2[2];
    float gw1[30], gb1 = 0.f, gw2[3] = {0.f, 0.f, 0.f}, gb2[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 30; ++i) gw1[i] = 0.f;
    float loss = 0.f, expl = 0.f;
    for (int r = group; r < rows; r += kRowGroups) {
        const int row = row0 + r;
        uint32_t s;
        float dz0, dz1, dz2;
        if (is_br) {
            const uint4 rec = s_rec ? s_rec[row - s_base] : A.rl[player][A.rl_idx[player][row]];
            s = rec.x;
            const uint32_t a = rec.w & 0xFFu, term = (rec.w >> 8) & 0xFFu;
            const float rew = __uint_as_float(rec.z);
            // online Q(s), target Q(s2), target Q(s) (exploitability proxy, agent.py:234-238)
            const float h = W.hidden(s), ht = T.hidden(rec.y), hs = T.hidden(s);
            float v[9] = {h * W.w2[0], h * W.w2[1], h * W.w2[2], ht * T.w2[0], ht * T.w2[1], ht * T.w2[2],
                          hs * T.w2[0], hs * T.w2[1], hs * T.w2[2]};
            cta_sum9(v, red, group);
            float z0 = v[0], z1 = v[1], z2 = v[2];
            const float y0 = v[3], y1 = v[4], y2 = v[5], e0 = v[6], e1 = v[7], e2 = v[8];
            const float qt0 = fmaxf(e0 + t2_0, 0.f), qt1 = fmaxf(e1 + t2_1, 0.f), qt2 = fmaxf(e2 + t2_2, 0.f);
            expl += fmaxf(fmaxf(qt0, qt1), qt2);
            const float qn = fmaxf(fmaxf(fmaxf(y0 + t2_0, 0.f), fmaxf(y1 + t2_1, 0.f)), fmaxf(y2 + t2_2, 0.f));
            const float target = rew + ((term && !A.terminal_bootstraps) ? 0.f : A.gamma * qn);
            z0 += b2_0; z1 += b2_1; z2 += b2_2;
            loss += br_loss(z0, z1, z2, qt0, qt1, qt2, a, target, A.others_to_target, dz0, dz1, dz2);
            group_sync(group);  // red[] slots are reused by the next row
            const float dh = (h > 0.f) ? (W.w2[0] * dz0 + W.w2[1] * dz1 + W.w2[2] * dz2) : 0.f;
            gw2[0] += h * dz0; gw2[1] += h * dz1; gw2[2] += h * dz2;
            gb1 += dh;
#pragma unroll
            for (int i = 0; i < 30; ++i) gw1[i] += ((s >> i) & 1u) ? dh : 0.f;
        } else {
            const uint4 rec = s_rec ? s_rec[row - s_base] : A.sl[player][2 * A.sl_idx[player][row]];
            s = rec.x;
            const float ya = __uint_as_float(rec.y), yb = __uint_as_float(rec.z), yc = __uint_as_float(rec.w);
            const float h = W.hidden(s);
            float z0 = h * W.w2[0], z1 = h * W.w2[1], z2 = h * W.w2[2];
            cta_sum3(z0, z1, z2, red, 0, group);
            z0 += b2_0; z1 += b2_1; z2 += b2_2;
            const float m = fmaxf(z0, fmaxf(z1, z2));
            const float x0 = expf(z0 - m), x1 = expf(z1 - m), x2 = expf(z2 - m);
            const float inv = 1.0f / (x0 + x1 + x2);
            const float p0 = x0 * inv, p1 = x1 * inv, p2 = x2 * inv;
            const float ysum = ya + yb + yc;
            loss += -(ya * logf(fmaxf(p0, 1e-7f)) + yb * logf(fmaxf(p1, 1e-7f)) + yc * logf(fmaxf(p2, 1e-7f)));
            dz0 = p0 * ysum - ya; dz1 = p1 * ysum - yb; dz2 = p2 * ysum - yc;
            group_sync(group);
            const float dh = (h > 0.f) ? (W.w2[0] * dz0 + W.w2[1] * dz1 + W.w2[2] * dz2) : 0.f;
            gw2[0] += h * dz0; gw2[1] += h * dz1; gw2[2] += h * dz2;
            gb1 += dh;
#pragma unroll
            for (int i = 0; i < 30; ++i) gw1[i] += ((s >> i) & 1u) ? dh : 0.f;
        }
        gb2[0] += dz0; gb2[1] += dz1; gb2[2] += dz2;
    }
#pragma unroll
    for (int i = 0; i < 30; ++i) part[group][i][j] = gw1[i];
    part[group][30][j] = gb1;
#pragma unroll
    for (int c = 0; c < 3; ++c) part[group][31 + c][j] = gw2[c];
    if (j == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) part[group][34][c] = gb2[c];
        part[group][34][3] = loss;
        part[group][34][4] = expl;
    }
    __syncthreads();
    if (group == 0) {
#pragma unroll
        for (int i = 0; i < 34; ++i) {
            float v = part[0][i][j];
#pragma unroll
            for (int k = 1; k < kRowGroups; ++k) v += part[k][i][j];
            part[0][i][j] = v;
        }
        if (j < 5) {
            float v = part[0][34][j];
#pragma unroll
            for (int k = 1; k < kRowGroups; ++k) v += part[k][34][j];
            part[0][34][j] = v;
        }
    }
    __syncthreads();
}

// stats: [0,1] exploitability-proxy sums of the BR nets, [2,3] their row counts, [4..7] loss sums per net
__device__ __forceinline__ void write_stats(float *stats, int net, int rows, float (*part)[40][64]) {
    if (threadIdx.x == 0) {
        stats[4 + net] = part[0][34][3];
        if (net & 1) { stats[net >> 1] = part[0][34][4]; stats[2 + (net >> 1)] = (float)rows; }
    }
}

__global__ void __launch_bounds__(kLearnThreads)
learner_grad_kernel(const LearnerArgs A) {
    __shared__ float red_all[kRowGroups][4][2][4];
    __shared__ float part[kRowGroups][40][64];  // per group: gw1[30], gb1, gw2[3] per hidden unit; row 34: gb2, loss, expl
    const int net = blockIdx.x, j = threadIdx.x & 63;
    float *g = A.grad + net * NFSP_NET_PARAMS;
    if (!((A.net_mask >> net) & 1)) {
        for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kLearnThreads) g[e] = 0.f;
        return;
    }
    __shared__ uint4 s_rec[kMaxFitRows];
    const bool pre = A.rows <= kMaxFitRows;
    if (pre) prefetch_rows(A, net, A.row0, A.rows, s_rec);
    NetState N;
    N.load(A, net, j);
    step_sums(A, N, net, A.row0, A.rows, red_all, part, pre ? s_rec : nullptr, A.row0);
    write_stats(A.stats, net, A.rows, part);
    if (threadIdx.x >= 64) return;
    const float inv_rows = 1.0f / (float)A.rows;
#pragma unroll
    for (int i = 0; i < 30; ++i) g[i * 64 + j] = part[0][i][j] * inv_rows;
    g[1920 + j] = part[0][30][j] * inv_rows;
#pragma unroll
    for (int c = 0; c < 3; ++c) g[1984 + j * 3 + c] = part[0][31 + c][j] * inv_rows;
    if (j < 3) g[2176 + j] = part[0][34][j] * inv_rows;
}

// Keras' fit() of all four nets on ONE GPU in one launch (no collective between the SGD steps): n_steps slices
// [row0_k, row0_k + rows_k) of the sampled minibatch, each step = the sums above, then w -= lr * mean gradient applied
// to the weights every thread holds in registers (all row groups keep the same copy).  The statistics are those of the
// first step, as the host-driven sequence reports them.
// The step schedule (and, with several GPUs, the peers): shared by every run of a launch.
struct FitSchedule {
    int n_steps, minibatch;
    int row0[NFSP_MAX_FIT_STEPS], rows[NFSP_MAX_FIT_STEPS];
    // several GPUs training together: every rank's exchange buffer as this process sees it (peer memory over NVLink)
    int world, rank;
    float *peer[NFSP_MAX_PEERS];
    uint32_t epoch0;     // SGD steps exchanged through these buffers so far
    uint32_t *err;       // set to 1 if a peer did not answer in time
    float *mc;           // multicast mapping of all ranks' buffers (NVLS), or null
};
// What a fit reads per run: the learner's arguments, the output weights and the four learning rates.
struct FitRun {
    LearnerArgs A;
    float *w_out;  // [4][2179], may alias A.w
    float lr[4];
};

// Exchange buffer of one rank (the RECEIVER owns it): two parities x four nets x one slot per sending rank of kPeerSlot
// 8-byte words {value, epoch} -- 2179 mean gradients, then loss sum, exploitability sum, rows.  A sender PUSHES its values
// into the slot it has in every rank's buffer (its own included); a receiver polls its own memory until a word carries
// the step's epoch.  The 8-byte store is atomic, so a word is either the old epoch's or complete: no flags, no fences,
// no round trip (NCCL's LL protocol).  Round 1 published into the sender's buffer, fenced at system scope, flagged the
// peers and had them read the values back over NVLink: ~15 us per SGD step at 8 GPUs.
constexpr int kPeerSlot = 2184;
static_assert(2 * 4 * NFSP_MAX_PEERS * kPeerSlot * 2 <= NFSP_PEER_BUF_FLOATS, "exchange buffer too small");
__device__ __forceinline__ size_t ll_index(uint32_t parity, int net, int src, int e) {
    return ((size_t)((parity * 4u + (uint32_t)net) * NFSP_MAX_PEERS + (uint32_t)src)) * kPeerSlot + (size_t)e;
}
__device__ __forceinline__ void ll_store(float *buf, size_t idx, float v, uint32_t epoch) {
    asm volatile("st.volatile.global.v2.b32 [%0], {%1, %2};" ::"l"(reinterpret_cast<uint2 *>(buf) + idx), "r"(__float_as_uint(v)),
                 "r"(epoch)
                 : "memory");
}
// spins until the word carries `epoch`; gives up after ~2 s (a peer is gone; never hang the GPU) and reports it in *lost
__device__ __forceinline__ float ll_wait(const float *buf, size_t idx, uint32_t epoch, int *lost) {
    const uint2 *p = reinterpret_cast<const uint2 *>(buf) + idx;
    uint32_t v, ep;
    long long t0 = 0;
    for (int spin = 0;; ++spin) {
        asm volatile("ld.volatile.global.v2.b32 {%0, %1}, [%2];" : "=r"(v), "=r"(ep) : "l"(p) : "memory");
        if (ep == epoch) break;
        if (spin == 64) t0 = clock64();
        if (spin > 64 && clock64() - t0 > 4000000000ll) {
            *lost = 1;
            break;
        }
    }
    return __uint_as_float(v);
}
__device__ __forceinline__ float ld_volatile_f32(const float *p) {
    float v;
    asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
// the register kernel's work on net `net` of run P
__device__ __forceinline__ void fit_regs_net(const FitSchedule &F, const FitRun &P, int net) {
    __shared__ float red_all[kRowGroups][4][2][4];
    __shared__ float part[kRowGroups][40][64];
    const LearnerArgs &A = P.A;
    const int j = threadIdx.x & 63;
    if (!((A.net_mask >> net) & 1)) {
        if (P.w_out != A.w)
            for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kLearnThreads) P.w_out[net * NFSP_NET_PARAMS + e] = A.w[net * NFSP_NET_PARAMS + e];
        return;
    }
    __shared__ uint4 s_rec[kMaxFitRows];
    const bool pre = F.minibatch <= kMaxFitRows;
    if (pre) prefetch_rows(A, net, 0, F.minibatch, s_rec);
    NetState N;
    N.load(A, net, j);
    const float lr = P.lr[net];
    for (int k = 0; k < F.n_steps; ++k) {
        step_sums(A, N, net, F.row0[k], F.rows[k], red_all, part, pre ? s_rec : nullptr, 0);
        if (k == 0) write_stats(A.stats, net, F.rows[k], part);
        const float inv_rows = 1.0f / (float)F.rows[k];
        // the same arithmetic as sgd_apply_kernel on the stored mean gradient: w -= lr * 1.0f * (sum * inv_rows)
#pragma unroll
        for (int i = 0; i < 30; ++i) N.W.w1[i] -= lr * 1.0f * (part[0][i][j] * inv_rows);
        N.W.b1 -= lr * 1.0f * (part[0][30][j] * inv_rows);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            N.W.w2[c] -= lr * 1.0f * (part[0][31 + c][j] * inv_rows);
            N.b2[c] -= lr * 1.0f * (part[0][34][c] * inv_rows);
        }
        __syncthreads();  // part[] is rewritten by the next step
    }
    if (threadIdx.x >= 64) return;
    float *w = P.w_out + net * NFSP_NET_PARAMS;
#pragma unroll
    for (int i = 0; i < 30; ++i) w[i * 64 + j] = N.W.w1[i];
    w[1920 + j] = N.W.b1;
#pragma unroll
    for (int c = 0; c < 3; ++c) w[1984 + j * 3 + c] = N.W.w2[c];
    if (j < 3) w[2176 + j] = N.b2[j];
}
__global__ void __launch_bounds__(kLearnThreads)
learner_fit_kernel(const FitSchedule S, const FitRun P) { fit_regs_net(S, P, blockIdx.x); }

// ---- fit(), the row-parallel formulation ------------------------------------------------------------
// The register kernel above is bound by instruction latency: a CTA of 256 threads per net, eight rows one after the
// other per 64-thread group, ~450 dependent instructions per row.  Here a net has 1024 threads and ONE WARP PER ROW (two
// hidden units per lane: the 64-wide sums of layer 2 are shuffles, no barrier), the weights live in shared memory in the
// reference's flat layout, so the hidden layer is one conflict-free LDS per SET input bit (<= 10) in the same order
// as the register kernel adds them.  A second phase assembles the gradient of each weight from the rows' dh / h / dz in
// row order and applies the SGD update in place.  Two barriers per SGD step.
constexpr int kRowThreads = 1024, kRowWarps = kRowThreads / 32, kMaxStepRows = NFSP_FIT_ROWS_MAX_STEP;
struct RowFitSmem {
    float w[2180], wt[2180];          // online net, target net (best response only)
    uint4 rec[kMaxFitRows];           // the sampled records of the minibatch
    float dh[kMaxStepRows][64], h[kMaxStepRows][64];
    float dz[kMaxStepRows][4];
    uint32_t obs[kMaxStepRows];
    float loss[kMaxStepRows], expl[kMaxStepRows];
};
__device__ __forceinline__ void warp_sum9(float (&v)[9]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 9; ++k) v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o);
    }
}
// the row-parallel kernel's work on net `net` of run P
__device__ __forceinline__ void fit_rows_net(const FitSchedule &F, const FitRun &P, int net) {
    extern __shared__ __align__(16) unsigned char fit_smem_raw[];
    RowFitSmem &S = *reinterpret_cast<RowFitSmem *>(fit_smem_raw);
    __shared__ int s_peer_lost;  // a peer did not answer within the time limit of the gradient exchange
    const LearnerArgs &A = P.A;
    const int player = net >> 1, is_br = net & 1, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) s_peer_lost = 0;
    if (!((A.net_mask >> net) & 1)) {
        if (P.w_out != A.w)
            for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) P.w_out[net * NFSP_NET_PARAMS + e] = A.w[net * NFSP_NET_PARAMS + e];
        return;
    }
    for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) {
        S.w[e] = A.w[net * NFSP_NET_PARAMS + e];
        if (is_br) S.wt[e] = A.w_target[player * NFSP_NET_PARAMS + e];
    }
    prefetch_rows(A, net, 0, F.minibatch, S.rec);  // ends with a CTA barrier
    const float lr = P.lr[net];
    for (int k = 0; k < F.n_steps; ++k) {
        const int row0 = F.row0[k], rows = F.rows[k];
        // phase 1: forward, loss, dz and dh of one row per warp
        for (int r = warp; r < rows; r += kRowWarps) {
            const uint4 rec = S.rec[row0 + r];
            const uint32_t s = rec.x;
            const int j0 = lane, j1 = lane + 32;
            // the hidden units of this lane for the online net on s and, for a best-response net, the target net on s
            // and s2: ONE loop over the set bits of s (four independent loads per bit) and one over those of s2, each
            // accumulator summed in ascending input order as in NetRegs::hidden
            float h0 = 0.f, h1 = 0.f, hs0 = 0.f, hs1 = 0.f, ht0 = 0.f, ht1 = 0.f;
            for (uint32_t m = s & 0x3FFFFFFFu; m; m &= m - 1u) {
                const int i = (__ffs(m) - 1) * 64;
                h0 += S.w[i + j0];
                h1 += S.w[i + j1];
                if (is_br) {
                    hs0 += S.wt[i + j0];
                    hs1 += S.wt[i + j1];
                }
            }
            h0 = fmaxf(h0 + S.w[1920 + j0], 0.f);
            h1 = fmaxf(h1 + S.w[1920 + j1], 0.f);
            float dz0, dz1, dz2, loss, expl = 0.f;
            if (is_br) {
                const uint32_t a = rec.w & 0xFFu, term = (rec.w >> 8) & 0xFFu;
                const float rew = __uint_as_float(rec.z);
                for (uint32_t m = rec.y & 0x3FFFFFFFu; m; m &= m - 1u) {
                    const int i = (__ffs(m) - 1) * 64;
                    ht0 += S.wt[i + j0];
                    ht1 += S.wt[i + j1];
                }
                hs0 = fmaxf(hs0 + S.wt[1920 + j0], 0.f);
                hs1 = fmaxf(hs1 + S.wt[1920 + j1], 0.f);
                ht0 = fmaxf(ht0 + S.wt[1920 + j0], 0.f);
                ht1 = fmaxf(ht1 + S.wt[1920 + j1], 0.f);
                float v[9];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    v[c] = h0 * S.w[1984 + j0 * 3 + c] + h1 * S.w[1984 + j1 * 3 + c];
                    v[3 + c] = ht0 * S.wt[1984 + j0 * 3 + c] + ht1 * S.wt[1984 + j1 * 3 + c];
                    v[6 + c] = hs0 * S.wt[1984 + j0 * 3 + c] + hs1 * S.wt[1984 + j1 * 3 + c];
                }
                warp_sum9(v);
                const float t2_0 = S.wt[2176], t2_1 = S.wt[2177], t2_2 = S.wt[2178];
                const float qt0 = fmaxf(v[6] + t2_0, 0.f), qt1 = fmaxf(v[7] + t2_1, 0.f), qt2 = fmaxf(v[8] + t2_2, 0.f);
                expl = fmaxf(fmaxf(qt0, qt1), qt2);  // agent.py:234-238
                const float qn = fmaxf(fmaxf(fmaxf(v[3] + t2_0, 0.f), fmaxf(v[4] + t2_1, 0.f)), fmaxf(v[5] + t2_2, 0.f));
                const float target = rew + ((term && !A.terminal_bootstraps) ? 0.f : A.gamma * qn);
                const float z0 = v[0] + S.w[2176], z1 = v[1] + S.w[2177], z2 = v[2] + S.w[2178];
                loss = br_loss(z0, z1, z2, qt0, qt1, qt2, a, target, A.others_to_target, dz0, dz1, dz2);
            } else {
                const float ya = __uint_as_float(rec.y), yb = __uint_as_float(rec.z), yc = __uint_as_float(rec.w);
                float v[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int c = 0; c < 3; ++c) v[c] = h0 * S.w[1984 + j0 * 3 + c] + h1 * S.w[1984 + j1 * 3 + c];
                warp_sum9(v);
                const float z0 = v[0] + S.w[2176], z1 = v[1] + S.w[2177], z2 = v[2] + S.w[2178];
                const float m = fmaxf(z0, fmaxf(z1, z2));
                const float x0 = expf(z0 - m), x1 = expf(z1 - m), x2 = expf(z2 - m);
                const float inv = 1.0f / (x0 + x1 + x2);
                const float p0 = x0 * inv, p1 = x1 * inv, p2 = x2 * inv;
                const float ysum = ya + yb + yc;
                loss = -(ya * logf(fmaxf(p0, 1e-7f)) + yb * logf(fmaxf(p1, 1e-7f)) + yc * logf(fmaxf(p2, 1e-7f)));
                dz0 = p0 * ysum - ya; dz1 = p1 * ysum - yb; dz2 = p2 * ysum - yc;
            }
            S.h[r][j0] = h0;
            S.h[r][j1] = h1;
            S.dh[r][j0] = h0 > 0.f ? (S.w[1984 + j0 * 3] * dz0 + S.w[1985 + j0 * 3] * dz1 + S.w[1986 + j0 * 3] * dz2) : 0.f;
            S.dh[r][j1] = h1 > 0.f ? (S.w[1984 + j1 * 3] * dz0 + S.w[1985 + j1 * 3] * dz1 + S.w[1986 + j1 * 3] * dz2) : 0.f;
            if (lane == 0) {
                S.dz[r][0] = dz0; S.dz[r][1] = dz1; S.dz[r][2] = dz2;
                S.obs[r] = s;
                S.loss[r] = loss;
                S.expl[r] = expl;
            }
        }
        __syncthreads();
        // phase 2: every weight's gradient summed over the rows in row order, then w -= lr * mean gradient in place.
        // With peers the mean gradient goes into this rank's exchange buffer first and the update uses the sum over
        // all ranks' buffers, read over NVLink in rank order: the all-reduce of the step, inside the kernel.
        const float inv_rows = 1.0f / (float)rows;
        const bool peers = F.world > 1;
        const uint32_t epoch = F.epoch0 + (uint32_t)k + 1u, parity = epoch & 1u;
        auto apply = [&](int e, float g) {
            if (peers) {
                // one store through the multicast mapping reaches every rank's buffer (the switch replicates it); without
                // NVLS the SM sends `world` copies itself
                const float v = g * inv_rows;
                if (F.mc) ll_store(F.mc, ll_index(parity, net, F.rank, e), v, epoch);
                else
                    for (int r = 0; r < F.world; ++r) ll_store(F.peer[r], ll_index(parity, net, F.rank, e), v, epoch);
            } else {
                S.w[e] -= lr * 1.0f * (g * inv_rows);
            }
        };
        // W1: warp i owns input i and both halves of the hidden units.  Only ~30 % of the input bits are set: the rows
        // that have bit i come from one ballot (lane r tests row r) and only those are added, in row order -- adding the
        // zeros of the other rows would not change a bit of the sum.
        for (int i = warp; i < 30; i += kRowWarps) {
            float g0 = 0.f, g1 = 0.f;
            for (int rb = 0; rb < rows; rb += 32) {
                const int r = rb + lane;
                for (uint32_t m = __ballot_sync(0xFFFFFFFFu, r < rows && ((S.obs[r] >> i) & 1u)); m; m &= m - 1u) {
                    const int rr = rb + __ffs(m) - 1;
                    g0 += S.dh[rr][lane];
                    g1 += S.dh[rr][lane + 32];
                }
            }
            apply(i * 64 + lane, g0);
            apply(i * 64 + lane + 32, g1);
        }
        // b1, W2, b2: one element per thread, summed over the rows in row order
        for (int e = 1920 + threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) {
            float g = 0.f;
            if (e < 1984) {
                const int j = e - 1920;
#pragma unroll 8
                for (int r = 0; r < rows; ++r) g += S.dh[r][j];
            } else if (e < 2176) {
                const int j = (e - 1984) / 3, c = (e - 1984) - 3 * j;
#pragma unroll 8
                for (int r = 0; r < rows; ++r) g += S.h[r][j] * S.dz[r][c];
            } else {
                const int c = e - 2176;
                for (int r = 0; r < rows; ++r) g += S.dz[r][c];
            }
            apply(e, g);
        }
        if (k == 0 && threadIdx.x == 0) {  // the statistics of the first step, as the host-driven sequence reports them
            float ls = 0.f, ex = 0.f;
            for (int r = 0; r < rows; ++r) { ls += S.loss[r]; ex += S.expl[r]; }
            if (peers) {
                for (int r = 0; r < (F.mc ? 1 : F.world); ++r) {
                    float *dst = F.mc ? F.mc : F.peer[r];
                    ll_store(dst, ll_index(parity, net, F.rank, 2180), ls, epoch);
                    ll_store(dst, ll_index(parity, net, F.rank, 2181), ex, epoch);
                    ll_store(dst, ll_index(parity, net, F.rank, 2182), (float)rows, epoch);
                }
            } else {
                A.stats[4 + net] = ls;
                if (is_br) { A.stats[player] = ex; A.stats[2 + player] = (float)rows; }
            }
        }
        if (peers) {
            // every thread of this CTA has read S.w for this step's gradients: the update may begin.  Each thread sums its
            // elements over the ranks' slots IN RANK ORDER as they arrive -- the same sum, and with it bit-identical
            // weights, on every rank
            __syncthreads();
            const float *mybuf = F.peer[F.rank];
            const float scale = 1.0f / (float)F.world;
            int lost = 0;
            for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) {
                float g = 0.f;
                for (int r = 0; r < F.world; ++r) g += ll_wait(mybuf, ll_index(parity, net, r, e), epoch, &lost);
                S.w[e] -= lr * scale * g;
            }
            if (k == 0 && threadIdx.x == 0) {
                float ls = 0.f, ex = 0.f, rw = 0.f;
                for (int r = 0; r < F.world; ++r) {
                    ls += ll_wait(mybuf, ll_index(parity, net, r, 2180), epoch, &lost);
                    ex += ll_wait(mybuf, ll_index(parity, net, r, 2181), epoch, &lost);
                    rw += ll_wait(mybuf, ll_index(parity, net, r, 2182), epoch, &lost);
                }
                A.stats[4 + net] = ls;
                if (is_br) { A.stats[player] = ex; A.stats[2 + player] = rw; }
            }
            if (lost) {
                *F.err = 1u;
                s_peer_lost = 1;
            }
            __syncthreads();
            if (s_peer_lost) {
                // a silent peer's slot is stale: summing it would make the replicas differ silently.  Give up on this net
                // instead: no further steps, NaN weights out (nobody can mistake them for a result), the error word set for
                // Learner.check_peers()
                for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) S.w[e] = __int_as_float(0x7FC00000);
                break;
            }
        }
        __syncthreads();
    }
    for (int e = threadIdx.x; e < NFSP_NET_PARAMS; e += kRowThreads) P.w_out[net * NFSP_NET_PARAMS + e] = S.w[e];
}
__global__ void __launch_bounds__(kRowThreads, 1)
learner_fit_rows_kernel(const FitSchedule S, const FitRun P) { fit_rows_net(S, P, blockIdx.x); }

// ---- the fits of independent runs in one launch (nfsp_learner_fit_runs): CTA 4 r + k = net k of run r ------------------
struct FitRuns {
    FitRun run[NFSP_MAX_RUNS];  // first: the row-parallel kernel then schedules as it did before the split (sass_check r05)
    FitSchedule S;              // world = 1
};
__global__ void __launch_bounds__(kLearnThreads)
learner_fit_runs_kernel(const __grid_constant__ FitRuns R) { fit_regs_net(R.S, R.run[blockIdx.x >> 2], blockIdx.x & 3); }
__global__ void __launch_bounds__(kRowThreads, 1)
learner_fit_rows_runs_kernel(const __grid_constant__ FitRuns R) { fit_rows_net(R.S, R.run[blockIdx.x >> 2], blockIdx.x & 3); }

// w[k] -= lr[k] * scale * grad[k]   (keras.optimizers.SGD without momentum, agent.py:45-46)
__global__ void sgd_apply_kernel(float *__restrict__ w, const float *__restrict__ grad, float lr0, float lr1, float lr2,
                                 float lr3, float scale) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= kGradFloats) return;
    const int net = e / NFSP_NET_PARAMS;
    const float lr = net == 0 ? lr0 : (net == 1 ? lr1 : (net == 2 ? lr2 : lr3));
    w[e] -= lr * scale * grad[e];
}

}  // namespace nfsp

using namespace nfsp;

static int make_learner_args(const nfsp_learner_io *io, LearnerArgs &A) {
    NFSP_CHECK_ARG(io != nullptr && io->d_weights && io->d_target_weights && io->d_stats, "null argument");
    A.w = io->d_weights; A.w_target = io->d_target_weights;
    for (int p = 0; p < 2; ++p) {
        A.rl[p] = (const uint4 *)io->d_rl[p]; A.rl_idx[p] = io->d_rl_idx[p];
        A.sl[p] = (const uint4 *)io->d_sl[p]; A.sl_idx[p] = io->d_sl_idx[p];
        if ((io->net_mask >> (2 * p + 1)) & 1) NFSP_CHECK_ARG(A.rl[p] && A.rl_idx[p], "missing RL batch of player %d", p);
        if ((io->net_mask >> (2 * p)) & 1) NFSP_CHECK_ARG(A.sl[p] && A.sl_idx[p], "missing SL batch of player %d", p);
    }
    A.row0 = io->row0; A.rows = io->rows; A.gamma = io->gamma; A.net_mask = io->net_mask;
    A.terminal_bootstraps = io->terminal_bootstraps; A.others_to_target = io->others_to_target;
    A.grad = io->d_grad; A.stats = io->d_stats;
    return NFSP_OK;
}

extern "C" int nfsp_learner_grads(const nfsp_learner_io *io, void *stream) {
    LearnerArgs A;
    const int rc = make_learner_args(io, A);
    if (rc != NFSP_OK) return rc;
    NFSP_CHECK_ARG(A.grad != nullptr, "null gradient buffer");
    NFSP_CHECK_ARG(io->rows >= 1 && io->row0 >= 0, "bad minibatch slice");
    learner_grad_kernel<<<4, kLearnThreads, 0, (cudaStream_t)stream>>>(A);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

// the SGD steps of Keras' fit(batch_size = fit_batch, epochs): slices [0, fit_batch), [fit_batch, 2 fit_batch), ... of the
// minibatch, `epochs` times; one GPU unless `peers` is given
static int fit_schedule(int minibatch, int fit_batch, int epochs, const nfsp_peers *peers, FitSchedule &F) {
    NFSP_CHECK_ARG(minibatch >= 1 && fit_batch >= 1 && epochs >= 1, "bad fit geometry");
    F.minibatch = minibatch;
    F.n_steps = 0;
    for (int e = 0; e < epochs; ++e)
        for (int row0 = 0; row0 < minibatch; row0 += fit_batch) {
            NFSP_CHECK_ARG(F.n_steps < NFSP_MAX_FIT_STEPS, "more than %d SGD steps per fit", NFSP_MAX_FIT_STEPS);
            F.row0[F.n_steps] = row0;
            F.rows[F.n_steps] = minibatch - row0 < fit_batch ? minibatch - row0 : fit_batch;
            ++F.n_steps;
        }
    F.world = 1; F.rank = 0; F.epoch0 = 0u; F.err = nullptr; F.mc = nullptr;
    for (int r = 0; r < NFSP_MAX_PEERS; ++r) F.peer[r] = nullptr;
    if (peers) {
        F.world = peers->world; F.rank = peers->rank; F.epoch0 = peers->epoch0; F.err = peers->d_err;
        F.mc = (float *)peers->d_mc;
        for (int r = 0; r < peers->world; ++r) F.peer[r] = (float *)peers->d_buf[r];
    }
    return NFSP_OK;
}

// The fits of n_runs runs on one schedule, CTA 4 r + k = net k of run r: the row-parallel kernel (one warp per row,
// weights in shared memory) when the minibatch and a step fit its shared memory, the register kernel otherwise; one run
// launches the single-run kernels, which read their arguments from the constant bank.
static int learner_fit(const nfsp_learner_io *io, int n_runs, int minibatch, int fit_batch, int epochs, const float *lr,
                       float *const *d_weights_out, const nfsp_peers *peers, cudaStream_t st) {
    NFSP_CHECK_ARG(io && lr && d_weights_out, "null argument");
    FitRuns R;
    int rc = fit_schedule(minibatch, fit_batch, epochs, peers, R.S);
    if (rc != NFSP_OK) return rc;
    for (int r = 0; r < n_runs; ++r) {
        NFSP_CHECK_ARG(d_weights_out[r], "null output weights of run %d", r);
        rc = make_learner_args(io + r, R.run[r].A);
        if (rc != NFSP_OK) return rc;
        R.run[r].w_out = d_weights_out[r];
        for (int k = 0; k < 4; ++k) R.run[r].lr[k] = lr[4 * r + k];
    }
    const bool rows = minibatch <= kMaxFitRows && fit_batch <= kMaxStepRows;
    void (*single)(FitSchedule, FitRun) = rows ? learner_fit_rows_kernel : learner_fit_kernel;
    void (*batch)(FitRuns) = rows ? learner_fit_rows_runs_kernel : learner_fit_runs_kernel;
    const int threads = rows ? kRowThreads : kLearnThreads, smem = rows ? (int)sizeof(RowFitSmem) : 0;
    if (rows)  // per call: the attribute belongs to the current device's context
        NFSP_CUDA(cudaFuncSetAttribute(n_runs == 1 ? (const void *)single : (const void *)batch,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (n_runs == 1) single<<<4, threads, smem, st>>>(R.S, R.run[0]);
    else batch<<<4 * n_runs, threads, smem, st>>>(R);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

extern "C" int nfsp_learner_fit(const nfsp_learner_io *io, int minibatch, int fit_batch, int epochs, const float lr[4],
                                float *d_weights_out, void *stream) {
    return learner_fit(io, 1, minibatch, fit_batch, epochs, lr, &d_weights_out, nullptr, (cudaStream_t)stream);
}

extern "C" int nfsp_learner_fit_peers(const nfsp_learner_io *io, int minibatch, int fit_batch, int epochs, const float lr[4],
                                      float *d_weights_out, const nfsp_peers *peers, void *stream) {
    NFSP_CHECK_ARG(peers && peers->world >= 2 && peers->world <= NFSP_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world,
                   "2..%d peers", NFSP_MAX_PEERS);
    NFSP_CHECK_ARG(peers->d_err, "null error word");
    for (int r = 0; r < peers->world; ++r) NFSP_CHECK_ARG(peers->d_buf[r], "null exchange buffer of rank %d", r);
    NFSP_CHECK_ARG(minibatch <= NFSP_FIT_ROWS_MAX_MINIBATCH && fit_batch <= NFSP_FIT_ROWS_MAX_STEP,
                   "the peer exchange lives in the row-parallel kernel: minibatch <= %d, fit_batch <= %d",
                   NFSP_FIT_ROWS_MAX_MINIBATCH, NFSP_FIT_ROWS_MAX_STEP);
    return learner_fit(io, 1, minibatch, fit_batch, epochs, lr, &d_weights_out, peers, (cudaStream_t)stream);
}

extern "C" int nfsp_learner_fit_runs(const nfsp_learner_io *io, int n_runs, int minibatch, int fit_batch, int epochs, const float *lr,
                                     float *const *d_weights_out, void *stream) {
    NFSP_CHECK_ARG(n_runs >= 1 && n_runs <= NFSP_MAX_RUNS, "n_runs must be in [1, %d]", NFSP_MAX_RUNS);
    return learner_fit(io, n_runs, minibatch, fit_batch, epochs, lr, d_weights_out, nullptr, (cudaStream_t)stream);
}

extern "C" int nfsp_sgd_apply(float *d_weights, const float *d_grad, const float lr[4], float scale, void *stream) {
    NFSP_CHECK_ARG(d_weights && d_grad && lr, "null argument");
    sgd_apply_kernel<<<(kGradFloats + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_weights, d_grad, lr[0], lr[1], lr[2],
                                                                                  lr[3], scale);
    NFSP_LAUNCH_CHECK();
    return NFSP_OK;
}

// ---- exchange buffers without torch's symmetric memory: plain CUDA IPC ---------------------------------------------
// A rank allocates its buffer with cudaMalloc (zeroed), hands the 64-byte IPC handle to its peers through any channel
// (the host code uses torch.distributed.all_gather_object), and maps theirs.  No multicast mapping on this route.
extern "C" int nfsp_peer_buffer_create(int device, void **d_buf, unsigned char *handle64) {
    NFSP_CHECK_ARG(d_buf && handle64, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", device);
    void *p = nullptr;
    NFSP_CUDA(cudaMalloc(&p, sizeof(float) * NFSP_PEER_BUF_FLOATS));
    NFSP_CUDA(cudaMemset(p, 0, sizeof(float) * NFSP_PEER_BUF_FLOATS));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return set_error(NFSP_E_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    }
    memcpy(handle64, &h, 64);
    *d_buf = p;
    return NFSP_OK;
}

extern "C" int nfsp_peer_buffer_open(int device, const unsigned char *handle64, void **d_buf) {
    NFSP_CHECK_ARG(d_buf && handle64, "null argument");
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    NFSP_CUDA(cudaIpcOpenMemHandle(d_buf, h, cudaIpcMemLazyEnablePeerAccess));
    return NFSP_OK;
}

extern "C" int nfsp_peer_buffer_close(int device, void *d_buf) {
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", device);
    if (d_buf) NFSP_CUDA(cudaIpcCloseMemHandle(d_buf));
    return NFSP_OK;
}

extern "C" int nfsp_peer_buffer_destroy(int device, void *d_buf) {
    DeviceGuard guard(device);
    if (!guard.ok) return set_error(NFSP_E_CUDA, "cannot select device %d", device);
    if (d_buf) NFSP_CUDA(cudaFree(d_buf));
    return NFSP_OK;
}
