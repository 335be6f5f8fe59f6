// Arguments and counters shared by the two variants of the fused rollout kernel (CUDA-core first layer in
// act_kernels.cu, tcgen05 first layer in act_tc_kernels.cu).  The decision logic itself -- everything of
// Agent.play (agent.py:130-156) and of main.train's inner loop (main.py:28-67) except the network forward --
// is in rollout_fast.cuh.
#pragma once
#include "common.cuh"
#include "nfsp_rules.cuh"
#include "philox.cuh"

namespace nfsp { struct RolloutArgs; }
// launches the tcgen05 variant of the fused rollout (act_tc_kernels.cu)
int nfsp_rollout_tc_launch(nfsp_env_t h, const nfsp::RolloutArgs &A, bool debug, cudaStream_t st);
// launches the warp-specialised tcgen05 rollout (rollout_tq.cu)
int nfsp_rollout_tq_launch(nfsp_env_t h, const nfsp::RolloutArgs &A, bool debug, int reserve_sms, cudaStream_t st);

// launches the net-sorted CUDA-core rollout (rollout_sorted.cu); sets its kernels' shared-memory attribute once per device
int nfsp_rollout_sorted_launch(nfsp_env_t h, const nfsp::RolloutArgs &A, const nfsp_rollout_io *io, bool debug, cudaStream_t st);
// validates nfsp_rollout_io.d_ring* and fills the direct-ring fields of A; *direct = the call appends directly
int nfsp_rollout_direct_args(const nfsp_rollout_io *io, nfsp::RolloutArgs &A, bool *direct);
int nfsp_rollout_sorted_configure();
// launches the two-games-per-lane CUDA-core rollout (rollout_pairs.cu)
int nfsp_rollout_pairs_launch(nfsp_env_t h, const nfsp::RolloutArgs &A, const nfsp_rollout_io *io, bool debug, cudaStream_t st);
int nfsp_rollout_pairs_configure();

// the rollout over a table of the nets' outputs per decision state (rollout_states.cu)
int nfsp_rollout_states_launch(nfsp_env_t h, const nfsp::RolloutArgs &A, const nfsp_rollout_io *io, bool debug, cudaStream_t st);
// rebuilds the state tables of n handles (1 <= n <= NFSP_MAX_RUNS) from their table images tab[r] in one launch and clears
// their st_dirty
int nfsp_states_pack(const nfsp_env_t *h, const float *const *tab, int n, cudaStream_t st);
int nfsp_states_floats();
int nfsp_states_upload_image(float *d_states);
int nfsp_rollout_states_configure();
// independent runs of one shape in one launch of the same rollout (nfsp_rollout_runs); A[r].pack = handle r's state table
int nfsp_rollout_states_runs_launch(nfsp_env_t h, const nfsp::RolloutArgs *A, int n_runs, int sms, cudaStream_t st);

namespace nfsp {

// ---- warp-aggregated record append -------------------------------------------------------------
// The staging arrays are split into n_seg segments (a power of two), each with its own ticket counter; a
// warp's 32 consecutive games always append to segment (first game / 32) % n_seg, so which records land
// in which segment does not depend on the launch geometry, and counters are not shared across the chip.
// Per step a warp claims its slots in the four arrays (RL and SL of both players) with FOUR atomics issued
// by four lanes at once: one global round trip.
struct RolloutArgs {
    uint64_t *state;
    int64_t n;
    uint64_t seed, game0, step0;
    PhiloxKeys keys;         // round keys of `seed` (constant-bank operands of the lean kernels)
    int n_steps;
    uint32_t eta_u32, eps_u32, eps1_u32;  // epsilon of player 0 / of player 1 (each agent decays its own, agent.py:253)
    const void *pack;  // weight image of the variant
    uint4 *rl[2];
    uint4 *sl[2];
    int64_t cap_rl, cap_sl;  // per segment
    uint32_t n_seg;          // power of two
    uint32_t *counts;        // [4][n_seg]: rl0, rl1, sl0, sl1
    uint32_t *work;          // next block of 32 games to hand out (zeroed before the launch)
    unsigned long long *stats;
    uint32_t *trace;
    float *vec;
    const float *forced;
    // direct ring append (nfsp_rollout_io.d_ring*): the RL records go straight into the players' rings
    uint4 *ring[2];
    unsigned long long *ring_total[2];  // records ever inserted = the ticket counter
    uint32_t ring_cap;
    uint64_t ring_magic;                // floor((2^64 - 1) / ring_cap): ticket % ring_cap without a division
};

// ticket % cap for a ring (replay_buffer.py:36-41: slot of the ticket-th record ever added)
__device__ __forceinline__ uint32_t ring_slot(unsigned long long ticket, uint32_t cap, uint64_t magic) {
    const unsigned long long q = __umul64hi(ticket, magic);  // floor(ticket / cap) or one less
    unsigned long long r = ticket - q * cap;
    if (r >= cap) r -= cap;
    return (uint32_t)r;
}

// per-thread counters; the action histogram packs 3 x 21-bit fields per player (flushed before overflow)
struct Counters {
    unsigned long long act0 = 0ull, act1 = 0ull;
    int rew0 = 0, rew1 = 0, hands = 0, trans = 0, drop = 0;

    // warp shuffle reduction, one shared atomic per warp and counter, then 13 global atomics per CTA;
    // call from every thread of the CTA
    __device__ __forceinline__ void commit(unsigned long long *s_stats, unsigned long long *g_stats) {
        long long v[11] = {(long long)(act0 & 0x1FFFFFull), (long long)((act0 >> 21) & 0x1FFFFFull), (long long)(act0 >> 42),
                           (long long)(act1 & 0x1FFFFFull), (long long)((act1 >> 21) & 0x1FFFFFull), (long long)(act1 >> 42),
                           rew0, rew1, hands, trans, drop};
#pragma unroll
        for (int k = 0; k < 11; ++k) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o);
        }
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
            for (int k = 0; k < 11; ++k)
                if (v[k]) atomicAdd(&s_stats[k < 6 ? k : k + 2], (unsigned long long)v[k]);
        }
        act0 = act1 = 0ull;
        __syncthreads();
        if (threadIdx.x == 6) s_stats[6] = s_stats[0] + s_stats[1] + s_stats[2];  // played = sum of the histogram
        if (threadIdx.x == 7) s_stats[7] = s_stats[3] + s_stats[4] + s_stats[5];
        __syncthreads();
        if (threadIdx.x < 13 && s_stats[threadIdx.x]) atomicAdd(g_stats + threadIdx.x, s_stats[threadIdx.x]);
    }
};

}  // namespace nfsp
