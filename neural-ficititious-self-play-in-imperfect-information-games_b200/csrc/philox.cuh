// Philox4x32-10 counter-based RNG (Salmon et al., SC'11), device side.
// Replaces the reference's global Mersenne-Twister `random` (deck.py:2,42-44; main.py:38-45;
// agent.py:125-128) with a stateless stream keyed by (seed; game id, step, purpose) so that a
// game's randomness does not depend on how games are sharded over GPUs.
#pragma once
#include <cstdint>

namespace nfsp {

struct Philox4 {
    uint32_t x, y, z, w;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += W0;
        k1 += W1;
    }
    return Philox4{c0, c1, c2, c3};
}

// The ten round keys (k0 + r*W0, k1 + r*W1) depend on the seed only: the hot kernels take them precomputed
// as a by-value kernel argument, so each key is a constant-bank operand of the round's XOR instead of an add.
struct PhiloxKeys {
    uint32_t k[20];
};
inline PhiloxKeys philox_keys(uint64_t seed) {
    PhiloxKeys K;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        K.k[2 * r] = k0;
        K.k[2 * r + 1] = k1;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return K;
}
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys &K) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        c0 = hi1 ^ c1 ^ K.k[2 * r];
        c1 = lo1;
        c2 = hi0 ^ c3 ^ K.k[2 * r + 1];
        c3 = lo0;
    }
    return Philox4{c0, c1, c2, c3};
}

// purposes (counter word 3), DESIGN.md "Philox streams":
//   STREAM_STEP   one block per (game, step): .x = uniform action (env-only) / epsilon test (NFSP),
//                 .y = deal index, .z/.w = per-hand policy draws of players 0/1 (used iff the hand is re-dealt
//                 at this step; legacy rules: .x/.y = the two actions, .z = deal index)
//   STREAM_VECTOR the random score vector of agent.py:128, computed only in the (rare) epsilon branch
enum : uint32_t { STREAM_STEP = 0, STREAM_VECTOR = 1, STREAM_RESERVOIR = 2, STREAM_SAMPLE = 3 };

__device__ __forceinline__ Philox4 game_block(uint64_t seed, uint64_t game, uint64_t step, uint32_t stream) {
    return philox4x32_10((uint32_t)game, (uint32_t)step, (uint32_t)(step >> 32), stream, (uint32_t)seed,
                         (uint32_t)(seed >> 32));
}

__device__ __forceinline__ Philox4 game_block(const PhiloxKeys &K, uint64_t game, uint64_t step, uint32_t stream) {
    return philox4x32_10((uint32_t)game, (uint32_t)step, (uint32_t)(step >> 32), stream, K);
}

// Counter (idx, idx >> 32 | call >> 32, call, stream).  No stream uses both high halves: the reservoir stream draws with
// call 0, the sample stream with idx = draw index < 1024.  So the whole 64-bit ticket and the whole 64-bit call key the
// draw, and every draw of a call below 2^32 is the one it always was.
__device__ __forceinline__ uint64_t buffer_u64(uint64_t seed, uint64_t idx, uint64_t call, uint32_t stream) {
    const Philox4 o = philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32) | (uint32_t)(call >> 32), (uint32_t)call, stream,
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    return (uint64_t)o.x | ((uint64_t)o.y << 32);
}

// Uniform ordered draw of 3 distinct cards out of the 6-card deck [r0s0,r0s1,r1s0,r1s1,r2s0,r2s1]
// (deck.py:35-50: shuffle, then pop p0, p1, public).  idx in [0,120).  Returns ranks packed
// c0 | c1<<2 | pub<<4.
__device__ __forceinline__ uint32_t deal_ranks(uint32_t idx) {
    const uint32_t i0 = idx / 20u, r = idx - i0 * 20u;
    const uint32_t j1 = r >> 2, j2 = r & 3u;
    const uint32_t i1 = j1 + (j1 >= i0);
    const uint32_t lo = min(i0, i1), hi = max(i0, i1);
    uint32_t i2 = j2;
    i2 += (i2 >= lo);
    i2 += (i2 >= hi);
    return (i0 >> 1) | ((i1 >> 1) << 2) | ((i2 >> 1) << 4);
}

}  // namespace nfsp
