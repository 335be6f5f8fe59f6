// ENV_NFSP as a finite-state machine: the representation of the env-only step kernel (K1, nfsp_step_fsm_kernel).
//
// ncu on the register formulation of nfsp_fast.cuh showed K1 bound by the integer ALU pipe (126 of 201
// instructions per transition are LOP3 / SEL / SHF / ISETP, which issue at half rate; load/store pipe idle).
// Here everything newenv.Env.step decides from (dealer, betting sequence, raw action) -- coercions, chips, the
// history bit, who acts next, round / hand over, the static part of the trace record -- is ONE table entry of eight
// words laid out so that each word is used as it is loaded (two LDS.128, no shifts or field extraction):
//
//   row    = (dealer d, sigma): sigma = 9*round + sequence id of the round (nfsp_fast.cuh); the player to act follows
//            from the row (main.py:55-65: the dealer opens both rounds, players alternate), q = d ^ (actions & 1)
//   entry  = row x raw action (np.argmax of the action vector), 32 bytes:
//     hc   history bit of this action (obs bit 12q + 2t + a - 1; none for a fold) | card mask of the round after the
//          step (bits 24-29) | hand over << 30 | q << 31
//     pa   what the actor's word gains: chips (twice, see the P word) | raw << 13 | 1 << 15 | t << 16
//     pm   all ones iff the turn passes to the other player
//     nx   shared-memory address of the next row (a terminal pseudo-row when the hand is over)
//     mw   trace word 3, per-step part: raw | effective action << 2 | round << 4 | round << 12
//     mb   trace word 3, accumulating part: chips << (13 + 4q)
//     ma, mo  masks that turn (PA, PO) into the byte offset of the actor's reward in the reward table:
//          fold: PA's chips; showdown: PA's showdown result and PO's chips (second copy); else 0 -> reward 0
//   row[3] = info word read when the game is packed: tt | q << 4 | kind << 8 | hand over << 16
//
// A re-deal (newenv.py:76-114 + main.py:28-45) is one LDS.128 from the deal table of the new dealer (both players'
// words in acting order and the static part of trace word 3) and one from a 4-entry table of the policy draws.
// Semantics are those of NfspW::step (nfsp_rules.cuh); parity tests run seeded rollouts through the general kernel,
// this one and the CPU restatement.
#pragma once
#include <cstdint>

#include "nfsp_rules.cuh"

namespace nfsp {
namespace fsm {

// per-player word P
//   2-5  chips in half chips (byte offset of a fold's reward)     6-7 showdown result if this player closes it:
//   0 draw, 1 wins, 2 loses      8-11 chips again (reward-table offset of the opponent's chips)      12 policy ('b' = 1)
//   13-14 last raw action     15 acted with a non-zero vector     16-18 time of the last step() call (7 = never)
//   19-20 card rank   21-22 public card rank   24-26 one-hot private card   27-29 private | public one-hot
constexpr uint32_t kPClear = 0x7E000u;  // last raw action, non-zero flag, time of the last step
constexpr uint32_t kCm0 = 0x07000000u, kCm1 = 0x3F000000u;
constexpr uint32_t kHxOver = 1u << 30;

enum : uint32_t { KIND_PASS = 0, KIND_ROUND = 1, KIND_SHOWDOWN = 2, KIND_FOLD = 3 };

// image layout, byte offsets (all 16-byte aligned)
constexpr int kLiveRows = 36, kTermRows = 16, kRows = kLiveRows + kTermRows;
// a row is 3 entries + the info word = 112 bytes = 7 bank groups of 16 bytes: 7 is coprime with the 8 bank groups an
// LDS.128 quarter-warp spans, so different rows with the same action do not collide (they did with 128-byte rows)
constexpr int kRowBytes = 112, kEntryBytes = 32, kInfoOff = 96;
constexpr int kFsmOff = 0;
constexpr int kDealOff = kFsmOff + kRows * kRowBytes;           // 5824
constexpr int kDealEntries = 120, kPolOff = kDealEntries * 16;  // the 4 policy entries follow a dealer's 120 deals
constexpr int kDealHalf = kPolOff + 4 * 16;                     // 1984
constexpr int kRewardOff = kDealOff + 2 * kDealHalf;            // 9792
constexpr int kRewardWords = 1024;
constexpr int kImageBytes = kRewardOff + 4 * kRewardWords;      // 13888
constexpr int kImageWords = kImageBytes / 4;

__host__ __device__ inline uint32_t seq_actions(uint32_t s) { return s == 0u ? 0u : (s < 3u ? 1u : 2u); }
__host__ __device__ inline uint32_t term_row(uint32_t kind, uint32_t tt, uint32_t q) {
    return (uint32_t)kLiveRows + (kind == KIND_FOLD ? 2u * tt + q : 12u + 2u * (tt - 5u) + q);
}
// ordered draw of 3 of 6 cards, deck.py:35-50 (same arithmetic as deal_ranks in philox.cuh, host-callable)
__host__ __device__ inline uint32_t deal_ranks_h(uint32_t idx) {
    const uint32_t i0 = idx / 20u, r = idx - i0 * 20u;
    const uint32_t j1 = r >> 2, j2 = r & 3u;
    const uint32_t i1 = j1 + (j1 >= i0 ? 1u : 0u);
    const uint32_t lo = i0 < i1 ? i0 : i1, hi = i0 < i1 ? i1 : i0;
    uint32_t i2 = j2;
    i2 += (i2 >= lo) ? 1u : 0u;
    i2 += (i2 >= hi) ? 1u : 0u;
    return (i0 >> 1) | ((i1 >> 1) << 2) | ((i2 >> 1) << 4);
}
// newenv.py:261-298 seen from player p as the one who closes the showdown: 0 draw, 1 wins, 2 loses.  The actor
// pairing the board is tested first, so with c0 == c1 == pub (set_hands accepts it) whoever closes wins.
__host__ __device__ inline uint32_t showdown_result(uint32_t p, uint32_t c0, uint32_t c1, uint32_t pub) {
    const uint32_t cp = p ? c1 : c0, co = p ? c0 : c1;
    if (cp == pub) return 1u;
    if (co == pub) return 2u;
    return cp < co ? 1u : (cp > co ? 2u : 0u);
}
__host__ __device__ inline uint32_t p_word(uint32_t p, uint32_t c0, uint32_t c1, uint32_t pub, uint32_t chips, uint32_t pol,
                                           uint32_t last, uint32_t nz, uint32_t tsnap) {
    const uint32_t c = p ? c1 : c0, row0 = 1u << c;
    return (chips << 2) | (showdown_result(p, c0, c1, pub) << 6) | (chips << 8) | (pol << 12) | (last << 13) | (nz << 15) |
           (tsnap << 16) | (c << 19) | (pub << 21) | (row0 << 24) | ((row0 | (1u << pub)) << 27);
}

// The whole image; addresses (nx, the first row of a hand) are byte offsets into it -- a CTA adds the shared-memory
// address of its copy (is_address() says which words).
// newenv.Env.step from (dealer, sigma, raw action): what both images (K1's and the rollout's) are built from
struct Move {
    uint32_t s, r, t, q, av, kind, add, hbit, tt_new, sigma_new;
    uint32_t fin0;  // the round-0 sequence a step into round 1 finishes (0 otherwise)
    bool term, pass;
};
inline Move move_of(uint32_t d, uint32_t sigma, uint32_t raw) {
    Move m;
    m.r = sigma >= 9u ? 1u : 0u;
    m.s = sigma - 9u * m.r;
    const uint32_t k = seq_actions(m.s);
    m.t = 3u * m.r + k;
    m.q = d ^ (k & 1u);
    m.av = raw;
    if (m.av == A_RAISE && m.s >= 3u) m.av = A_CALL;  // newenv.py:141-145: s in {4,6} are the two coercion cases
    m.add = 0u;
    m.hbit = 0u;
    m.tt_new = m.t;
    m.sigma_new = sigma;
    m.fin0 = 0u;
    if (m.av == A_FOLD) {
        m.kind = KIND_FOLD;
    } else {
        const uint32_t s = m.s, t = m.t;
        const bool prev_raise = s != 0u && !(s & 1u);                                        // s in {2,4,6}
        m.add = (m.av == A_RAISE ? 2u : 0u) + (prev_raise ? 2u : 0u) + (t == 0u ? 1u : 0u);  // newenv.py:157-176
        m.hbit = 1u << (12u * m.q + 2u * t + m.av - 1u);
        const uint32_t sn = s < 3u ? 2u * s + m.av : 5u + (s >> 1);
        const bool over = s >= 3u || (s != 0u && m.av == A_CALL);                             // newenv.py:180-190
        if (!over) { m.kind = KIND_PASS; m.tt_new = t + 1u; m.sigma_new = 9u * m.r + sn; }
        else if (m.r == 0u) { m.kind = KIND_ROUND; m.tt_new = 3u; m.sigma_new = 9u; }         // newenv.py:215-242
        else { m.kind = KIND_SHOWDOWN; m.tt_new = t + 1u; }                                   // newenv.py:261-298
        if (m.kind == KIND_ROUND) m.fin0 = (sn >> 1) - 1u;  // 0 CC, 1 RC, 2 CRC, 3 RRC
    }
    m.term = m.kind >= KIND_SHOWDOWN;
    m.pass = !m.term && (m.kind == KIND_PASS || m.q != d);  // round 1 opens with the dealer
    return m;
}

// The whole image; addresses (nx, the first row of a hand) are byte offsets into it -- a CTA adds the shared-memory
// address of its copy (is_address() says which words).
inline void build_image(uint32_t *img) {
    for (int i = 0; i < kImageWords; ++i) img[i] = 0u;
    for (uint32_t d = 0; d < 2; ++d)
        for (uint32_t sigma = 0; sigma < 18; ++sigma) {
            uint32_t *row = img + (kFsmOff + (int)(d * 18u + sigma) * kRowBytes) / 4;
            if (sigma % 9u >= 7u) continue;  // [C,R,C] / [R,R,C] end the round: never a state to act in
            const Move m0 = move_of(d, sigma, 0u);
            row[kInfoOff / 4] = m0.t | (m0.q << 4);
            for (uint32_t raw = 0; raw < 3; ++raw) {
                const Move m = move_of(d, sigma, raw);
                uint32_t *e = row + raw * (kEntryBytes / 4);
                const uint32_t r_new = m.tt_new >= 3u ? 1u : 0u;
                e[0] = m.hbit | ((m.r == 1u || m.kind == KIND_ROUND) ? kCm1 : kCm0) | ((uint32_t)m.term << 30) | (m.q << 31);
                e[1] = (m.add << 2) | (m.add << 8) | (raw << 13) | (1u << 15) | (m.t << 16);
                e[2] = m.pass ? 0xFFFFFFFFu : 0u;
                e[3] = (uint32_t)(kFsmOff + (int)(m.term ? term_row(m.kind, m.tt_new, m.q) : d * 18u + m.sigma_new) * kRowBytes);
                e[4] = raw | (m.av << 2) | (r_new << 4) | (r_new << 12);
                e[5] = m.add << (13u + 4u * m.q);
                e[6] = m.kind == KIND_FOLD ? 0x3Cu : (m.kind == KIND_SHOWDOWN ? 0xC0u : 0u);
                e[7] = m.kind == KIND_SHOWDOWN ? 0xF00u : 0u;
            }
        }
    for (uint32_t kind = KIND_SHOWDOWN; kind <= KIND_FOLD; ++kind)
        for (uint32_t tt = (kind == KIND_FOLD ? 0u : 5u); tt <= (kind == KIND_FOLD ? 5u : 6u); ++tt)
            for (uint32_t q = 0; q < 2; ++q)
                img[(kFsmOff + (int)term_row(kind, tt, q) * kRowBytes + kInfoOff) / 4] = tt | (q << 4) | (kind << 8) | (1u << 16);
    for (uint32_t d = 0; d < 2; ++d) {
        uint32_t *half = img + (kDealOff + (int)d * kDealHalf) / 4;
        for (uint32_t idx = 0; idx < (uint32_t)kDealEntries; ++idx) {
            const uint32_t c = deal_ranks_h(idx), c0 = c & 3u, c1 = (c >> 2) & 3u, pub = (c >> 4) & 3u;
            const uint32_t b0 = d == 0u ? 1u : 2u, b1 = d == 0u ? 2u : 1u;  // small blind 0.5 / big blind 1.0 (newenv.py:80-82)
            const uint32_t P0 = p_word(0, c0, c1, pub, b0, 0, 0, 0, 7), P1 = p_word(1, c0, c1, pub, b1, 0, 0, 0, 7);
            half[4 * idx + 0] = d ? P1 : P0;  // the dealer opens: it is the player to act
            half[4 * idx + 1] = d ? P0 : P1;
            half[4 * idx + 2] = (d << 5) | (c0 << 6) | (c1 << 8) | (pub << 10) | (b0 << 13) | (b1 << 17);
        }
        for (uint32_t pw = 0; pw < 4; ++pw) {  // pw = policy of player 0 | policy of player 1 << 1 (main.py:38-45)
            uint32_t *e = half + kPolOff / 4 + 4 * pw;
            const uint32_t pol0 = pw & 1u, pol1 = pw >> 1;
            e[0] = (d ? pol1 : pol0) << 12;
            e[1] = (d ? pol0 : pol1) << 12;
            e[2] = (pol0 << 22) | (pol1 << 23);
            e[3] = (uint32_t)(kFsmOff + (int)(d * 18u) * kRowBytes);
        }
    }
    float *rew = reinterpret_cast<float *>(img + kRewardOff / 4);
    for (int i = 0; i < kRewardWords; ++i) {  // word index = fold chips | showdown result << 4 | opponent chips << 6
        const int low = i & 15, sd = (i >> 4) & 3, bo = i >> 6;
        int half_chips = 0;
        if (bo == 0 && sd == 0) half_chips = -low;                   // fold: newenv.py:252-255
        else half_chips = sd == 1 ? bo : (sd == 2 ? -bo : 0);        // showdown won / lost / drawn
        rew[i] = 0.5f * (float)half_chips;
    }
}
// word w of the image holds a byte offset that becomes a shared-memory address
__host__ __device__ inline bool is_address(int w) {
    if (w < kDealOff / 4) return (w % (kRowBytes / 4)) < 24 && ((w % (kRowBytes / 4)) & 7) == 3;
    if (w >= kRewardOff / 4) return false;
    const int v = (w - kDealOff / 4) % (kDealHalf / 4);
    return v >= kPolOff / 4 && (v & 3) == 3;
}

// ---- the fused rollout's image (rollout_states_kernel) ---------------------------------------------------------------
// The same rows (dealer, sigma) and entries (row, raw action), every word used as loaded, with what a decision of the
// rollout needs beside the game step (32 bytes an entry):
//   hc, pm, nx  as above
//   pa     as above without the non-zero flag: the decision sets it (bit 15 of the state table's fourth word)
//   ds     change of the state-table offset 16 * (fin0 * 18 + sigma), fin0 = the finished round-0 sequence (round 1)
//   mx     raw | effective action << 2 | round after the step << 4 | 1 << 8 | the same round << 12 | q << 16: & 0x10103 is
//          the last word of the actor's terminal RL record, & 0x101F the per-step part of trace word 3
//   rm     mask of (PA & 0xFF) | (PO & 0xF00) giving the reward word's byte offset: fold 0x3C, showdown 0xFFC, else 0
//   inc    1 << 5 * (3q + raw): the step's count in the action histogram
// Terminal pseudo-rows keep only their info word, 16 bytes apart (a row address is its info word's minus kInfoOff).
// A deal entry holds both players' P words (bit 23 set in player 1's) and both state-table offsets without the policy,
// 16 * (2 * player * 1296 + card * 432 + pub * 144 + dealer * 72); a policy entry the policy bits and 16 * 1296 * policy
// per player.  A dealer's deal table is as long as its rows, so its first row is at dl - kRDealOff.  Reward word: index
// fold chips | showdown result << 4 | opponent chips << 6, the actor's half chips in byte 0 and the other player's in
// byte 1 (int8).
// Addresses are byte offsets from the state table, which the image follows `at` bytes later in shared memory.
constexpr uint32_t kPPlayer = 1u << 23;  // rollout P words: this is player 1
constexpr int kNetSlots = 72 * 18;       // state-table slots per net (rollout_states.cu)
constexpr int kRTermOff = kLiveRows * kRowBytes;                // 4032
constexpr int kRDealOff = kRTermOff + kTermRows * 16;           // 4288
constexpr int kRDealHalf = 18 * kRowBytes;                      // 2016
constexpr int kRRewardOff = kRDealOff + 2 * kRDealHalf;         // 8320
constexpr int kRImageBytes = kRRewardOff + 4 * kRewardWords;    // 12416
constexpr int kRImageWords = kRImageBytes / 4;
static_assert(kPolOff + 4 * 16 <= kRDealHalf, "a dealer's deal and policy entries fit beside its rows' stride");

__host__ __device__ inline uint32_t state_offset(uint32_t net, uint32_t card, uint32_t pub, uint32_t dealer, uint32_t fin0,
                                                 uint32_t sigma) {
    return 16u * (net * (uint32_t)kNetSlots + ((((card * 3u + pub) * 2u + dealer) * 4u + fin0) * 18u + sigma));
}

inline void build_rollout_image(uint32_t *img, uint32_t at) {
    for (int i = 0; i < kRImageWords; ++i) img[i] = 0u;
    for (uint32_t d = 0; d < 2; ++d)
        for (uint32_t sigma = 0; sigma < 18; ++sigma) {
            uint32_t *row = img + (int)(d * 18u + sigma) * kRowBytes / 4;
            if (sigma % 9u >= 7u) continue;
            const Move m0 = move_of(d, sigma, 0u);
            row[kInfoOff / 4] = m0.t | (m0.q << 4);
            for (uint32_t raw = 0; raw < 3; ++raw) {
                const Move m = move_of(d, sigma, raw);
                uint32_t *e = row + raw * (kEntryBytes / 4);
                const uint32_t r_new = m.tt_new >= 3u ? 1u : 0u;
                const uint32_t g_new = m.term ? sigma : m.fin0 * 18u + m.sigma_new;  // fin0 is 0 until round 1 starts
                e[0] = m.hbit | ((m.r == 1u || m.kind == KIND_ROUND) ? kCm1 : kCm0) | ((uint32_t)m.term << 30) | (m.q << 31);
                e[1] = (m.add << 2) | (m.add << 8) | (raw << 13) | (m.t << 16);
                e[2] = m.pass ? 0xFFFFFFFFu : 0u;
                e[3] = at + (m.term ? (uint32_t)(kRTermOff + 16 * ((int)term_row(m.kind, m.tt_new, m.q) - kLiveRows) - kInfoOff)
                                    : (d * 18u + m.sigma_new) * (uint32_t)kRowBytes);
                e[4] = 16u * (g_new - sigma);  // within round 1 fin0 does not change
                e[5] = raw | (m.av << 2) | (r_new << 4) | (1u << 8) | (r_new << 12) | (m.q << 16);
                e[6] = m.kind == KIND_FOLD ? 0x3Cu : (m.kind == KIND_SHOWDOWN ? 0xFFCu : 0u);
                e[7] = 1u << (5u * (3u * m.q + raw));
            }
        }
    for (uint32_t kind = KIND_SHOWDOWN; kind <= KIND_FOLD; ++kind)
        for (uint32_t tt = (kind == KIND_FOLD ? 0u : 5u); tt <= (kind == KIND_FOLD ? 5u : 6u); ++tt)
            for (uint32_t q = 0; q < 2; ++q)
                img[(kRTermOff + 16 * ((int)term_row(kind, tt, q) - kLiveRows)) / 4] = tt | (q << 4) | (kind << 8) | (1u << 16);
    for (uint32_t d = 0; d < 2; ++d) {
        uint32_t *half = img + (kRDealOff + (int)d * kRDealHalf) / 4;
        for (uint32_t idx = 0; idx < (uint32_t)kDealEntries; ++idx) {
            const uint32_t c = deal_ranks_h(idx), c0 = c & 3u, c1 = (c >> 2) & 3u, pub = (c >> 4) & 3u;
            const uint32_t b0 = d == 0u ? 1u : 2u, b1 = d == 0u ? 2u : 1u;
            const uint32_t P0 = p_word(0, c0, c1, pub, b0, 0, 0, 0, 7), P1 = p_word(1, c0, c1, pub, b1, 0, 0, 0, 7) | kPPlayer;
            half[4 * idx + 0] = d ? P1 : P0;
            half[4 * idx + 1] = d ? P0 : P1;
            half[4 * idx + 2] = state_offset(2u * d, d ? c1 : c0, pub, d, 0u, 0u);
            half[4 * idx + 3] = state_offset(2u * (d ^ 1u), d ? c0 : c1, pub, d, 0u, 0u);
        }
        for (uint32_t pw = 0; pw < 4; ++pw) {
            uint32_t *e = half + kPolOff / 4 + 4 * pw;
            const uint32_t pol0 = pw & 1u, pol1 = pw >> 1, pa = d ? pol1 : pol0, po = d ? pol0 : pol1;
            e[0] = pa << 12;
            e[1] = po << 12;
            e[2] = pa * 16u * (uint32_t)kNetSlots;
            e[3] = po * 16u * (uint32_t)kNetSlots;
        }
    }
    uint32_t *rew = img + kRRewardOff / 4;
    for (int i = 0; i < kRewardWords; ++i) {
        const int ba = i & 15, sd = (i >> 4) & 3, bo = i >> 6;
        int ra = 0, ro = 0;
        if (bo == 0 && sd == 0) { ra = -ba; ro = ba; }      // fold: newenv.py:252-255
        else if (sd == 1) { ra = bo; ro = -ba; }            // showdown won by the actor
        else if (sd == 2) { ra = -bo; ro = ba; }            // lost; drawn: 0
        rew[i] = (uint32_t)(uint8_t)(int8_t)ra | (uint32_t)(uint8_t)(int8_t)ro << 8;
    }
}
// word w of the rollout image holds an offset that becomes a shared-memory address
__host__ __device__ inline bool is_rollout_address(int w) {
    if (w < kRTermOff / 4) return (w % (kRowBytes / 4)) < 24 && ((w % (kRowBytes / 4)) & 7) == 3;
    if (w < kRDealOff / 4 || w >= kRRewardOff / 4) return false;
    const int v = (w - kRDealOff / 4) % (kRDealHalf / 4);
    return v < kPolOff / 4 && (v & 3) >= 2;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
// One game in registers for the steps of a launch; kDeal / kHalf: where the image keeps the deal tables.
template <int kDeal, int kHalf>
struct GameAt {
    uint32_t HX;   // history (0-23) | card mask of the round (24-29) | hand over (30) | actor of the last step (31)
    uint32_t PA, PO;  // words of the player to act / the other one; swap when the turn passes
    uint32_t ms;   // trace word 3: dealer, cards, policies, both players' chips
    uint32_t tix;  // shared-memory address of the row
    uint32_t dl;   // shared-memory address of the dealer's deal table

    __device__ __forceinline__ void unpack(uint64_t w, uint32_t base) {
        const NfspW g{w};
        const uint32_t H = g.hist(), both = H | (H >> 12);
        const uint32_t r = g.round(), d = g.dealer(), q = (uint32_t)g.to_act();
        const uint32_t rnd = (both >> (6u * r)) & 63u, s0 = rnd & 3u, s1 = (rnd >> 2) & 3u, s2 = (rnd >> 4) & 3u;
        const uint32_t seq = s2 ? 6u + s0 : (s1 ? 2u * s0 + s1 : s0);
        // a hand that is over (also one finished without the re-deal flag) is re-dealt at the first step
        const bool over = g.need_reset() || g.terminated();
        HX = H | (r ? kCm1 : kCm0) | (over ? kHxOver : 0u);
        const uint32_t c0 = g.card(0), c1 = g.card(1), pub = g.pub();
        const uint32_t P0 = p_word(0, c0, c1, pub, g.bets(0), g.policy(0), g.last_a(0), g.acted_nz(0), g.t_snap(0));
        const uint32_t P1 = p_word(1, c0, c1, pub, g.bets(1), g.policy(1), g.last_a(1), g.acted_nz(1), g.t_snap(1));
        PA = q ? P1 : P0;
        PO = q ? P0 : P1;
        ms = (d << 5) | (c0 << 6) | (c1 << 8) | (pub << 10) | (g.bets(0) << 13) | (g.bets(1) << 17) | (g.policy(0) << 22) |
             (g.policy(1) << 23);
        tix = base + (uint32_t)kFsmOff + (d * 18u + (over ? 0u : 9u * r + seq)) * (uint32_t)kRowBytes;
        dl = base + (uint32_t)kDeal + d * (uint32_t)kHalf;
    }

    __device__ __forceinline__ uint64_t pack(uint32_t base) const {
        const uint32_t info = lds32(tix + (uint32_t)kInfoOff);
        const uint32_t tt = info & 7u, q = (info >> 4) & 1u, kind = (info >> 8) & 3u, over = (info >> 16) & 1u;
        const uint32_t d = dl != base + (uint32_t)kDeal ? 1u : 0u;
        const uint32_t P0 = q ? PO : PA, P1 = q ? PA : PO;
        const uint32_t r = tt >= 3u ? 1u : 0u, k = tt - 3u * r;
        const uint32_t sd = (PA >> 6) & 3u;  // PA is the actor of the terminating step
        const uint32_t oc = (over && kind == KIND_SHOWDOWN) ? (sd == 0u ? 3u : sd) : 0u;
        const uint32_t lo = (HX & 0xFFFFFFu) | (((P0 >> 19) & 3u) << 24) | (((P1 >> 19) & 3u) << 26) | (((P0 >> 21) & 3u) << 28) |
                            (d << 30) | (r << 31);
        const uint32_t hi = k | (((P0 >> 2) & 15u) << 2) | (((P1 >> 2) & 15u) << 6) | (over << 10) | (over << 11) |
                            (((P0 >> 12) & 1u) << 12) | (((P1 >> 12) & 1u) << 13) | (((P0 >> 13) & 3u) << 14) |
                            (((P1 >> 13) & 3u) << 16) | (((P0 >> 15) & 1u) << 18) | (((P1 >> 15) & 1u) << 19) |
                            (((P0 >> 16) & 7u) << 20) | (((P1 >> 16) & 7u) << 23) | ((over ? q : 0u) << 26) | (oc << 27);
        return (uint64_t)lo | ((uint64_t)hi << 32);
    }
};
using Game = GameAt<kDealOff, kDealHalf>;

// The rollout's game: the snapshots s[p] (newenv.py:200-202) and the players' state-table addresses at the current row
// (FA + 16 * slot of this row's (fin0, sigma) is added as the game moves: entry word ds) beside the words of Game; all
// per-player registers swap with the turn.  ibase / sbase: shared-memory addresses of the image / the state table.
struct RolloutGame : GameAt<kRDealOff, kRDealHalf> {
    uint32_t SA, SO, FA, FO;

    __device__ __forceinline__ void unpack(uint64_t w, uint32_t ibase, uint32_t sbase) {
        GameAt<kRDealOff, kRDealHalf>::unpack(w, ibase);
        const NfspW g{w};
        const uint32_t H = g.hist(), both = H | (H >> 12), r = g.round(), d = g.dealer(), q = (uint32_t)g.to_act();
        const auto seq = [](uint32_t rnd) {
            const uint32_t s0 = rnd & 3u, s1 = (rnd >> 2) & 3u, s2 = (rnd >> 4) & 3u;
            return s2 ? 6u + s0 : (s1 ? 2u * s0 + s1 : s0);
        };
        const uint32_t fin0 = r ? (seq(both & 63u) >> 1) - 1u : 0u, sigma = r ? 9u + seq((both >> 6) & 63u) : seq(both & 63u);
        PA |= q ? kPPlayer : 0u;
        PO |= q ? 0u : kPPlayer;
        FA = sbase + state_offset(2u * q + g.policy((int)q), g.card((int)q), g.pub(), d, fin0, sigma);
        FO = sbase + state_offset(2u * (q ^ 1u) + g.policy((int)(q ^ 1u)), g.card((int)(q ^ 1u)), g.pub(), d, fin0, sigma);
        SA = g.snapshot((int)q);
        SO = g.snapshot((int)(q ^ 1u));
    }
};
#endif  // __CUDACC__

}  // namespace fsm
}  // namespace nfsp
