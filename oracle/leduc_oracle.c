/* CPU oracle -- TEST INFRASTRUCTURE ONLY (see leduc_oracle.h).
 * Every function cites the reference file:line it restates. */
#include "leduc_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ======================= Philox4x32-10 =========================================== */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

static inline uint32_t mulhi32(uint32_t x, uint32_t n) { return (uint32_t)(((uint64_t)x * n) >> 32); }
static inline uint64_t mulhi64(uint64_t x, uint64_t n) { return (uint64_t)(((unsigned __int128)x * n) >> 64); }

/* generation spec (DESIGN.md "Philox streams"): key = seed, counter = (game, step_lo, step_hi, stream) */
static void game_block(uint64_t seed, uint64_t game, uint64_t step, uint32_t stream, uint32_t out[4]) {
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    uint32_t ctr[4] = {(uint32_t)game, (uint32_t)step, (uint32_t)(step >> 32), stream};
    orc_philox4x32_10(ctr, key, out);
}

/* deck.py:35-50: list [r0s0,r0s1,r1s0,r1s1,r2s0,r2s1] shuffled, popped p0,p1,public: a uniform ordered
 * draw of 3 distinct cards out of 6 (120 outcomes).  idx in [0,120) -> ranks. */
static void deal_from_index(uint32_t idx, int ranks[3]) {
    int deck[6] = {0, 1, 2, 3, 4, 5};
    int n = 6;
    int picks[3] = {(int)(idx / 20), (int)((idx % 20) / 4), (int)(idx % 4)};
    for (int i = 0; i < 3; ++i) {
        int j = picks[i];
        ranks[i] = deck[j] / 2;
        for (int k = j; k < n - 1; ++k) deck[k] = deck[k + 1];
        --n;
    }
}

/* ======================= leduc/env.py ============================================= */
static int argmax3(const double a[3]) { /* np.argmax: first maximum */
    int m = 0;
    if (a[1] > a[m]) m = 1;
    if (a[2] > a[m]) m = 2;
    return m;
}
static int argmax3f(const float a[3]) {
    int m = 0;
    if (a[1] > a[m]) m = 1;
    if (a[2] > a[m]) m = 2;
    return m;
}

void orc_legacy_init(OrcLegacyEnv *e) { /* env.py:13-32, config.ini:12,22 */
    memset(e, 0, sizeof(*e));
    e->penalty = -1;
    e->choices = 4;
    e->pub = -1;
}

void orc_legacy_reset(OrcLegacyEnv *e, int c0, int c1) { /* env.py:46-72 */
    e->pub = -1; /* deck.py:33,46-47 fake public card */
    e->pot[0] = e->pot[1] = 0;
    e->left[0] = e->left[1] = e->choices;
    e->card[0] = c0;
    e->card[1] = c1;
    for (int p = 0; p < 2; ++p) {
        e->st_pot[p] = 0;
        e->st_reward[p] = 0;
        e->st_terminal[p] = 0;
        e->st_action[p] = 3;
    }
}

void orc_legacy_step(OrcLegacyEnv *e, const double action[3], int p) { /* env.py:84-158 */
    int o = 1 - p;
    int terminal = 0;
    /* env.py:97-101: reveal block is dead code (fake card rank is -1, never 0) */
    if (e->left[p] > 0) {
        int av = argmax3(action);
        if (av == 0) { /* env.py:114-120 */
            if (e->left[p] == 4 && e->left[o] == 4) e->st_reward[p] = e->penalty;
            terminal = 1;
        }
        if (av == 1) { /* env.py:122-128 */
            e->left[p] -= 1;
            if (e->pot[p] < e->pot[o]) e->pot[p] += 1;
            terminal = (e->left[p] == 0) ? 1 : 0;
        }
        if (av == 2) { /* env.py:130-139 */
            if (e->left[p] % 2 != 0) e->st_reward[p] = e->penalty;
            e->left[p] -= 2;
            if (e->pot[p] <= e->pot[o]) e->pot[p] += 1;
            terminal = (e->left[p] == 0) ? 1 : 0;
        }
    } else {
        terminal = 1; /* env.py:140-141 */
    }
    e->st_terminal[p] = terminal;          /* env.py:145,155 */
    e->st_pot[p] = e->pot[p] + e->pot[o];  /* env.py:148-150 */
    e->st_action[p] = argmax3(action);     /* env.py:152 (vector kept; we keep its argmax) */
}

void orc_legacy_get_new_state(OrcLegacyEnv *e, int p, int out[5]) { /* env.py:160-205 */
    int o = 1 - p;
    e->st_pot[p] = e->pot[p] + e->pot[o];
    e->st_terminal[p] = e->st_terminal[o]; /* env.py:174 */
    if (e->st_terminal[p] == 1) {
        if (e->card[p] == e->pub) e->st_reward[p] += e->pot[o];        /* env.py:179-184 */
        else if (e->card[o] == e->pub) e->st_reward[p] += -e->pot[p];  /* env.py:186-187 */
        else if (e->card[p] > e->card[o]) e->st_reward[p] += -e->pot[p]; /* env.py:189-190 */
        else if (e->card[p] < e->card[o]) e->st_reward[p] += e->pot[o];  /* env.py:192-199 */
        /* else draw: += 0 */
    }
    out[0] = e->card[p];
    out[1] = e->pub;
    out[2] = e->st_pot[p];
    out[3] = e->st_reward[p];
    out[4] = e->st_terminal[p];
}

/* ======================= leduc/newenv.py ========================================== */
void orc_nfsp_reset(OrcNfspEnv *e, int dealer, int c0, int c1, int pub) { /* newenv.py:76-114 */
    int anomalies = e->anomalies;
    memset(e, 0, sizeof(*e));
    e->anomalies = anomalies;
    e->dealer = dealer;
    int n = dealer == 0 ? 1 : 0;
    e->overall_raises[dealer] += 0.5; /* small blind */
    e->overall_raises[n] += 1.0;      /* big blind   */
    e->deck[0] = c0; e->deck[1] = c1; e->deck[2] = pub;
    e->deck_pos = 0;
    for (int k = 0; k < 2; ++k) { /* newenv.py:109-114: player 0 pops first regardless of dealer */
        int card_index = e->deck[e->deck_pos++];
        e->specific_cards[k][e->round][card_index] = 1.0;
    }
}

void orc_nfsp_state_vector(const OrcNfspEnv *e, int p, double out[30]) { /* newenv.py:118 */
    int i = 0;
    for (int q = 0; q < 2; ++q)
        for (int r = 0; r < 2; ++r)
            for (int k = 0; k < 3; ++k)
                for (int b = 0; b < 2; ++b) out[i++] = e->history[q][r][k][b];
    for (int r = 0; r < 2; ++r)
        for (int c = 0; c < 3; ++c) out[i++] = e->specific_cards[p][r][c];
}

uint32_t orc_mask30(const double v[30]) {
    uint32_t m = 0;
    for (int i = 0; i < 30; ++i)
        if (v[i] != 0.0) m |= 1u << i;
    return m;
}

int orc_nfsp_get_state(const OrcNfspEnv *e, int p, double s[30], double a[3], double *r, double s2[30]) {
    /* newenv.py:116-129 */
    if (s) memcpy(s, e->s[p], sizeof(double) * 30);
    if (a) memcpy(a, e->last_action[p], sizeof(double) * 3);
    if (s2) orc_nfsp_state_vector(e, p, s2);
    if (r) *r = e->terminated ? e->reward[p] : 0.0;
    return e->terminated;
}

static int nfsp_do_action(OrcNfspEnv *e, const double action[3], int p) { /* newenv.py:131-178 */
    int av = argmax3(action);
    memcpy(e->last_action[p], action, sizeof(double) * 3);
    if (e->raises[p] > 0 && av == 2) av = 1; /* newenv.py:141-142 */
    if (e->n_done == 2 && e->actions_done[0] == ORC_CALL && e->actions_done[1] == ORC_RAISE && av == 2)
        av = 1; /* newenv.py:143-145 */
    if (av == 0) {
        e->actions_done[e->n_done++] = ORC_FOLD;
        return 1;
    } else if (av == 1) {
        e->history[p][e->round][e->round_raises][0] = 1.0;
        e->round_raises += 1;
        if (e->n_done > 0 && e->actions_done[e->n_done - 1] == ORC_RAISE) e->overall_raises[p] += 1.0;
        if (e->round == 0 && e->n_done == 0) e->overall_raises[p] += 0.5;
        e->actions_done[e->n_done++] = ORC_CALL;
        return 0;
    } else {
        e->history[p][e->round][e->round_raises][1] = 1.0;
        e->raises[p] += 1.0;
        if (e->n_done > 0 && e->actions_done[e->n_done - 1] == ORC_RAISE) e->overall_raises[p] += 2.0;
        else e->overall_raises[p] += 1.0;
        e->round_raises += 1;
        if (e->round == 0 && e->n_done == 0) e->overall_raises[p] += 0.5;
        e->actions_done[e->n_done++] = ORC_RAISE;
        return 0;
    }
}

static int nfsp_round_over(const OrcNfspEnv *e) { /* newenv.py:180-190 */
    const int *d = e->actions_done;
    if (e->n_done == 2) {
        if ((d[0] == ORC_CALL && d[1] == ORC_CALL) || (d[0] == ORC_RAISE && d[1] == ORC_CALL)) return 1;
    } else if (e->n_done == 3) {
        if ((d[0] == ORC_CALL && d[1] == ORC_RAISE && d[2] == ORC_CALL) ||
            (d[0] == ORC_RAISE && d[1] == ORC_RAISE && d[2] == ORC_CALL))
            return 1;
    }
    return 0;
}

static int count_nonzero3(const double v[3]) { return (v[0] != 0) + (v[1] != 0) + (v[2] != 0); }
static int argmax3d(const double v[3]) { return argmax3(v); }

void orc_nfsp_step(OrcNfspEnv *e, const double action[3], int p) { /* newenv.py:192-349 */
    orc_nfsp_state_vector(e, p, e->s[p]); /* newenv.py:200-202 snapshot, even when terminated */
    if (e->terminated) {
        e->anomalies++; /* newenv.py:346-348 "tried to step while terminated" */
        return;
    }
    int o = 1 - p;
    e->terminated = nfsp_do_action(e, action, p);
    if (!e->terminated && nfsp_round_over(e)) {
        if (e->round == 1) {
            e->terminated = 1;
        } else { /* newenv.py:215-242 */
            memcpy(e->specific_cards[p][1], e->specific_cards[p][0], sizeof(double) * 3);
            memcpy(e->specific_cards[o][1], e->specific_cards[o][0], sizeof(double) * 3);
            e->public_card_index = e->deck[e->deck_pos++];
            e->specific_cards[p][1][e->public_card_index] = 1.0;
            e->specific_cards[o][1][e->public_card_index] = 1.0;
            e->round = 1;
            e->raises[0] = e->raises[1] = 0.0;
            e->round_raises = 0;
            e->n_done = 0;
        }
        if (fabs(e->reward[p]) - fabs(e->reward[o]) != 0) e->anomalies++; /* newenv.py:246-247 */
    }
    if (e->terminated) {
        int av = argmax3(action);
        if (av == 0) { /* newenv.py:252-258 */
            e->reward[p] = e->overall_raises[p] * -1.0;
            e->reward[o] = e->overall_raises[p];
        } else { /* newenv.py:261-298 */
            double *pc = e->specific_cards[p][e->round];
            double *oc = e->specific_cards[o][e->round];
            e->reward[p] = e->overall_raises[o];
            e->reward[o] = e->overall_raises[p];
            if (count_nonzero3(pc) == 1) {
                e->reward[o] *= -1.0;
            } else if (count_nonzero3(oc) == 1) {
                e->reward[p] *= -1.0;
            } else {
                if (e->round == 1) { pc[e->public_card_index] = 0; oc[e->public_card_index] = 0; }
                int ap = argmax3d(pc), ao = argmax3d(oc);
                if (ap < ao) e->reward[o] *= -1.0;
                else if (ap > ao) e->reward[p] *= -1.0;
                else { e->reward[0] = 0; e->reward[1] = 0; }
                if (e->round == 1) { pc[e->public_card_index] = 1; oc[e->public_card_index] = 1; }
            }
        }
        if (e->reward[p] + e->reward[o] != 0) e->anomalies++; /* newenv.py:344-345 */
    }
}

/* ======================= agent/agent.py nets (fp32) =============================== */
static void mlp_hidden(const OrcNet *n, const float x[30], float h[64]) { /* agent.py:102,111 */
    for (int j = 0; j < 64; ++j) {
        float acc = 0.f;
        for (int i = 0; i < 30; ++i) acc += x[i] * n->W1[i * 64 + j];
        acc += n->b1[j];
        h[j] = acc > 0.f ? acc : 0.f;
    }
}
static void mlp_logits(const OrcNet *n, const float h[64], float z[3]) {
    for (int c = 0; c < 3; ++c) {
        float acc = 0.f;
        for (int j = 0; j < 64; ++j) acc += h[j] * n->W2[j * 3 + c];
        z[c] = acc + n->b2[c];
    }
}
void orc_mlp_br(const OrcNet *n, const float x[30], float q[3]) { /* agent.py:101-103 */
    float h[64], z[3];
    mlp_hidden(n, x, h);
    mlp_logits(n, h, z);
    for (int c = 0; c < 3; ++c) q[c] = z[c] > 0.f ? z[c] : 0.f;
}
void orc_mlp_avg(const OrcNet *n, const float x[30], float pi[3]) { /* agent.py:110-112 */
    float h[64], z[3];
    mlp_hidden(n, x, h);
    mlp_logits(n, h, z);
    float m = z[0] > z[1] ? z[0] : z[1];
    m = m > z[2] ? m : z[2];
    float e0 = expf(z[0] - m), e1 = expf(z[1] - m), e2 = expf(z[2] - m);
    float s = e0 + e1 + e2;
    pi[0] = e0 / s; pi[1] = e1 / s; pi[2] = e2 / s;
}

/* ======================= batched seeded rollouts ================================== */
typedef struct {
    OrcNfspEnv env;
    int need_reset, policy[2], acted_nonzero[2], last_a[2];
    int hand_count;
} NfspGame;

struct OrcNfspBatch {
    int n;
    uint64_t seed, game0;
    NfspGame *g;
};

OrcNfspBatch *orc_nfsp_batch_create(int n_games, uint64_t seed, uint64_t game0) {
    OrcNfspBatch *b = (OrcNfspBatch *)calloc(1, sizeof(*b));
    b->n = n_games;
    b->seed = seed;
    b->game0 = game0;
    b->g = (NfspGame *)calloc((size_t)n_games, sizeof(NfspGame));
    return b;
}
void orc_nfsp_batch_destroy(OrcNfspBatch *b) {
    if (!b) return;
    free(b->g);
    free(b);
}
const OrcNfspEnv *orc_nfsp_batch_env(const OrcNfspBatch *b, int g) { return &b->g[g].env; }
void orc_nfsp_batch_flags(const OrcNfspBatch *b, int g, int out[4]) {
    out[0] = b->g[g].need_reset;
    out[1] = b->g[g].policy[0];
    out[2] = b->g[g].policy[1];
    out[3] = b->g[g].hand_count;
}

static void nfsp_game_reset(const OrcNfspBatch *b, int gi, int dealer, uint64_t step, uint32_t eta_u32) {
    NfspGame *g = &b->g[gi];
    uint32_t x[4];
    int ranks[3];
    /* generation spec: the step block (stream 0) carries .x action / epsilon, .y deal, .z .w policies */
    game_block(b->seed, b->game0 + (uint64_t)gi, step, 0u, x);
    deal_from_index(mulhi32(x[1], 120u), ranks);
    orc_nfsp_reset(&g->env, dealer, ranks[0], ranks[1], ranks[2]);
    /* main.py:38-45: policy 'a' iff random.random() > eta; here 'b' iff u32 draw < eta*2^32 */
    g->policy[0] = x[2] < eta_u32;
    g->policy[1] = x[3] < eta_u32;
    g->acted_nonzero[0] = g->acted_nonzero[1] = 0;
    g->last_a[0] = g->last_a[1] = 0;
    g->need_reset = 0;
    g->hand_count += 1;
}

void orc_nfsp_batch_reset(OrcNfspBatch *b, const int32_t *dealer, uint64_t step, uint32_t eta_u32) {
    for (int i = 0; i < b->n; ++i) {
        int d = dealer ? (dealer[i] & 1) : (int)((b->game0 + (uint64_t)i) & 1u);
        nfsp_game_reset(b, i, d, step, eta_u32);
    }
}

/* replay mode: install an explicit hand (dealer, deck, policies) instead of a Philox deal */
void orc_nfsp_batch_inject(OrcNfspBatch *b, int gi, int dealer, int c0, int c1, int pub, int pol0, int pol1) {
    NfspGame *g = &b->g[gi];
    orc_nfsp_reset(&g->env, dealer, c0, c1, pub);
    g->policy[0] = pol0;
    g->policy[1] = pol1;
    g->acted_nonzero[0] = g->acted_nonzero[1] = 0;
    g->last_a[0] = g->last_a[1] = 0;
    g->need_reset = 0;
    g->hand_count += 1;
}

static uint32_t trace_misc(const NfspGame *g, int raw, int started) {
    const OrcNfspEnv *e = &g->env;
    int eff = e->n_done > 0 ? e->actions_done[e->n_done - 1] : 0;
    /* after a round change actions_done was cleared: the closing action is always a call */
    if (e->n_done == 0) eff = ORC_CALL;
    uint32_t m = 0;
    m |= (uint32_t)raw;
    m |= (uint32_t)eff << 2;
    m |= (uint32_t)e->round << 4;
    m |= (uint32_t)e->dealer << 5;
    m |= (uint32_t)e->deck[0] << 6;
    m |= (uint32_t)e->deck[1] << 8;
    m |= (uint32_t)e->deck[2] << 10;
    m |= (uint32_t)(e->round == 1) << 12;
    m |= (uint32_t)(int)(e->overall_raises[0] * 2.0) << 13;
    m |= (uint32_t)(int)(e->overall_raises[1] * 2.0) << 17;
    m |= (uint32_t)started << 21;
    m |= (uint32_t)g->policy[0] << 22;
    m |= (uint32_t)g->policy[1] << 23;
    return m;
}

static int to_act(const OrcNfspEnv *e) { /* main.py:55-65: dealer opens both rounds, players alternate */
    return (e->round_raises % 2 == 0) ? e->dealer : 1 - e->dealer;
}

void orc_nfsp_batch_rollout_env(OrcNfspBatch *b, uint64_t step0, int n_steps, const int8_t *actions,
                                const int8_t *players, uint32_t eta_u32, OrcTraceRec *trace, int n_threads) {
    int n = b->n;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#pragma omp parallel for schedule(static)
#endif
    for (int gi = 0; gi < n; ++gi) {
        NfspGame *g = &b->g[gi];
        for (int t = 0; t < n_steps; ++t) {
            uint64_t step = step0 + (uint64_t)t;
            int started = 0;
            if (g->need_reset) {
                nfsp_game_reset(b, gi, 1 - g->env.dealer, step, eta_u32);
                started = 1;
            }
            int p = players ? players[(size_t)t * n + gi] : to_act(&g->env);
            int a;
            if (actions && actions[(size_t)t * n + gi] >= 0) {
                a = actions[(size_t)t * n + gi];
            } else {
                uint32_t x[4];
                game_block(b->seed, b->game0 + (uint64_t)gi, step, 0u, x);
                a = (int)mulhi32(x[0], 3u);
            }
            double vec[3] = {0, 0, 0};
            vec[a] = 1.0;
            orc_nfsp_step(&g->env, vec, p);
            if (trace) {
                double s2[30];
                orc_nfsp_state_vector(&g->env, p, s2);
                OrcTraceRec *r = &trace[(size_t)t * n + gi];
                r->obs = orc_mask30(s2) | ((uint32_t)g->env.terminated << 30) | ((uint32_t)p << 31);
                r->reward = g->env.terminated ? (float)g->env.reward[p] : 0.f;
                r->misc = trace_misc(g, a, started);
            }
            if (g->env.terminated) g->need_reset = 1;
        }
    }
}

static void push_rl(OrcRolloutOut *out, int p, uint32_t s, int a, float r, uint32_t s2, int t) {
    if (!out || !out->rl[p]) return;
    if (out->n_rl[p] < out->cap_rl[p]) {
        OrcRlRec *rec = &out->rl[p][out->n_rl[p]];
        rec->s = s; rec->s2 = s2; rec->r = r;
        rec->a = (uint8_t)a; rec->t = (uint8_t)t; rec->player = (uint8_t)p; rec->flags = 0;
    }
    out->n_rl[p]++;
}
static void push_sl(OrcRolloutOut *out, int p, uint32_t s, const float a[3]) {
    if (!out || !out->sl[p]) return;
    if (out->n_sl[p] < out->cap_sl[p]) {
        OrcSlRec *rec = &out->sl[p][out->n_sl[p]];
        rec->s = s; rec->a[0] = a[0]; rec->a[1] = a[1]; rec->a[2] = a[2];
    }
    out->n_sl[p]++;
}

/* One decision of Agent.play (agent.py:130-156) + main.train terminal observations (main.py:55-67),
 * for every game; canonical record order = (step, game, [prev transition, terminal]). Sequential over
 * games so that the per-player record order is well defined. */
void orc_nfsp_batch_rollout_act(OrcNfspBatch *b, uint64_t step0, int n_steps, const OrcNet nets[4],
                                uint32_t eta_u32, uint32_t eps_u32, const float *forced_vec, float *vec_out,
                                OrcTraceRec *trace, OrcRolloutOut *out, int n_threads) {
    orc_nfsp_batch_rollout_act2(b, step0, n_steps, nets, eta_u32, eps_u32, eps_u32, forced_vec, vec_out, trace, out, n_threads);
}

/* the same with one epsilon per player: every Agent decays its own (agent.py:78,253) */
void orc_nfsp_batch_rollout_act2(OrcNfspBatch *b, uint64_t step0, int n_steps, const OrcNet nets[4], uint32_t eta_u32,
                                 uint32_t eps0_u32, uint32_t eps1_u32, const float *forced_vec, float *vec_out,
                                 OrcTraceRec *trace, OrcRolloutOut *out, int n_threads) {
    (void)n_threads;
    int n = b->n;
    for (int t = 0; t < n_steps; ++t) {
        uint64_t step = step0 + (uint64_t)t;
        for (int gi = 0; gi < n; ++gi) {
            NfspGame *g = &b->g[gi];
            OrcNfspEnv *e = &g->env;
            int started = 0;
            if (g->need_reset) {
                nfsp_game_reset(b, gi, 1 - e->dealer, step, eta_u32);
                started = 1;
                if (out) out->hands++;
            }
            int p = to_act(e), o = 1 - p;
            double s2d[30];
            orc_nfsp_state_vector(e, p, s2d);
            uint32_t obs = orc_mask30(s2d);
            /* agent.py:132-136: remember the previous transition of this player */
            if (g->acted_nonzero[p]) push_rl(out, p, orc_mask30(e->s[p]), g->last_a[p], 0.f, obs, 0);
            float x[30], vec[3];
            for (int i = 0; i < 30; ++i) x[i] = (float)s2d[i];
            uint32_t u[4];
            game_block(b->seed, b->game0 + (uint64_t)gi, step, 0u, u);
            int is_br = g->policy[p];
            if (!is_br) {
                orc_mlp_avg(&nets[p * 2 + 0], x, vec); /* agent.py:143 */
            } else if (u[0] < (p ? eps1_u32 : eps0_u32)) { /* agent.py:125-128: random score vector, stream 1 */
                uint32_t y[4];
                game_block(b->seed, b->game0 + (uint64_t)gi, step, 1u, y);
                for (int c = 0; c < 3; ++c) vec[c] = (float)(y[c] >> 8) * (1.0f / 16777216.0f);
            } else {
                orc_mlp_br(&nets[p * 2 + 1], x, vec);
            }
            size_t vi = ((size_t)t * n + gi) * 3;
            if (vec_out) { vec_out[vi] = vec[0]; vec_out[vi + 1] = vec[1]; vec_out[vi + 2] = vec[2]; }
            if (forced_vec) { vec[0] = forced_vec[vi]; vec[1] = forced_vec[vi + 1]; vec[2] = forced_vec[vi + 2]; }
            if (is_br) push_sl(out, p, obs, vec); /* agent.py:151: raw a_t goes to the SL memory */
            int a = argmax3f(vec);
            double vd[3] = {vec[0], vec[1], vec[2]};
            orc_nfsp_step(e, vd, p);
            g->last_a[p] = a;
            g->acted_nonzero[p] = (vec[0] != 0.f) || (vec[1] != 0.f) || (vec[2] != 0.f); /* agent.py:134 */
            if (out) { out->played[p]++; out->actions[p][a]++; }
            if (trace) {
                double after[30];
                orc_nfsp_state_vector(e, p, after);
                OrcTraceRec *r = &trace[(size_t)t * n + gi];
                r->obs = orc_mask30(after) | ((uint32_t)e->terminated << 30) | ((uint32_t)p << 31);
                r->reward = e->terminated ? (float)e->reward[p] : 0.f;
                r->misc = trace_misc(g, a, started);
            }
            if (e->terminated) {
                /* main.py:55-67: both players observe the terminal state once via Agent.play */
                int order[2] = {p, o};
                for (int k = 0; k < 2; ++k) {
                    int q = order[k];
                    double fin[30];
                    orc_nfsp_state_vector(e, q, fin);
                    if (out) out->reward_half[q] += (int64_t)llround(e->reward[q] * 2.0); /* agent.py:133 */
                    if (g->acted_nonzero[q])
                        push_rl(out, q, orc_mask30(e->s[q]), g->last_a[q], (float)e->reward[q], orc_mask30(fin), 1);
                }
                g->need_reset = 1;
            }
        }
    }
}

/* ---------------- legacy batch ------------------------------------------------------ */
typedef struct {
    OrcLegacyEnv env;
    int hand_count, need_reset;
} LegacyGame;
struct OrcLegacyBatch {
    int n;
    uint64_t seed, game0;
    LegacyGame *g;
};
OrcLegacyBatch *orc_legacy_batch_create(int n_games, uint64_t seed, uint64_t game0) {
    OrcLegacyBatch *b = (OrcLegacyBatch *)calloc(1, sizeof(*b));
    b->n = n_games; b->seed = seed; b->game0 = game0;
    b->g = (LegacyGame *)calloc((size_t)n_games, sizeof(LegacyGame));
    for (int i = 0; i < n_games; ++i) orc_legacy_init(&b->g[i].env);
    return b;
}
void orc_legacy_batch_destroy(OrcLegacyBatch *b) {
    if (!b) return;
    free(b->g);
    free(b);
}
const OrcLegacyEnv *orc_legacy_batch_env(const OrcLegacyBatch *b, int g) { return &b->g[g].env; }

static void legacy_game_reset(const OrcLegacyBatch *b, int gi, uint64_t step) {
    uint32_t x[4];
    int ranks[3];
    game_block(b->seed, b->game0 + (uint64_t)gi, step, 0u, x);   /* legacy: .x .y actions, .z deal */
    deal_from_index(mulhi32(x[2], 120u), ranks);
    orc_legacy_reset(&b->g[gi].env, ranks[0], ranks[1]);
    b->g[gi].hand_count++;
    b->g[gi].need_reset = 0;
}
void orc_legacy_batch_reset(OrcLegacyBatch *b, uint64_t step) {
    for (int i = 0; i < b->n; ++i) legacy_game_reset(b, i, step);
}

void orc_legacy_batch_rollout(OrcLegacyBatch *b, uint64_t step0, int n_iters, const int8_t *actions,
                              OrcLegacyRec *out, int n_threads) {
    int n = b->n;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#pragma omp parallel for schedule(static)
#endif
    for (int gi = 0; gi < n; ++gi) {
        LegacyGame *g = &b->g[gi];
        for (int t = 0; t < n_iters; ++t) {
            uint64_t step = step0 + (uint64_t)t;
            int started = 0;
            if (g->need_reset) {
                legacy_game_reset(b, gi, step);
                started = 1;
            }
            int a[2];
            uint32_t x[4];
            game_block(b->seed, b->game0 + (uint64_t)gi, step, 0u, x);
            for (int p = 0; p < 2; ++p) {
                size_t ai = ((size_t)t * n + gi) * 2 + p;
                a[p] = (actions && actions[ai] >= 0) ? actions[ai] : (int)mulhi32(x[p], 3u);
            }
            /* README.md:15-38 driver: both players step, then both read the new state */
            for (int p = 0; p < 2; ++p) {
                double vec[3] = {0, 0, 0};
                vec[a[p]] = 1.0;
                orc_legacy_step(&g->env, vec, p);
            }
            int term = 0;
            for (int p = 0; p < 2; ++p) {
                int o5[5];
                orc_legacy_get_new_state(&g->env, p, o5);
                term |= o5[4];
                if (out) {
                    OrcLegacyRec *r = &out[((size_t)t * n + gi) * 2 + p];
                    r->card = (int8_t)o5[0]; r->pub = (int8_t)o5[1]; r->pot = (int8_t)o5[2];
                    r->terminal = (int8_t)o5[4];
                    r->reward = o5[3];
                    r->misc = (uint32_t)a[p] | ((uint32_t)(g->env.left[p] + 1) << 2) |
                              ((uint32_t)g->env.pot[p] << 5) | ((uint32_t)started << 8);
                }
            }
            if (term) g->need_reset = 1;
        }
    }
}

/* ======================= buffers ==================================================== */
void orc_ring_insert(OrcRing *r, const void *recs, int64_t n) { /* replay_buffer.py:30-41 */
    const uint8_t *src = (const uint8_t *)recs;
    for (int64_t i = 0; i < n; ++i) {
        int64_t slot = r->total % r->cap; /* append; when full, popleft() then append == overwrite oldest */
        memcpy(r->data + slot * r->rec_bytes, src + i * r->rec_bytes, (size_t)r->rec_bytes);
        r->total++;
        if (r->count < r->cap) r->count++;
    }
}

/* counter (idx, idx >> 32 | call >> 32, call, stream): the reservoir stream draws with call 0, the sample stream with
   idx < 1024, so the whole 64-bit ticket and the whole 64-bit call key the draw (DESIGN.md "Philox streams") */
static uint64_t buffer_u64(uint64_t seed, uint64_t idx, uint64_t call, uint32_t stream) {
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    uint32_t ctr[4] = {(uint32_t)idx, (uint32_t)(idx >> 32) | (uint32_t)(call >> 32), (uint32_t)call, stream};
    uint32_t o[4];
    orc_philox4x32_10(ctr, key, o);
    return (uint64_t)o[0] | ((uint64_t)o[1] << 32);
}

int64_t orc_reservoir_slot(uint64_t seed, int64_t ticket, int64_t cap, int mode) {
    if (ticket < cap) return ticket; /* ReservoirBuffer.py:22-24 fill phase */
    uint64_t u = buffer_u64(seed, (uint64_t)ticket, 0, 2u);
    if (mode == 1) { /* ReservoirBuffer.py:26-28: j = randrange(1, B+1); if j < B: buffer[j] = exp */
        int64_t j = 1 + (int64_t)mulhi64(u, (uint64_t)cap);
        return j < cap ? j : -1;
    }
    /* Algorithm R (Vitter 1985): item #ticket (0-based) replaces slot j ~ U[0, ticket] iff j < cap */
    int64_t j = (int64_t)mulhi64(u, (uint64_t)ticket + 1u);
    return j < cap ? j : -1;
}

void orc_reservoir_insert(OrcReservoir *r, const void *recs, int64_t n) {
    const uint8_t *src = (const uint8_t *)recs;
    for (int64_t i = 0; i < n; ++i) {
        int64_t slot = orc_reservoir_slot(r->seed, r->total, r->cap, r->mode);
        if (slot >= 0) memcpy(r->data + slot * r->rec_bytes, src + i * r->rec_bytes, (size_t)r->rec_bytes);
        r->total++;
        if (r->count < r->cap) r->count++;
    }
}

/* random.sample(buffer, B) (replay_buffer.py:46-51) -> uniform WITHOUT replacement; Floyd 1987 */
void orc_sample_indices(uint64_t seed, uint64_t call_idx, int64_t count, int batch, int64_t *out) {
    if (batch > count) batch = (int)count;
    int m = 0;
    for (int64_t i = count - batch; i < count; ++i) {
        uint64_t u = buffer_u64(seed, (uint64_t)(i - (count - batch)), call_idx, 3u);
        int64_t t = (int64_t)mulhi64(u, (uint64_t)i + 1u);
        int dup = 0;
        for (int k = 0; k < m; ++k)
            if (out[k] == t) { dup = 1; break; }
        out[m++] = dup ? i : t;
    }
}

int orc_hw_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
