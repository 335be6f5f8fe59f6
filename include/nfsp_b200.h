/* nfsp_b200.h -- C ABI of libnfsp_b200.so: the B200-native batched Leduc Hold'em + NFSP rollout
 * path (env step, NFSP act, replay/reservoir memories).
 *
 * The reference (dantodor/Neural-Ficititious-Self-Play-in-Imperfect-Information-Games) has no
 * FFI: its boundary is four duck-typed Python classes.  Each entry point below names the
 * reference method it replaces (file:line in the reference tree); INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every call returns 0 on success, a negative NFSP_E_* code on failure; the message of the
 *     last failure on the calling thread is nfsp_last_error();
 *   - all `d_*` pointers are DEVICE pointers owned by the caller (the Python host allocates them
 *     with torch); nothing here allocates or synchronises in a hot call;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - a handle is bound to one device, is not thread-safe, and distinct handles are independent;
 *   - there is NO CPU fallback: without a CUDA device every compute entry fails with
 *     NFSP_E_CUDA.
 */
#ifndef NFSP_B200_H
#define NFSP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFSP_OK 0
#define NFSP_E_ARG (-1)
#define NFSP_E_CUDA (-2)
#define NFSP_E_STATE (-3)

#define NFSP_RULES_LEGACY 0 /* leduc/env.py    */
#define NFSP_RULES_NFSP 1   /* leduc/newenv.py */

#define NFSP_OBS_DIM 30        /* newenv.py:68-74 */
#define NFSP_ACTIONS 3         /* newenv.py:63-66 */
#define NFSP_HIDDEN 64         /* config.ini:4    */
#define NFSP_NET_PARAMS 2179   /* 30*64 + 64 + 64*3 + 3 (agent.py:101-103) */
#define NFSP_EXPORT_FIELDS 24  /* int32 columns of nfsp_env_export   */
#define NFSP_LEGACY_EXPORT_FIELDS 14
#define NFSP_STATS_FIELDS 16   /* uint64 counters, see nfsp_rollout  */

typedef struct nfsp_env_s *nfsp_env_t;

int nfsp_version(void);
const char *nfsp_last_error(void);
/* number of SMs / device name of `device`, for sizing (no handle needed) */
int nfsp_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len);

/* ------------------------------------------------------------------ lifecycle ------------- */
/* One packed 64-bit word per game in HBM.  Games are numbered game0 .. game0+n_games-1; all
 * randomness is Philox4x32-10 keyed by (seed; global game id, step counter, purpose), so a
 * game's trace does not depend on how games are sharded over GPUs.
 * Replaces Env.__init__ (env.py:13-32, newenv.py:14-55). */
int nfsp_env_create(int rules, int64_t n_games, uint64_t seed, uint64_t game0, int device, nfsp_env_t *out);
int nfsp_env_destroy(nfsp_env_t h);
int64_t nfsp_env_num_games(nfsp_env_t h);
int nfsp_env_rules(nfsp_env_t h);
/* the Philox step counter: advanced by one per reset call and per stepped transition */
uint64_t nfsp_env_step_counter(nfsp_env_t h);
int nfsp_env_set_step_counter(nfsp_env_t h, uint64_t step);
/* device pointer to the n_games packed words */
void *nfsp_env_state_ptr(nfsp_env_t h);
/* Protocol-error word of the rollout kernels (synchronises the device): 0 = none.  The warp-specialised rollout bounds
 * every wait it makes (queues, mbarriers); a wait that runs out sets a bit here and the kernel ends instead of hanging
 * the GPU -- the launch's results are then invalid.  Nothing comparable exists in the reference (single thread). */
int nfsp_env_kernel_error(nfsp_env_t h, uint32_t *out);
/* copy the n_games packed 64-bit words out of / into the handle (checkpoint / resume, sharding tests) */
int nfsp_env_save_state(nfsp_env_t h, uint64_t *d_out, void *stream);
int nfsp_env_load_state(nfsp_env_t h, const uint64_t *d_in, void *stream);

/* ------------------------------------------------------------------ ENV_NFSP -------------- */
/* newenv.Env.reset(dealer) (newenv.py:76-114) for every game: d_dealer int8[n] or NULL
 * (NULL => global game id & 1).  Deals from Philox; draws the per-hand policies of
 * main.py:38-45 with P('b') = eta. */
int nfsp_env_reset(nfsp_env_t h, const int8_t *d_dealer, double eta, void *stream);
/* replay mode: install explicit hands. d_cards int8[n][3] = ranks popped by p0, p1, public
 * (deck.py:49-50); d_policy int8[n][2] (0 = 'a', 1 = 'b') or NULL. */
int nfsp_env_set_hands(nfsp_env_t h, const int8_t *d_dealer, const int8_t *d_cards, const int8_t *d_policy,
                       void *stream);
/* newenv.Env.step(action, p_index) (newenv.py:192-349) n_steps times for every game.
 *   d_actions int8[n_steps][n] or NULL: 0/1/2 = np.argmax(action); 3 = the all-zero vector (a fold
 *             that Agent.play does not remember, agent.py:134); -1 or NULL = uniform Philox action;
 *             4 = the game sits this step out (per-game call sequences).
 *   d_players int8[n_steps][n] or NULL: NULL => main.train's turn order (main.py:55-65).
 *   auto_reset: re-deal a finished hand at its next step (dealer alternates, main.py:28-31).
 *   d_trace   uint32[3][n_steps][n] or NULL: planes obs|terminal<<30|player<<31, reward (float
 *             bits), misc (DESIGN.md "trace record").
 * With d_actions = d_players = NULL and auto_reset (the throughput configuration) the call runs the state-machine
 * kernel (one table entry per (dealer, betting sequence, action), csrc/nfsp_fsm.cuh); every other combination runs
 * the general kernel on the packed word.  Both produce identical words and traces. */
int nfsp_env_step(nfsp_env_t h, const int8_t *d_actions, const int8_t *d_players, int n_steps, int auto_reset,
                  double eta, uint32_t *d_trace, void *stream);
/* Host only, no device needed: copies the table image of the state-machine step kernel (rows of newenv.Env.step /
 * main.train's turn order, the deal and reward tables; layout in csrc/nfsp_fsm.cuh) into out if capacity_words is
 * large enough.  Returns the image size in 32-bit words. */
int nfsp_fsm_image(uint32_t *out, int capacity_words);
/* The same for the legacy rules (leduc/env.py README iteration; layout in csrc/legacy_fsm.cuh); *n_rows receives the
 * number of states a rollout can reach. */
int nfsp_legacy_fsm_image(uint32_t *out, int capacity_words, int *n_rows);
/* The image the default rollout (variant 6) steps its games on (layout in csrc/nfsp_fsm.cuh, "the fused rollout's
 * image"; addresses are byte offsets from the state table it follows); returns its size in words. */
int nfsp_rollout_image(uint32_t *out, int capacity_words);
/* newenv.Env.do_action (newenv.py:131-178) called on its own, for callers that drive the pieces of step() themselves:
 * raise->call coercions, history bit, round_raises, chips, last_action -- no snapshot, no round change, no showdown,
 * `terminated` untouched.  d_actions int8[n]: np.argmax(action), 3 = all-zero vector (argmax 0 = fold), negative =
 * no call for this game; d_players
 * int8[n]; d_fold int8[n] or NULL receives the return value (1 = the player folded). */
int nfsp_env_do_action(nfsp_env_t h, const int8_t *d_actions, const int8_t *d_players, int8_t *d_fold, void *stream);
/* newenv.Env.get_state(p) (newenv.py:116-129), packed: player < 0 => per-game d_players.
 * Outputs (any may be NULL): d_s snapshot mask, d_s2 current observation mask, d_reward,
 * d_term, d_last_a (argmax of last_action[p], 3 if it was never set / all-zero). */
int nfsp_env_observe(nfsp_env_t h, const int8_t *d_players, int player, uint32_t *d_s, uint32_t *d_s2,
                     float *d_reward, uint8_t *d_term, uint8_t *d_last_a, void *stream);
/* unpacked view int32[n][NFSP_EXPORT_FIELDS] (tests / debugging) */
int nfsp_env_export(nfsp_env_t h, int32_t *d_fields, void *stream);

/* ------------------------------------------------------------------ ENV_LEGACY ------------ */
/* env.Env.reset() (env.py:46-72), Philox deal */
int nfsp_legacy_reset(nfsp_env_t h, void *stream);
/* replay mode: d_cards int8[n][2] */
int nfsp_legacy_set_hands(nfsp_env_t h, const int8_t *d_cards, void *stream);
/* env.Env.step(action, player_index) (env.py:84-158); d_actions int8[n] = np.argmax(action), 4 = the
 * game sits this call out; player < 0 => per-game d_players int8[n] (a value > 1 also sits out) */
int nfsp_legacy_step(nfsp_env_t h, const int8_t *d_actions, const int8_t *d_players, int player, void *stream);
/* env.Env.get_new_state(player_index) (env.py:160-205); d_out int32[n][5] =
 * {card, public(-1), pot, reward, terminal} or NULL (state still mutates, as in the reference) */
int nfsp_legacy_get_new_state(nfsp_env_t h, const int8_t *d_players, int player, int32_t *d_out, void *stream);
/* n_iters README iterations (README.md:15-38): step(a0,0); step(a1,1); get_new_state(0);
 * get_new_state(1); auto re-deal when either reports terminal.  d_actions int8[n_iters][n][2] or
 * NULL (Philox).  d_rec uint32[3][n_iters][n][2] or NULL: planes card|pub<<8|pot<<16|terminal<<24
 * (signed bytes), reward (int32), misc. 2 transitions per game per iteration. */
int nfsp_legacy_rollout(nfsp_env_t h, const int8_t *d_actions, int n_iters, uint32_t *d_rec, void *stream);
int nfsp_legacy_export(nfsp_env_t h, int32_t *d_fields, void *stream);

/* ------------------------------------------------------------------ dense views ----------- */
/* 30-bit masks -> float32 [n][30] rows of 0/1 (the reference's state vectors, newenv.py:118-122) */
int nfsp_expand_obs(const uint32_t *d_masks, int64_t n, float *d_out, void *stream);

/* ------------------------------------------------------------------ NFSP acting ----------- */
/* Four acting nets, index player*2 + policy (policy 0 = average 'a', 1 = best response 'b'),
 * each NFSP_NET_PARAMS floats in Keras Dense order W1[30][64], b1[64], W2[64][3], b2[3]
 * (agent.py:90-116).  Repacks them into the kernels' layouts inside the handle. */
int nfsp_act_set_weights(nfsp_env_t h, const float *d_weights, void *stream);
/* The same from host memory (pinned for a truly asynchronous copy): float[4][2179] is copied into d_weights on the
 * stream, then the images are built from it -- one call for the learner -> actor weight hand-over of a step. */
int nfsp_act_set_weights_from_host(nfsp_env_t h, const float *h_weights, float *d_weights, void *stream);
/* batched Model.predict (agent.py:126,143): d_obs uint32[n] masks, d_net int8[n] net index;
 * d_out float[n][3] = Q-values (relu head) for BR nets, softmax probabilities for average nets */
int nfsp_act_forward(nfsp_env_t h, const uint32_t *d_obs, const int8_t *d_net, int64_t n, float *d_out,
                     void *stream);

/* Same contract as nfsp_act_forward, first layer on the 5th-generation tensor cores: tcgen05.mma with the
 * accumulator in TMEM, the four nets stacked along K, fp32 weights as an exact 3-way bf16 split. */
int nfsp_act_forward_tc(nfsp_env_t h, const uint32_t *d_obs, const int8_t *d_net, int64_t n, float *d_out,
                        void *stream);

/* Record formats (16 B each):
 *   RL  {u32 s, u32 s2, f32 r, u8 a, u8 t, u8 player, u8 flags}   replay_buffer.py:30-41, by value
 *   SL  {u32 s, f32 a[3]}                                          ReservoirBuffer.py:18-28       */
typedef struct {
    void *d_rl[2];        /* per-player staging, RL records: [n_segments][cap_rl]               */
    void *d_sl[2];        /* per-player staging, SL records: [n_segments][cap_sl]               */
    int64_t cap_rl, cap_sl; /* slots PER SEGMENT                                                */
    int32_t n_segments;   /* power of two; the 32 consecutive games starting at g append to segment
                             (g / 32) % n_segments, each segment has its own ticket counter      */
    uint32_t *d_counts;   /* uint32[4][n_segments]: rl0, rl1, sl0, sl1 appended so far (device)  */
    uint64_t *d_stats;    /* uint64[NFSP_STATS_FIELDS] or NULL: actions[2][3], played[2],
                             reward_half[2] (two's complement), hands, transitions, dropped     */
    uint32_t *d_trace;    /* as nfsp_env_step, or NULL                                          */
    float *d_vec;         /* float[n_steps][n][3] score vectors actually used, or NULL          */
    const float *d_forced_vec; /* float[n_steps][n][3] or NULL: use these instead of the nets   */
    int32_t variant;      /* first layer on: 1 = CUDA cores (sum of two precombined weight rows, bank-conflict-free
                             shared-memory gathers), 2 = tensor cores, one mixed-net tile per 128-thread group,
                             3 = tensor cores, warp-specialised: env warps -> per-net tile queues -> tcgen05.mma on
                             net-homogeneous M128 N64 tiles -> epilogue warpgroups (TMEM -> relu -> 64x3 with W2 from
                             the constant bank), 4 = CUDA cores with net-sorted warp groups (see below), 5 = CUDA cores, two
                             games per lane, the second layer's weights loaded once for a pair of same-net decisions
                             (csrc/rollout_pairs.cu), 6 = no per-decision forward at all: the nets' outputs on the 702
                             decision states of the game, recomputed by one small launch whenever the weights have
                             changed (same arithmetic as variant 1), one 16-byte shared-memory read per decision, records
                             collected in warp-private shared-memory buffers (csrc/rollout_states.cu: the default),
                             0 = library default */
    int32_t reserve_sms;  /* variants 1, 3, 4, 5 and 6: SMs left free for kernels of other streams (the learner's fit running
                             beside the rollout); the persistent grid is sm_count - reserve_sms CTAs.  0 = use them all */
    /* variants 1, 4, 5 and 6, all NULL / 0 otherwise: the RL records go straight into the players' rings instead of d_rl
     * (ReplayBuffer.add, replay_buffer.py:30-41, done by the rollout kernel itself): ticket = atomic add on
     * *d_ring_total[p] (records ever inserted, advanced by the kernel), slot = ticket % ring_cap.  d_rl is not
     * written and needs no nfsp_ring_insert afterwards.  Requires 2 * n * n_steps <= ring_cap: the records of one
     * launch must not lap the ring (their order inside a launch is the order of the atomic tickets). */
    void *d_ring[2];
    uint64_t *d_ring_total[2];
    int64_t ring_cap;
    /* each Agent of the reference decays its own epsilon (agent.py:253): with epsilon_per_player != 0 the `epsilon`
     * argument of nfsp_rollout is player 0's and epsilon_p1 player 1's; otherwise both use `epsilon` */
    int32_t epsilon_per_player;
    double epsilon_p1;
} nfsp_rollout_io;
/* 4 = CUDA cores, the decisions of a four-warp group sorted by net so that warps are net-homogeneous, records appended
 * with one set of atomics per group: n_segments must be 1 (csrc/rollout_sorted.cu).  An experiment kept for the record:
 * an LDS.128 costs four shared-memory cycles whatever its lanes read, so net-homogeneous warps save nothing
 * (profiles/r02/sorted_rollout_notes.txt) */
#define NFSP_ROLLOUT_DEFAULT_VARIANT 6

/* The fused hot path: for n_steps, every game does one Agent.play decision (agent.py:130-156)
 * -- observe, remember the previous transition, eta-mixed policy (average net argmax /
 * epsilon-greedy best-response net), env.step -- plus the terminal observations of main.py:55-67,
 * with auto re-deal.  Records are appended to the segmented staging arrays with warp-aggregated
 * atomics; move them into the memories with nfsp_ring_insert / nfsp_reservoir_insert. */
int nfsp_rollout(nfsp_env_t h, int n_steps, double eta, double epsilon, const nfsp_rollout_io *io, void *stream);
/* The learner -> actor hand-over and the rollout in one call (one trip through the binding instead of two at the head of
 * every step): nfsp_act_set_weights_from_host(h, h_weights, d_weights, stream) followed by nfsp_rollout(...).  With
 * h_weights = NULL the nets are already in d_weights (a learner on the same device has just written them):
 * nfsp_act_set_weights(h, d_weights, stream) followed by nfsp_rollout(...). */
int nfsp_rollout_with_weights(nfsp_env_t h, const float *h_weights, float *d_weights, int n_steps, double eta, double epsilon,
                              const nfsp_rollout_io *io, void *stream);
/* Independent runs side by side: n_runs handles, each with its own games, step counter, seed, weight images, state table,
 * memories and counters, whose hot launches are shared.  Run r does exactly what it would do alone, bit for bit.
 * The same as n_runs calls nfsp_rollout(h[r], n_steps, eta[r], epsilon[r], &io[r], stream) -- preceded by
 * nfsp_act_set_weights(h[r], d_weights[r], stream) when d_weights is not NULL -- with variant 6 and no debug outputs
 * (io[r].variant 0 or 6; d_trace, d_vec, d_forced_vec NULL; player 1's epsilon through io[r].epsilon_p1 as there).
 *   - d_weights (float[4][2179] per run) or NULL: the weight images and state tables of all runs are rebuilt first, in one
 *     launch each (the run on blockIdx.y); every handle is then left as nfsp_act_set_weights leaves it.
 *   - the rollout is ONE launch: the CTAs are split into contiguous ranges of floor((SMs - reserve_sms) / n_runs) or
 *     fewer, one range per run, and a CTA serves its run as the run's own launch on that many CTAs would.
 * The runs must share their shape: device, game count, direct or staged records, n_segments, ring_cap and reserve_sms;
 * otherwise, or with n_runs outside [1, min(NFSP_MAX_RUNS, SMs - reserve_sms)], the call returns NFSP_E_ARG before
 * anything is launched.  Every handle's step counter advances by n_steps. */
#define NFSP_MAX_RUNS 32
int nfsp_rollout_runs(const nfsp_env_t *h, int n_runs, int n_steps, const double *eta, const double *epsilon,
                      const nfsp_rollout_io *io, float *const *d_weights, void *stream);
/* Tuning of variant 3: SM cycles a partly filled tile of an average-policy / a best-response net may wait for more rows
 * before its MMAs are issued anyway (defaults 1500 / 700). */
int nfsp_rollout_tune(nfsp_env_t h, int patience_avg, int patience_br);
/* Cycle counters of variant 3's three roles (only counted by a library built with -DNFSP_TQ_PROF, else zeros);
 * layout in csrc/rollout_tq.cu.  Synchronises the device. */
int nfsp_rollout_profile(nfsp_env_t h, uint64_t *out24);

/* ------------------------------------------------------------------ memories -------------- */
/* A staged batch is n_segments segments of seg_cap 16-byte slots with one device count each
 * (d_counts uint32[n_segments]); n_segments = 1 is a plain dense array.  Batch order = segment order, then
 * slot order.  The batch is consumed: on the stream, *d_total += records and the counts are zeroed.
 * Every insert is ONE cooperative launch (segment prefixes, grid barrier, the moves, commit); d_scratch is
 * uint64[n_segments + NFSP_INSERT_SCRATCH_WORDS] of device memory per memory, zeroed once by the caller and left to
 * the library afterwards (barrier words + the prefix table); calls that share a scratch block must be stream-ordered.
 *
 * ReplayBuffer.add (replay_buffer.py:30-41) for a batch: FIFO ring of cap 16-byte records, slot = ticket % cap where
 * ticket counts records ever inserted (*d_total); of a batch larger than the ring only the last `cap` survive. */
#define NFSP_INSERT_SCRATCH_WORDS 4
int nfsp_ring_insert(void *d_ring, int64_t cap, uint64_t *d_total, const void *d_recs, uint32_t *d_counts,
                     int n_segments, int64_t seg_cap, uint64_t *d_scratch, void *stream);
/* ReservoirBuffer.add (ReservoirBuffer.py:18-28) for a batch.  mode 0 = Algorithm R (Vitter):
 * ticket t >= cap replaces slot j ~ U[0,t] iff j < cap; mode 1 = the reference's law
 * (j = randrange(1, cap+1), replace iff j < cap).  Same-slot collisions inside a batch are
 * resolved as in the sequential algorithm (largest ticket wins).
 * Storage: d_res is cap slots of NFSP_RESERVOIR_SLOT_BYTES = 32 bytes (one DRAM sector), zeroed once:
 *   {16-byte SL record, uint64 stamp = ticket + 1 of the record that owns the slot, uint64 unused}
 * so the stamp's atomic and the record's store touch the same sector.  Record j is at d_res + 32 * j. */
#define NFSP_RESERVOIR_SLOT_BYTES 32
int nfsp_reservoir_insert(void *d_res, int64_t cap, uint64_t *d_total, const void *d_recs, uint32_t *d_counts,
                          int n_segments, int64_t seg_cap, uint64_t seed, int mode, uint64_t *d_scratch, void *stream);
/* The same for several memories in one launch: request k is exactly nfsp_ring_insert (reservoir = 0) /
 * nfsp_reservoir_insert (reservoir = 1) with these arguments; seed and mode are read for reservoirs only.
 * nfsp_insert_multi takes any mix -- after a rollout both players' rings and reservoirs travel together --
 * nfsp_ring_insert_multi / nfsp_reservoir_insert_multi insist on one kind.  The barrier words of request 0 serve
 * the whole launch. */
#define NFSP_MAX_INSERT_REQS 4
typedef struct {
    void *d_mem;
    int64_t cap;
    uint64_t *d_total;
    uint64_t *d_scratch;
    const void *d_recs;
    uint32_t *d_counts;
    int32_t n_segments;
    int64_t seg_cap;
    uint64_t seed;
    int32_t mode;
    int32_t reservoir;
} nfsp_insert_req;
int nfsp_insert_multi(const nfsp_insert_req *reqs, int n, void *stream);
int nfsp_ring_insert_multi(const nfsp_insert_req *reqs, int n, void *stream);
int nfsp_reservoir_insert_multi(const nfsp_insert_req *reqs, int n, void *stream);
/* random.sample(buffer, batch) (replay_buffer.py:46-51, ReservoirBuffer.py:33-37): `batch`
 * distinct positions (Floyd's algorithm, Philox keyed by (seed; call_idx)); d_idx int64[batch]
 * receives storage slots, d_n_out the number drawn = min(batch, size).  is_ring: positions are
 * deque positions (oldest first) mapped to ring slots. */
int nfsp_sample_indices(uint64_t seed, uint64_t call_idx, const uint64_t *d_total, int64_t cap, int is_ring,
                        int batch, int64_t *d_idx, uint32_t *d_n_out, void *stream);
/* sample_batch(batch) of up to NFSP_MAX_SAMPLE_REQS memories in one launch (Agent.update_strategy draws from the RL and
 * the SL memory of a player back to back, agent.py:212-262): request m draws its positions exactly as
 * nfsp_sample_indices(seed, call_idx, ...) does and expands the rows as nfsp_gather_rl / nfsp_gather_sl do into d_out,
 * one contiguous block: ring (RL)  s[batch][30] a[batch][3] r[batch] s2[batch][30] t[batch]  = 65 * batch floats,
 * reservoir (SL)  s[batch][30] a[batch][3]  = 33 * batch floats.  d_idx int64[n_reqs][batch] (storage slots, -1 beyond
 * the records held) and d_n_out uint32[n_reqs] (rows sampled) may be NULL.  A request with d_out = NULL only reports its
 * positions in d_idx (the learner kernels read the packed records themselves); with d_rec_out NULL as well it reads no
 * record and d_mem may be NULL. */
#define NFSP_MAX_SAMPLE_REQS 128 /* 4 * NFSP_MAX_RUNS: the four memories of every run of a batch */
typedef struct {
    const void *d_mem;        /* ring (16-byte records) / reservoir (32-byte slots, the record first) storage */
    const uint64_t *d_total;  /* records ever inserted (device) */
    int64_t cap;
    uint64_t seed, call_idx;
    int32_t is_ring;
    float *d_out;
    void *d_rec_out;          /* or NULL: packed copies of the sampled slots, row k at the memory's slot size (16 bytes for a
                                 ring, 32 for a reservoir, the record first) -- a snapshot the learner kernels can read in
                                 place of the memory (slots 0 .. batch-1) while the memory itself moves on */
} nfsp_sample_req;
int nfsp_sample_minibatches(const nfsp_sample_req *reqs, int n_reqs, int batch, int64_t *d_idx, uint32_t *d_n_out,
                            void *stream);
/* gather + expand to the dense float32 batches the learner consumes (replay_buffer.py:53-59):
 * s [b][30], a [b][3] (one-hot of the stored argmax), r [b], s2 [b][30], t [b] */
int nfsp_gather_rl(const void *d_ring, const int64_t *d_idx, int batch, float *d_s, float *d_a, float *d_r,
                   float *d_s2, float *d_t, void *stream);
/* ReservoirBuffer.sample_batch (ReservoirBuffer.py:39-43): s [b][30], a [b][3]; d_res = 32-byte slots */
int nfsp_gather_sl(const void *d_res, const int64_t *d_idx, int batch, float *d_s, float *d_a, void *stream);

/* ------------------------------------------------------------------ learner (SURVEY 8 f-1) */
#define NFSP_LEARNER_STATS 8
typedef struct {
    const float *d_weights;        /* [4][NFSP_NET_PARAMS] acting nets, index player*2 + policy               */
    const float *d_target_weights; /* [2][NFSP_NET_PARAMS] target best-response nets (agent.py:70-72)         */
    const void *d_rl[2];           /* the players' rings and the sampled slots (nfsp_sample_indices)          */
    const int64_t *d_rl_idx[2];
    const void *d_sl[2];           /* the players' reservoirs (32-byte slots) and the sampled slots           */
    const int64_t *d_sl_idx[2];
    int32_t row0, rows;            /* minibatch = sampled rows [row0, row0+rows) (Keras fit batches of 32)    */
    float gamma;                   /* config.ini Agent.Gamma                                                  */
    int32_t net_mask;              /* bit k: net k trains (its memory holds > MiniBatchSize, agent.py:215,259) */
    int32_t terminal_bootstraps;   /* 1 = reference quirk agent.py:227 (terminal transitions bootstrap too)   */
    int32_t others_to_target;      /* 1 = the two Q outputs of a row that were not taken regress to the target net's
                                      predictions on s, as `target = target_br_model.predict(s_batch)` makes them
                                      (agent.py:220,243); 0 = they have zero error                                */
    float *d_grad;                 /* out [4][NFSP_NET_PARAMS] mean gradients: the flat all-reduce buffer ... */
    float *d_stats;                /* out [NFSP_LEARNER_STATS], laid out right behind it by the host:
                                      expl_sum_p0, expl_sum_p1, rows_p0, rows_p1, loss sums of the 4 nets      */
} nfsp_learner_io;
/* Agent.update_best_response_network / update_avg_response_network (agent.py:209-264), gradient part:
 * forward + backward of all four nets on one minibatch, read straight from the packed memories. */
int nfsp_learner_grads(const nfsp_learner_io *io, void *stream);
/* Keras' fit(x, y, batch_size = fit_batch, epochs = epochs) of all four nets (agent.py:243,261) on ONE GPU in a single
 * launch: the SGD steps over the slices [0, fit_batch), [fit_batch, 2 fit_batch), ... of the `minibatch` sampled rows,
 * `epochs` times, each step = the gradients of nfsp_learner_grads followed by nfsp_sgd_apply with scale 1 -- the
 * weights stay in registers between the steps.  io->row0 / rows / d_grad are not read; io->d_stats receives the
 * statistics of the first step.  d_weights_out float[4][2179] may be io->d_weights.  With more than one GPU the steps
 * need a collective between gradient and update: use nfsp_learner_grads + all-reduce + nfsp_sgd_apply. */
#define NFSP_MAX_FIT_STEPS 64
int nfsp_learner_fit(const nfsp_learner_io *io, int minibatch, int fit_batch, int epochs, const float lr[4],
                     float *d_weights_out, void *stream);
/* The fits of n_runs independent runs in ONE launch of 4 * n_runs CTAs (blockIdx.x = 4 * run + net): the same as n_runs
 * calls nfsp_learner_fit(&io[r], minibatch, fit_batch, epochs, lr + 4 * r, d_weights_out[r], stream), each with its own
 * memories, sampled slots, net_mask, gamma, flags, target nets, statistics and output weights (d_weights_out[r] may be
 * io[r].d_weights).  The SGD step schedule (minibatch, fit_batch, epochs) is shared; 1 <= n_runs <= NFSP_MAX_RUNS. */
int nfsp_learner_fit_runs(const nfsp_learner_io *io, int n_runs, int minibatch, int fit_batch, int epochs, const float *lr,
                          float *const *d_weights_out, void *stream);
/* The same fit when several GPUs of one box train together (SURVEY 8e, C1 + C2): the all-reduce of every SGD step runs
 * INSIDE the kernel over peer memory (NVLink).  Each rank owns an exchange buffer of NFSP_PEER_BUF_FLOATS floats, zeroed
 * once, that every other rank can address (CUDA IPC / torch symmetric memory); d_buf[r] is rank r's buffer as THIS
 * process sees it.  Per step a rank pushes its mean gradients and statistics as 8-byte {value, epoch} words into its
 * slot of EVERY rank's buffer and polls its own buffer until all slots carry the step's epoch (no flags, no fences, no
 * round trip), then sums them in rank order -- so the weights stay bit-identical on every rank.  epoch0 = SGD steps
 * exchanged through these buffers so far (the same on all ranks; add the steps of this call afterwards).  *d_err becomes
 * 1 if a peer did not answer within ~2 s (the kernel then gives up on that net instead of hanging the GPU and writes NaN
 * weights for it: the result is invalid and visibly so).  Every rank must make the same call.
 * The exchange lives in the row-parallel fit kernel (one warp per sampled row, the weights in shared memory), which holds
 * at most NFSP_FIT_ROWS_MAX_MINIBATCH sampled rows and NFSP_FIT_ROWS_MAX_STEP rows per SGD step: larger geometries are
 * refused here.  nfsp_learner_fit and nfsp_learner_fit_runs run them on the register kernel instead. */
#define NFSP_FIT_ROWS_MAX_MINIBATCH 256
#define NFSP_FIT_ROWS_MAX_STEP 64
#define NFSP_MAX_PEERS 8
#define NFSP_PEER_BUF_FLOATS 279552 /* 2 parities x 4 nets x NFSP_MAX_PEERS senders x 2184 words of 8 bytes */
typedef struct {
    int32_t world, rank;
    void *d_buf[NFSP_MAX_PEERS];
    uint32_t epoch0;
    uint32_t *d_err;
    void *d_mc;   /* or NULL: a multicast mapping of the SAME buffers (NVLS: one store through it lands in every rank's
                     buffer at that offset); the pushes then leave the SM once instead of `world` times */
} nfsp_peers;
int nfsp_learner_fit_peers(const nfsp_learner_io *io, int minibatch, int fit_batch, int epochs, const float lr[4],
                           float *d_weights_out, const nfsp_peers *peers, void *stream);
/* Exchange buffers for nfsp_learner_fit_peers without any framework help: a rank creates its buffer (cudaMalloc,
 * zeroed) and gets its 64-byte CUDA IPC handle, sends the handle to the other ranks of the box over any channel, and
 * opens theirs; nfsp_peers.d_buf[r] = rank r's buffer as this process maps it, d_mc = NULL (no multicast mapping on this
 * route).  close = unmap a peer's buffer, destroy = free one's own (after every peer has closed it). */
int nfsp_peer_buffer_create(int device, void **d_buf, unsigned char *handle64);
int nfsp_peer_buffer_open(int device, const unsigned char *handle64, void **d_buf);
int nfsp_peer_buffer_close(int device, void *d_buf);
int nfsp_peer_buffer_destroy(int device, void *d_buf);
/* keras SGD step (agent.py:45-46,243,261): w[k] -= lr[k] * scale * grad[k]; scale = 1/world after a SUM
 * all-reduce.  lr is a HOST array of 4 floats. */
int nfsp_sgd_apply(float *d_weights, const float *d_grad, const float lr[4], float scale, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NFSP_B200_H */
