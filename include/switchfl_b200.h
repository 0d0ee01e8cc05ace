/* switchfl_b200.h -- C-ABI of the B200 backend for SwitchFL's lockstep hot path.
 *
 * The reference (AI4REALNET/network-distributed-q-learning) is pure Python and has no FFI of its own;
 * the seam this library sits behind is the pair of Python classes used by main.py / test_model.py /
 * hyperparam_tuning.py (SURVEY.md section 8b).  Each entry point names the reference interface it
 * replaces (paths relative to the reference repository root).
 *
 * Conventions: every function returns 0 on success or a negative SFL_E_* code and never throws; all
 * bulk buffers are CALLER-OWNED device pointers (the Python host allocates them as torch tensors) and
 * the library never frees them; only the small map-constant block is owned by the context.  One
 * context per GPU per map, driven from one host thread; work is enqueued on the caller's stream
 * (a cudaStream_t passed as void*).  Several contexts (maps, devices) may live in one process and run on different streams at
 * the same time: a launch carries its map / layout / arguments as kernel parameters, there is no process-global device
 * state.  Every entry point runs on the device of its context and restores the caller's current device.  There is no CPU
 * path: without a CUDA device sfl_create fails.
 */
#ifndef SWITCHFL_B200_H
#define SWITCHFL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFL_ABI_VERSION 10

enum {
  SFL_OK = 0,
  SFL_E_ARG = -1,       /* bad argument / unsupported size                                   */
  SFL_E_CUDA = -2,      /* CUDA runtime error (see sfl_last_error)                           */
  SFL_E_NOMEM = -3,     /* caller buffer too small                                           */
  SFL_E_STATE = -4      /* call order (e.g. run before bind)                                 */
};

/* per-environment error bits, reported in sfl_env_counters.err (the reference raises instead)       */
enum {
  SFL_ERR_NO_TRAIN_AT_SWITCH = 1,   /* observer.py:294-307: the reference logs "Bug detected" and then dies on an unbound
                                       local (:307); here the episode is abandoned (counted in `aborted`) and the env resets */
  SFL_ERR_INF_DISTANCE = 2,         /* observer.py:35-36  ValueError                                 */
  SFL_ERR_Q_FULL = 4,               /* per-env Q hash table full                                     */
  SFL_ERR_PEND_FULL = 8,            /* pending-update list of a train full (distr_q.py:340-342)      */
  SFL_ERR_PLAN_FULL = 16,           /* train_action_plan longer than 4                               */
  SFL_ERR_REPLAY_UNDERRUN = 32,     /* replay action stream exhausted                                */
  SFL_ERR_BAD_ACTION = 64,          /* switch_env.py:213-215 assertion                               */
  SFL_ERR_REPLAY_DIVERGED = 128     /* replay: an action recorded as greedy is not the argmax here   */
};

/* run modes (sfl_run) */
enum {
  SFL_MODE_LEARN = 0,    /* distr_q.py:296-366  epsilon-greedy + Q-update (Philox, or the reference's PCG64: sfl_config.rng) */
  SFL_MODE_GREEDY = 1,   /* distr_q.py:195-224  test(): max_action only, no update                   */
  SFL_MODE_REPLAY = 2,   /* learn() with the actions (and malfunction events) of a recorded trace; an action
                            with bit 6 set was an exploit choice: the row is looked up (inserted) and the
                            recorded action must equal the argmax                                     */
  SFL_MODE_STEP = 3      /* host-driven AEC protocol (switch_env.py:616-666): one launch applies the action the
                            host chose for the waiting decision (replay_act[env * act_cap]), advances the trains to
                            the next decision point and reports it in step_out; no learning on the device            */
};

/* Map + line + timetable constants, all HOST pointers; copied by sfl_create.
 * Replaces the construction work of ASyncSwitchEnv.__init__ -> RailNetwork.__init__
 * (switch_env.py:30-52, rail_network.py:84-133) and the per-reset constants of switch_env.py:93-158;
 * the tables are produced by railmap.py (rows A0, F6, Q4 of SURVEY.md section 8a).                   */
typedef struct sfl_map_desc {
  int32_t H, W;                 /* grid size (square: rail_graph.py:43-48)                            */
  int32_t S, NP, NA, T, NT;     /* switches, ports, moving actions (sum of A-1), trains, targets      */
  int32_t max_episode_steps;    /* flatland timetable (flatland_patch/timetable_generators.py:94-101) */
  const uint16_t *grid;         /* [H*W] flatland 16-bit transitions                                  */
  const int32_t *cell_switch;   /* [H*W] switch index or -1                                           */
  const int32_t *sw_P, *sw_A, *sw_port0, *sw_act0;   /* [S], [S], [S+1], [S+1]                        */
  const int32_t *port_nbr, *port_dist, *port_n_intra, *port_intra0;   /* [NP]                         */
  const int32_t *act_in, *act_out, *act_move;        /* [NA] local port indices, RailEnvActions       */
  const int32_t *init_cell, *init_dir, *target_cell, *ed, *la;        /* [T]                          */
  const int32_t *first_port, *first_dist, *init_delay, *tgt_index;    /* [T] (switch_env.py:507-568)  */
  const int32_t *dist;          /* [NT*H*W*4] distance map, 0x3FFFFFFF = unreachable                  */
  const int8_t *qinit_act;      /* [NP*NT] optimistic action or -1 (distr_q.py:81-181)                */
  const uint8_t *qinit_final;   /* [NP*NT] 1 -> 1000. (last leg), 0 -> 500.                           */
} sfl_map_desc;

typedef struct sfl_config {
  int32_t n_envs;
  int32_t q_cap;                /* Q hash rows per environment, power of two                          */
  int32_t pend_cap;             /* pending updates per train (update_dict, distr_q.py:283)            */
  int32_t max_steps;            /* ASyncSwitchEnv max_steps (100000 in every script)                  */
  int32_t dec_cap, tick_cap;    /* trace capacities per env (0 = tracing off)                         */
  int32_t ep_cap;               /* episode-log capacity per env                                       */
  int32_t act_cap, ev_cap;      /* replay capacities per env                                          */
  int32_t trace_sem;            /* 1: also log the semaphore table after each decision                */
  int32_t shared_q;             /* 1: shared-table mode (extension, no counterpart in the reference): every environment
                                   of this context reads ONE dense Q table and accumulates its TD steps into a delta
                                   buffer; sfl_shared_q_apply folds the mean step into the table (see DESIGN.md)  */
  int32_t rng;                  /* epsilon-greedy stream of SFL_MODE_LEARN: SFL_RNG_PHILOX (0) or SFL_RNG_REFERENCE (1)      */
  int32_t malf_rng;             /* malfunction draws: SFL_MALF_PHILOX (0) or SFL_MALF_REFERENCE (1)                           */
  int32_t eval_q;               /* 1: evaluation context -- greedy runs on ONE read-only Q table (sfl_set_eval_table) shared by
                                   every environment; no per-environment tables.  0: today's layout                       */
} sfl_config;

/* sfl_config.rng.
 * SFL_RNG_PHILOX: counter-based Philox4x32-10 draws (DESIGN.md section 4); the specialised learn kernels.
 * SFL_RNG_REFERENCE: the reference learner's own numpy stream, so that a seeded learn() makes the reference's decisions.
 *   distr_q.py:269 creates rng = np.random.default_rng(seed) at the start of learn(); per decision (:315-317)
 *     if rng.random() < epsilon * epsilon_decay_rate ** n:      n = interactions of the deciding switch
 *         action_space.seed(int(rng.integers(0, 2**31 - 1)))  then  action = action_space.sample(mask)
 *   i.e. Generator(PCG64(SeedSequence(sd))).choice(where(mask)).  Here: per environment one PCG64 generator (SeedSequence
 *   seeding, XSL-RR output, random() = (next_uint64 >> 11) * 2^-53, integers() = Lemire's method on 32-bit draws with
 *   the carried half-word), seeded from sfl_hparams.seed by every sfl_reset that does not keep the interaction counters
 *   (keep bit 1 clear: the start of a learn() call) and continued by every other reset; consumed by SFL_MODE_LEARN only,
 *   one random() per decision, exploit included.  The comparison with epsilon is exact (the power is recomputed when the
 *   draw is within rounding of it); decisions equal the reference's when lr_decay_rate == 1 (else Q-values agree to
 *   1e-12 relative, and so do decisions unless a tie is that close).  Learn runs use the full kernel; a bound
 *   malfunction schedule (ev_cap > 0) replaces the Philox malfunction draws in learn mode too.  Not with shared_q.
 *   The stream's state takes 48 bytes of every env block, after the header; with SFL_RNG_PHILOX it takes none.      */
enum { SFL_RNG_PHILOX = 0, SFL_RNG_REFERENCE = 1 };

/* sfl_config.malf_rng.
 * SFL_MALF_PHILOX: the two-stage Philox malfunction draw (sfl_hparams.malf_threshold, DESIGN.md section 4), unless a
 *   schedule is bound (ev_cap > 0: replay, greedy and step mode, and learn mode with SFL_RNG_REFERENCE).
 * SFL_MALF_REFERENCE: flatland's own stream, so that a seeded run has the reference's malfunctions.  rail_env.reset
 *   (random_seed=seed) creates np_random = np.random.RandomState(seed) at every episode (switch_env.py:99); each tick
 *   1 .. max_episode_steps, for every train in handle order, ParamMalfunctionGen draws rand() < 1 - exp(-rate) and, on a
 *   hit, randint(min_duration, max_duration + 1) + 1 steps.  No draw depends on the actions, so the schedule is a function
 *   of (seed, rate, min, max, T, max_episode_steps), the same in every episode.  sfl_malf_schedule writes it into replay_ev;
 *   every mode then applies it (learn mode on the full kernel), an event only while the train's counter is 0.  Needs
 *   ev_cap >= 1; not with shared_q.                                                                                    */
enum { SFL_MALF_PHILOX = 0, SFL_MALF_REFERENCE = 1 };

/* sfl_config.eval_q: evaluating one learned policy on many environments (eval.py:31-97 runs test() ten times).
 * Greedy rollouts never change a decision by writing: the only write test() makes is the insert-on-lookup of a default
 * row (distr_q.py:482 -> :56-57), and a missing row and a fresh default row give the same max_action.  So an evaluation
 * context keeps no per-environment Q region (env_stride ends after the per-switch records) and q_cap is the capacity of
 * ONE open-addressing table (same row format, hash and probing as the private tables) in the caller-owned buffer
 * sfl_buffers.eval_q (sfl_sizes.eval_q_bytes), filled by sfl_set_eval_table.  The greedy kernel probes it through the
 * non-coherent path and never inserts: a miss reads as the default row (default_q x A).  The table is not mutated and
 * q_rows stays 0; lazy Q-init (sfl_enable_q_init) does not apply -- put the optimistic rows into the table.
 * sfl_run accepts SFL_MODE_GREEDY only, without traces or the phase clock.  Not with shared_q or SFL_RNG_REFERENCE
 * (a greedy run draws no epsilon); SFL_MALF_REFERENCE is allowed (flatland's malfunctions of every seed).               */

/* DistrQLearning.__init__ arguments (distr_q.py:32) + MalfunctionParameters (main.py:28-33), per env */
typedef struct sfl_hparams {
  double gamma, epsilon, epsilon_decay_rate, lr, lr_decay_rate, default_q;
  uint64_t seed;                /* Philox key; the reference's seed (SFL_RNG_REFERENCE, SFL_MALF_REFERENCE) */
  uint32_t malf_threshold;      /* floor((1 - exp(-rate)) * 2^32), 0 = no malfunctions                */
  int32_t malf_min, malf_max;   /* duration = min + U{0..max-min} + 1                                 */
  int32_t episodes;             /* halt after this many episodes since sfl_reset (<0: never)          */
  int32_t episode_base;         /* global index of the first episode after sfl_reset (RNG stream offset) */
  uint32_t malf_thr2;           /* floor(malf_threshold * 256 / ceil(malf_threshold / 2^24)): stage-2 threshold of the
                                   two-stage malfunction draw (DESIGN.md section 4); 0 when malf_threshold is 0  */
} sfl_hparams;

/* byte sizes of the caller-owned buffers for a (map, config) pair */
typedef struct sfl_sizes {
  uint64_t state_bytes;         /* env state incl. Q tables                                           */
  uint64_t env_stride;          /* bytes per env inside state                                         */
  uint64_t hparams_bytes;       /* n_envs * sizeof(sfl_hparams)                                       */
  uint64_t trace_dec_bytes, trace_tick_bytes, trace_sem_bytes;
  uint64_t ep_log_bytes, ep_delay_bytes;
  uint64_t replay_act_bytes, replay_ev_bytes;
  uint64_t counters_bytes;      /* n_envs * sizeof(sfl_env_counters)                                  */
  uint64_t step_out_bytes;      /* n_envs * sizeof(sfl_step_rec) (SFL_MODE_STEP only)                 */
  uint64_t shared_q_bytes;      /* shared-table mode: NP*NT*48 rows x a_max doubles (the table)       */
  uint64_t shared_d_bytes;      /*   ... x a_max int64 (sum of TD steps, fixed point 2^-24)           */
  uint64_t shared_c_bytes;      /*   ... x a_max int32 (number of TD steps)                           */
  int32_t q_stride;             /* doubles per Q row (1 key slot + A_max)                             */
  int32_t a_max;
  uint64_t rng_offset;          /* SFL_RNG_REFERENCE: byte offset of the stream's state in an env block: uint64 state_hi,
                                   state_lo, inc_hi, inc_lo, uint32 has_uint32, uinteger (numpy's PCG64 state); 0 otherwise */
  uint64_t eval_q_bytes;        /* sfl_config.eval_q: q_cap rows x q_stride doubles (the evaluation table); 0 otherwise     */
} sfl_sizes;

typedef struct sfl_buffers {    /* all device pointers; optional ones may be NULL                     */
  void *state; void *hparams; void *counters;
  void *trace_dec; void *trace_tick; void *trace_sem;
  void *ep_log; void *ep_delay;
  void *replay_act; void *replay_ev;
  void *step_out;
  void *shared_q; void *shared_d; void *shared_c;    /* shared-table mode; shared_d / shared_c may be all-reduced (sum) by the caller */
  void *eval_q;                                      /* sfl_config.eval_q: the evaluation table (eval_q_bytes); mandatory there */
} sfl_buffers;

typedef struct sfl_env_counters {      /* written by sfl_run for every env                            */
  uint64_t decisions, ticks, train_ticks;   /* lifetime totals                                        */
  int32_t episodes, err, q_rows, halted;
  int32_t n_dec_logged, n_tick_logged, n_ep_logged, elapsed;
  int32_t aborted, reserved;                /* episodes abandoned on SFL_ERR_NO_TRAIN_AT_SWITCH      */
  uint64_t forced_stops;                    /* decisions whose action mask allowed STOP only (switch_agents.py:104-134)   */
  uint64_t stop_actions;                    /* decisions that chose STOP                                                   */
  uint64_t arrived_trains;                  /* trains at their destination, summed over the finished episodes (distr_q.py:364) */
  uint64_t reserved2;
  uint64_t phase_cycles[6];                 /* sfl_set_phase_clock: SM cycles spent per phase -- 0 train ticks (rail_env.step + _move_trains
                                               bookkeeping), 1 observe (last()), 2 action selection, 3 apply + reward (rest of step()),
                                               4 Q-update, 5 episode reset: the split behind the timers main.py:72-78 prints     */
} sfl_env_counters;

typedef struct sfl_dec_rec {           /* one switch-agent decision (trace)                           */
  int32_t ep, tick, sw, train;
  uint32_t key;                        /* dense state index (see DESIGN.md)                           */
  int32_t mask, action, next_sw, reward, done;
  uint64_t arrived;                    /* trains 0..63 at their destination after the decision, bit t = train t       */
  uint64_t arrived_hi;                 /* trains 64..127 (bit t - 64); 0 when T <= 64                                 */
} sfl_dec_rec;

/* SFL_MODE_STEP output per environment: what AECEnv.last() returns for the waiting decision (observer.py:246-308)
 * plus what the previous ASyncSwitchEnv.step() returned (switch_env.py:663-666)                              */
typedef struct sfl_step_rec {
  int32_t pending;                     /* 1: (sw, train) waits for an action; 0: episode over (see done)             */
  int32_t sw, train;
  uint32_t key;                        /* dense state index of the observation                                        */
  int32_t mask;                        /* action mask, bit a = action a allowed                                       */
  int32_t done;                        /* terminated | truncated << 1                                                 */
  int32_t elapsed;                     /* rail_env._elapsed_steps                                                     */
  int32_t last_next_sw;                /* "next_switch" of the decision just applied, -1 if none                      */
  uint64_t arrived;                    /* "arrived_trains" as a bit set: trains 0..63                                 */
  int32_t rewards[128];                /* _cumulative_rewards[sw][train] for every train (switch_env.py:130, 289)     */
  uint64_t arrived_hi;                 /* trains 64..127 of "arrived_trains" (bit t - 64); 0 when T <= 64             */
} sfl_step_rec;

typedef struct sfl_tick_rec { int32_t pos; int8_t dir, state; int16_t malf; } sfl_tick_rec;
typedef struct sfl_ep_rec {            /* one finished episode (distr_q.py:360-366)                   */
  double cum_reward; int32_t decisions, arrived, num_malfunctions, ticks;
  uint64_t arrived_mask;               /* the trains at their destination ("arrived_trains", :345, 371): trains 0..63 */
  uint64_t arrived_mask_hi;            /* trains 64..127 (bit t - 64); 0 when T <= 64                 */
} sfl_ep_rec;

/* Distance map (flatland DistanceMap as vendored in flatland_patch/distance_map.py:62-167; SURVEY.md row F6 / N1):
 * dist[k][r][c][heading] = moves from (cell, heading) to target_cells[k], 0x3FFFFFFF if unreachable; all four headings
 * of a target cell are 0.  Host pointers in and out (one-off map preprocessing); computed on `device` by one CTA per
 * target relaxing d(cell, o) = 1 + min over the exits h of (cell, o) of d(cell + step(h), h) to its fixed point.     */
int sfl_distance_map(const uint16_t *grid, int32_t H, int32_t W, const int32_t *target_cells, int32_t n_targets,
                     int32_t *dist, int device);

/* Known-answer hook (SURVEY.md Appendix C KAT-3): the library's Q-update arithmetic -- distr_q.py:441-447, fp64, the
 * reference's operator order, no FMA contraction -- evaluated ON THE DEVICE for n rows of host operands
 * {q, lr, reward, gamma, max_next, bootstrap (0: the train stayed at the same switch, :444-447)}; out[i] = new Q(s, a). */
int sfl_kat_q_update(const double *operands, int32_t n, double *out, int device);

/* Known-answer hooks of SFL_RNG_REFERENCE, evaluated ON THE DEVICE with the kernel's own functions.
 * sfl_kat_pcg64: n generators, gens[6 g ..] = {state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger}, or -- when inc_lo is
 * even (a PCG64 increment is odd) -- the generator np.random.default_rng(state_lo); then n_codes draws each, codes[g n_codes + k]:
 *   0                     random()                                     -> the double's bits
 *   1 .. 2^32             integers(0, code)                            -> the value
 *   2^63 | mask           one exploring decision (distr_q.py:316-317)  -> the action: the integers(0, 2**31 - 1)-th seed's
 *                         Generator(PCG64(SeedSequence(sd))).choice over the set bits of mask
 * out[(12 + n_codes) g ..] = the 6 words after seeding, the n_codes results, the 6 words of the final state.
 * sfl_kat_explore: rows {u, epsilon, decay, n, running product of the decay over n interactions}; out[i] = 1 iff the
 * kernel explores, i.e. u < epsilon * decay ** n as the reference evaluates it (distr_q.py:315).                      */
int sfl_kat_pcg64(const uint64_t *gens, const uint64_t *codes, int32_t n, int32_t n_codes, uint64_t *out, int device);
int sfl_kat_explore(const double *rows, int32_t n, int32_t *out, int device);

/* SFL_MALF_REFERENCE: flatland's malfunction schedule of every environment, generated ON THE DEVICE (numpy's MT19937:
 * init_genrand, twist, tempering; rand() from two words; legacy randint by masked rejection on 32-bit words) into the
 * bound replay_ev: the events (tick, train, duration) drawn for ticks 1 .. max_episode_steps in tick order, -1 after the
 * last.  Seed, min_duration and max_duration come from the bound sfl_hparams (seed.. malf_max; malf_threshold is not
 * used); hit_below[n_envs] (host) = ceil(p * 2^53) with p = 1 - exp(-rate) (0 for rate <= 0), so that a draw hits iff its
 * 53-bit integer k < hit_below.  *max_events = the largest number of events of an environment.  SFL_E_ARG for a seed
 * RandomState refuses (not below 2^32) or min_duration > max_duration; SFL_E_NOMEM when a schedule has more than ev_cap
 * events (nothing is truncated).  Synchronises `stream`.                                                            */
int sfl_malf_schedule(void *ctx, const uint64_t *hit_below, int32_t *max_events, void *stream);

int sfl_abi_version(void);
const char *sfl_last_error(void);

/* Sizes of everything the caller must allocate.  No counterpart in the reference, where the Python objects own their
 * memory (env: switch_env.py:42-73, learner: distr_q.py:33-57); here PyTorch does, and the library is told how much.  */
int sfl_query_sizes(const sfl_map_desc *map, const sfl_config *cfg, sfl_sizes *out);

/* replaces ASyncSwitchEnv(rail_env, ...) + DistrQLearning(env, ...)   (main.py:51-60).  T must be in 1..128;
 * shared-table mode (sfl_config.shared_q) takes at most 64 trains and neither SFL_RNG_REFERENCE nor SFL_MALF_REFERENCE
 * (the reference has no shared table, and its learner one stream).  SFL_MALF_REFERENCE needs ev_cap >= 1.            */
int sfl_create(const sfl_map_desc *map, const sfl_config *cfg, int device, void **ctx);
int sfl_destroy(void *ctx);                       /* env.close() (switch_env.py, called at distr_q.py:241, 379) + garbage collection */
int sfl_bind(void *ctx, const sfl_buffers *bufs); /* hand over the caller-owned device buffers sized by sfl_query_sizes            */

/* zero state + mark every env "needs reset"; the first sfl_run performs env.reset (switch_env.py:93-158)
 * on the device.  keep bit 0 keeps the Q tables, bit 1 the per-switch interaction counters (and, with SFL_RNG_REFERENCE,
 * continues the random stream; without bit 1 every environment's stream restarts from sfl_hparams.seed).              */
int sfl_reset(void *ctx, int keep_q, void *stream);

/* Lanes of a warp that cooperate on one environment (1, 2, 4, 8, 16 or 32; 32/lanes environments share a warp and
 * one instruction stream).  sfl_create picks max(lanes that cover the trains in one pass, lanes that still give the
 * batch ~3.5 warps per SM scheduler); this overrides it.  A scheduling choice only: results do not depend on it.
 * Maps with more than 64 trains run on 8, 16 or 32 lanes.                                              */
int sfl_set_lanes(void *ctx, int lanes);
int sfl_get_lanes(void *ctx);
/* Warps per CTA of the hot-path kernel: 0 = automatic (4, halved while the launch has fewer than 8 CTAs per SM), or 1, 2,
 * 4.  A scheduling choice only.                                                                        */
int sfl_set_cta_warps(void *ctx, int warps);

/* Compile-time variant of the large-map learn kernel: 1 = the one built for 4 CTAs per SM (more registers), 0 = the one
 * for 7, -1 = automatic (roomy when the launch fits one wave anyway).  A scheduling choice only.                   */
int sfl_set_roomy(void *ctx, int roomy);
/* Per-phase cycle counters (sfl_env_counters.phase_cycles) for the wall-clock breakdown main.py:68-78 prints
 * (switch_env.py:67-73 accumulators).  Instrumented runs use the full kernel (the one that also carries the traces);
 * off by default: the production kernels carry no clock reads.                                                       */
int sfl_set_phase_clock(void *ctx, int on);
/* Which kernel instantiation and launch configuration sfl_run(mode) would use now (traced != 0: with decision / tick
 * traces), as text: "k_run<G=..,KIND=..,TH=..,SQ=..,ONE=..,ROOMY=..> grid=.. block=.. smem=..", with ",NW=2" after ROOMY
 * on maps with more than 64 trains (two words per train set); learn with SFL_RNG_REFERENCE or SFL_MALF_REFERENCE is KIND=full.  Evaluation
 * contexts (sfl_config.eval_q) name their kernel "k_eval<G=..,KIND=greedy,TH=..,SQ=0,ONE=..,ROOMY=0[,NW=2],EVQ=1> ...".  No counterpart in the
 * reference; it lets the parity tests name -- and force, with sfl_set_lanes / sfl_set_roomy -- exactly the
 * instantiations the benchmark launches.  Needs no bound buffers.                                                  */
int sfl_describe_launch(void *ctx, int mode, int traced, char *buf, int cap);

/* enable the optimistic initialisation of distr_q.py:299-300 for rows created from now on           */
int sfl_enable_q_init(void *ctx, int on);

/* __init_q_table runs at the first episode of EVERY learn() call and ASSIGNS its rows (distr_q.py:299-300, 156-158, 179-181):
 * overwrite, in every environment's table, the rows of optimistic-init states that already exist (an earlier learn(),
 * load() or test() created them) with their initial values.  Device-side; uses the bound hparams (default_q).            */
int sfl_reapply_q_init(void *ctx, void *stream);

/* advance every env by up to max_ticks flatland ticks (all decisions in between included);
 * replaces the loop body of DistrQLearning.learn / test  (distr_q.py:302-362, 199-224)               */
int sfl_run(void *ctx, int mode, int max_ticks, void *stream);

/* Shared-table mode: Q[s][a] += (sum of the TD steps proposed for (s, a) since the last apply) / (their number), then
 * the delta buffers are cleared.  Across GPUs the caller all-reduces shared_d and shared_c (integer sums: order
 * independent, bit-reproducible) before calling this, which leaves identical tables on every rank.                 */
int sfl_shared_q_apply(void *ctx, void *stream);
/* The same on explicit buffers: q_dst = q_src + mean step of (d, cnt), which are cleared.  With two tables and two
 * accumulator pairs bound alternately (sfl_bind is a pointer swap) the all-reduce + apply of step k can run on a second
 * stream while sfl_run of step k+1 reads the other table: see Engine.run_shared in backend.py and DESIGN.md section 6.   */
int sfl_shared_q_apply_to(void *ctx, const void *q_src, void *q_dst, void *d, void *cnt, void *stream);

/* Sum over all envs of the decisions taken (num_iter, distr_q.py:284, 361) and of the flatland ticks
 * (rail_env._elapsed_steps) after the last run: device reduction, 16-byte D2H.                         */
int sfl_total_decisions(void *ctx, uint64_t *decisions, uint64_t *ticks, void *stream);

/* Q-table export for distr_q_model.pkl (distr_q.py:492-523): rows of env `env` as (key, A_max values) */
int sfl_export_q(void *ctx, int env, uint32_t *keys_host, double *vals_host, int cap_rows, int *n_rows, void *stream);
/* Q-table import (distr_q.py:510-527 load) */
int sfl_import_q(void *ctx, int env, const uint32_t *keys_host, const double *vals_host, int n_rows, void *stream);
/* sfl_config.eval_q: fill the bound evaluation table with n_rows (key, A_max values) rows -- the hash image sfl_import_q
 * builds, once, uploaded into sfl_buffers.eval_q; a repeated key overwrites its row.  SFL_E_NOMEM when n_rows >= q_cap.
 * Synchronises `stream`.  Export / import of per-environment rows do not exist in these contexts.                    */
int sfl_set_eval_table(void *ctx, const uint32_t *keys_host, const double *vals_host, int n_rows, void *stream);

#ifdef __cplusplus
}
#endif
#endif
