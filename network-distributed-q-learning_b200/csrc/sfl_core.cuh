// sfl_core.cuh -- per-environment logic of SwitchFL's lockstep hot path.
//
// Restates (not ports) rows E1-E7, O1-O3, R1, Q1-Q3, F1-F5 of SURVEY.md section 8a for a batched,
// structure-of-arrays device layout.  Citations "file:line" are relative to the reference repository.
//
// Execution model: a GROUP of G lanes (G = 1, 2, 4, ... 32, a template parameter chosen per launch from the batch
// size) owns one environment for the whole launch; 32/G environments share a warp and ONE instruction stream: every
// sync and vote is issued by the whole warp at warp-uniform points of the control flow, the groups differ only in
// their predicates (see Grp below).  The per-tick train phase is lane-parallel inside the group (lane = train, in
// chunks of G when T > G); the per-decision phase is inherently serial inside an environment (every _apply_action
// mutates the semaphores the next observe reads, switch_env.py:648) and runs on the group's first lane -- for all
// groups of the warp at once.  What a launch cannot need is compiled out (kernel KIND, TH, SQ, ONE, EVQ: DESIGN.md section 4).
//
// The same source compiles for a single "lane" on the host: tests/emul builds it with g++ (-DSFL_HOST_EMUL) to
// unit-test the logic on the CPU box that has no GPU.  That build is test infrastructure; the product library
// has no CPU path.
#pragma once
#include <stdint.h>
#include "switchfl_b200.h"

#if defined(__CUDACC__) && !defined(SFL_HOST_EMUL)
#define SFL_DEV 1
#define SFL_FN __device__ __forceinline__
#define SFL_NI __device__ __forceinline__          // the Q probe / update: inline (see SFL_RARE)
#define SFL_RARE __device__ __noinline__          // once-per-episode paths: out of line (instruction cache), even though a
                                                  // noinline callee reads the kernel parameter block through a generic pointer
#define SFL_NU _Pragma("unroll 1")
#define SFL_U4 _Pragma("unroll 4")
#define SFL_UA _Pragma("unroll")
#else
#define SFL_DEV 0
#include <math.h>
#include <string.h>
#define SFL_FN inline
#define SFL_NI inline
#define SFL_RARE inline
#define SFL_NU
#define SFL_U4
#define SFL_UA
struct int4 { int x, y, z, w; };
struct int2 { int x, y; };
static inline int4 make_int4(int x, int y, int z, int w) { int4 r = {x, y, z, w}; return r; }
static inline int2 make_int2(int x, int y) { int2 r = {x, y}; return r; }
#endif

namespace sfl {

// flatland enums (SURVEY.md Appendix B)
enum { A_NOTHING = 0, A_LEFT = 1, A_FWD = 2, A_RIGHT = 3, A_STOP = 4, A_NONE = 0xFF };
enum { ST_WAITING = 0, ST_READY = 1, ST_MALF_OFF = 2, ST_MOVING = 3, ST_STOPPED = 4, ST_MALF = 5, ST_DONE = 6 };
enum { SEM_IN = 0, SEM_OUT = 1 };
#define SFL_INF_DIST 0x3FFFFFFF
#define SFL_MAX_T 128
#define SFL_PLAN_CAP 4

// ------------------------------------------------------------------------------------------------ lane groups
// A group = G consecutive lanes of a warp working on one environment.  Every collective below is issued by the WHOLE
// warp (full member mask) at warp-uniform points of the control flow: group-masked __syncwarp / votes let the groups of
// a warp drift apart, after which the warp executes the sum of their instruction streams instead of one shared stream.
// Branch conditions that guard a collective are therefore made warp-uniform with wany(); a group for which the
// condition does not hold walks through with its own predicate false.
#if SFL_DEV
template <int G> struct Grp {
  int gl;                    // my lane inside the group
  int shift;                 // first lane of my group inside the warp
  SFL_FN Grp() {
    int lane = threadIdx.x & 31;
    gl = lane & (G - 1);
    shift = lane & ~(G - 1);
  }
  SFL_FN void sync() const { __syncwarp(); }
  SFL_FN int wany(int p) const { return __any_sync(0xffffffffu, p); }          // over the warp
  SFL_FN unsigned wor(unsigned v) const { return __reduce_or_sync(0xffffffffu, v); }   // over the warp (one REDUX)
  // bit i = predicate of the group's lane i
  SFL_FN unsigned ballot(int p) const {
    unsigned b = __ballot_sync(0xffffffffu, p);
    return G == 32 ? b : (b >> shift) & ((1u << (G & 31)) - 1u);
  }
  SFL_FN int any(int p) const { return ballot(p) != 0u; }                       // over the group
};
SFL_FN int popc64(unsigned long long v) { return __popcll(v); }
SFL_FN int ffs64(unsigned long long v) { return __ffsll((long long)v) - 1; }
SFL_FN int popc32(unsigned v) { return __popc(v); }
SFL_FN double dmul(double a, double b) { return __dmul_rn(a, b); }
SFL_FN double dadd(double a, double b) { return __dadd_rn(a, b); }
SFL_FN double dfma(double a, double b, double c) { return __fma_rn(a, b, c); }
SFL_FN unsigned long long mulhi64(unsigned long long a, unsigned long long b) { return __umul64hi(a, b); }
template <class T> SFL_FN T ldg(const T *p) { return __ldg(p); }
#else
template <int G> struct Grp {
  int gl, shift;
  Grp() : gl(0), shift(0) {}
  void sync() const {}
  int wany(int p) const { return p; }
  unsigned wor(unsigned v) const { return v; }
  unsigned ballot(int p) const { return p ? 1u : 0u; }
  int any(int p) const { return p; }
};
SFL_FN int popc64(unsigned long long v) { return __builtin_popcountll(v); }
SFL_FN int ffs64(unsigned long long v) { return __builtin_ffsll((long long)v) - 1; }
SFL_FN int popc32(unsigned v) { return __builtin_popcount(v); }
SFL_FN double dmul(double a, double b) { volatile double r = a * b; return r; }
SFL_FN double dadd(double a, double b) { volatile double r = a + b; return r; }
SFL_FN double dfma(double a, double b, double c) { return fma(a, b, c); }
SFL_FN unsigned long long mulhi64(unsigned long long a, unsigned long long b) { return (unsigned long long)(((unsigned __int128)a * b) >> 64); }
template <class T> SFL_FN T ldg(const T *p) { return *p; }
#endif

// ------------------------------------------------------------------------------------------------ train sets
// A set of trains in NW 64-bit words, train t = bit (t & 63) of word (t >> 6): NW = 1 up to 64 trains, NW = 2 up to 128
// (SFL_MAX_T: the semaphore-holder mirror and the occupancy scratch hold train indices in one byte).  The words are
// named, never indexed by a runtime value, so that they stay in registers.  With NW = 1 every operation is the plain
// one-word expression.
template <int NW> struct TSet {
  static_assert(NW == 1 || NW == 2, "one or two words of trains");
  unsigned long long w[NW];
  SFL_FN void clear() { w[0] = 0ull; if (NW > 1) w[NW - 1] = 0ull; }
  // or in a group ballot whose bit 0 is train `base` (G divides 64: the chunk lies inside one word)
  SFL_FN void or_ballot(unsigned b, int base) {
    if (NW == 1) { w[0] |= (unsigned long long)b << base; return; }
    const unsigned long long v = (unsigned long long)b << (base & 63);
    if (base < 64) w[0] |= v; else w[NW - 1] |= v;
  }
  SFL_FN unsigned long long test(int t) const {
    if (NW == 1) return (w[0] >> t) & 1ull;
    return ((t < 64 ? w[0] : w[NW - 1]) >> (t & 63)) & 1ull;
  }
  SFL_FN int any() const { return NW == 1 ? w[0] != 0ull : (w[0] | w[NW - 1]) != 0ull; }
  SFL_FN int popc() const { return NW == 1 ? popc64(w[0]) : popc64(w[0]) + popc64(w[NW - 1]); }
  // lowest train of the set, removed from it: word 0 first (train-handle order)
  SFL_FN int pop() {
    if (NW == 1 || w[0]) { const int t = ffs64(w[0]); w[0] &= w[0] - 1; return t; }
    const int t = 64 + ffs64(w[NW - 1]); w[NW - 1] &= w[NW - 1] - 1; return t;
  }
  // the set is all of trains 0..T-1
  SFL_FN int all(int T) const {
    if (NW == 1) return w[0] == (T >= 64 ? ~0ull : ((1ull << T) - 1ull));
    return w[0] == ~0ull && w[NW - 1] == (T >= 128 ? ~0ull : ((1ull << (T - 64)) - 1ull));
  }
  SFL_FN TSet andnot(const TSet &o) const { TSet r; r.w[0] = w[0] & ~o.w[0]; if (NW > 1) r.w[NW - 1] = w[NW - 1] & ~o.w[NW - 1]; return r; }
  SFL_FN int operator==(const TSet &o) const { return NW == 1 ? w[0] == o.w[0] : (w[0] == o.w[0]) & (w[NW - 1] == o.w[NW - 1]); }
};

// ------------------------------------------------------------------------------------------------ device views
// read-only map table: loads go through the non-coherent path (LDG.CONSTANT, L1-resident across the launch)
template <class T> struct RO {
  const T *p;
  SFL_FN T operator[](size_t i) const { return ldg(p + i); }
};

struct DevMap {            // map constants (device pointers)
  int H, W, Hp, Wp, S, NP, NA, T, NT, max_episode_steps, a_max, pad0;
  RO<uint16_t> move;           // [Hp*Wp*4] per (cell, heading): 3 bits per RailEnvAction (valid | new heading << 1), bit 15 = rail cell
  RO<int16_t> cell_switch;     // [Hp*Wp]
  RO<int4> sw;                 // [S]  {P, A, port0, act0}
  RO<int4> port;               // [NP] {neighbour port, distance to it, forced-path port of this port inside its switch or -1, switch}
  RO<int4> pexit;              // [NP] exits of an in-port: {n, e0, e1, e2}, e = action | out_local << 4 | move << 8
  RO<int4> act;                // [NA] {in_local, out_local, move, 0}
  RO<int4> train0;             // [T]  {init_cell, init_dir, target_cell, tgt_index}   (padded cell ids)
  RO<int4> train1;             // [T]  {ed, la, first_port, first_dist}
  RO<int> init_delay;          // [T]
  RO<int> dist;                // [NT][Hp*Wp][4]
  RO<int8_t> qinit;            // [NP*NT]  -1 | action | final<<4
};

struct Layout {            // byte offsets inside one env block
  int T, S, NP, NT, a_max, q_cap, q_stride, pend_cap;
  unsigned off_tra, off_trb, off_pend, off_sem, off_rewards, off_sws, off_q;
  unsigned off_rng;          // the reference's random stream (Pcg, SFL_RNG_REFERENCE), right after the header; 0: Philox
  unsigned long long env_stride;
};

// The header at the start of every env block.  It holds word 0 of the four train sets; with NW = 2 (T > 64) word 1 of
// each follows the header (Layout: zero bytes when T <= 64), in the order of the HM_* indices below.
struct EnvHdr {
  int elapsed, episode, step_counter, num_malf;
  int terminated, truncated, need_reset, halted;
  int err, q_rows, pending_fin, cur_dec;
  int act_cursor, ev_cursor, n_dec_logged, n_tick_logged;
  int n_ep_logged, q_init_on, aborted, cur_train;     // cur_train: SFL_MODE_STEP, the train whose decision waits for the host (-1: none)
  unsigned long long active_mask, malf_prev_mask, at_dest_mask, done_mask;
  unsigned long long decisions, ticks, train_ticks;
  double cum_reward;
  int last_next_sw;                    // "next_switch" of the most recent decision (SFL_MODE_STEP)
  int eps_tag;                         // epsilon-greedy draw cache: pair of decisions (step_counter >> 1) the words below belong to
  unsigned eps_z, eps_w;               //   words 2 and 3 of that pair's Philox block (the odd decision of the pair uses them)
  unsigned long long forced_stops, stop_actions, arrived_trains;     // lifetime statistics (sfl_env_counters)
  int dec_t, dec_go;                   // drain loop of the shared-table kernels: the train whose decision is next / whether there is one
  unsigned long long ph[6], ph_t0;      // phase clock (full kernel, sfl_set_phase_clock): cycles per phase, start of the running one
};

// Per-train records (16 bytes each, one vector load per phase):
//   TrA {pos, dir | state<<8 | saved<<16 | prev_act<<24, plan (4 bits per entry, head lowest) | plan_len<<16, malf (u16) | next_port<<16}
//   TrB {prev_port (u16) | source_port<<16 (0xFFFF = none), act_switch (u16) | pend_n<<16, last_delay, stop_tick}
//   stop_tick: the last tick of the episode the train ended STOPPED or MALFUNCTION (SFL_NO_STOP: none yet; see t0_eff)
// Per-switch record SwS {interactions, 0, eps_pow (f64) = epsilon_decay_rate ** interactions}.
// Pending update (distr_q.py:340-342): {key, next_sw | prev_sw<<12 | action<<24}; part of the tail (decision phase only).
// Semaphore record (rail_network.py:133 [train, in/out, dir, t0, t1]): {t0, t1 - t0, train (-1 = absent), type} -- start
// as written and LENGTH of the window; the window starts at t0_eff, the start with extend_semaphores applied.
struct SwS { int ninter, pad; double eps_pow; };
enum { HM_ACTIVE = 0, HM_MALF = 1, HM_DEST = 2, HM_DONE = 3 };   // the header's train sets: active, malf_prev, at_dest, done

struct RunArgs {           // per-launch arguments
  int mode, max_ticks, n_envs, trace_sem;
  int dec_cap, tick_cap, ep_cap, act_cap, ev_cap, max_steps, q_init_on, phase_clock;
  unsigned hot_bytes, env_smem, tail_hot, pad2;
  char *state;
  const sfl_hparams *hp;
  sfl_env_counters *counters;
  sfl_dec_rec *trace_dec; sfl_tick_rec *trace_tick; int4 *trace_sem_buf;
  sfl_ep_rec *ep_log; int *ep_delay;
  sfl_step_rec *step_out;
  double *sq_q; long long *sq_d; int *sq_c;           // shared-table mode (null otherwise): table, delta sums (2^-24), delta counts
  const int8_t *replay_act; const int *replay_ev;     // ev: [env][ev_cap][3] = (tick, train, duration), tick-sorted, tick<0 ends
  const double *eval_q;                               // evaluation contexts (EVQ kernels): the one read-only table; null otherwise
};

// Map constants, env-block layout and launch arguments travel as ONE __grid_constant__ kernel parameter (constant bank,
// the same operand cost as __constant__ symbols) -- so contexts are independent of each other: any stream, any device,
// several maps in flight at once.  Device functions receive it as `K`; c_m / c_L / c_ra name its three parts.
struct KArgs { DevMap m; Layout L; RunArgs ra; };
#define SFL_K const KArgs &K
#define c_m (K.m)
#define c_L (K.L)
#define c_ra (K.ra)

#if SFL_DEV
extern __shared__ __align__(16) char g_smem[];     // the CTA's dynamic shared memory
typedef unsigned hot_t;                            // staged env block: byte offset inside g_smem (32-bit LDS/STS addressing)
SFL_FN char *hot_ptr(hot_t o) { return g_smem + o; }
#else
typedef char *hot_t;
SFL_FN char *hot_ptr(hot_t o) { return o; }
#endif

// TH ("tail hot"): semaphores, rewards and per-switch records are part of the staged block; else they stay in HBM / L2
// SQ ("shared Q"): the shared-table extension; a compile-time variant, because even an untaken runtime branch in the
// Q-row functions cost the private-table kernels 20-25 % on large maps (registers / code size at 72 registers)
template <bool TH, bool SQ_ = false> struct EnvT {
  static const bool SQ = SQ_;
  static const bool EVQ = false;           // EnvEval: greedy decisions read the evaluation table
  static const bool HOT_TAIL = TH;
  static const int NW = 1;                 // 64-bit words per train set (EnvW: 2)
  const KArgs *kp;         // the launch's parameter block (methods below read the layout through it)
  hot_t hot;               // staged copy of the first hot_bytes of the env block (the env block itself on the host build)
  char *gb;                // the env block in HBM
  SFL_FN EnvHdr *h() const { return (EnvHdr *)hot_ptr(hot); }
  SFL_FN int4 *tra() const { return (int4 *)(hot_ptr(hot) + kp->L.off_tra); }
  SFL_FN int4 *trb() const { return (int4 *)(hot_ptr(hot) + kp->L.off_trb); }
  SFL_FN char *tail() const { return TH ? hot_ptr(hot) : gb; }
  SFL_FN int2 *pend() const { return (int2 *)(tail() + kp->L.off_pend); }
  SFL_FN int4 *sem() const { return (int4 *)(tail() + kp->L.off_sem); }
  SFL_FN int *rewards() const { return (int *)(tail() + kp->L.off_rewards); }
  SFL_FN SwS *sws() const { return (SwS *)(tail() + kp->L.off_sws); }
  SFL_FN double *q() const { return (double *)(gb + kp->L.off_q); }
  // Who holds the record of port p (-1: nobody).  When the semaphore table stays in HBM (large maps) a byte mirror of
  // the holders lives in shared memory: "is there a record / is it mine / is its holder stopped" -- most of what the
  // decision and the per-tick semaphore phases ask -- is then answered without touching global memory.
  hot_t own;
  SFL_FN uint8_t *own_ptr() const { return (uint8_t *)hot_ptr(own); }
  SFL_FN int owner(int p) const { return TH ? sem()[p].z : (int)(int8_t)own_ptr()[p]; }
  SFL_FN void sem_put(int p, int4 r) const { sem()[p] = r; if (!TH) own_ptr()[p] = (uint8_t)r.z; }
  SFL_FN void sem_drop(int p) const { sem()[p].z = -1; if (!TH) own_ptr()[p] = 0xFFu; }
  SFL_FN int stop_tick(int t) const { return trb()[t].w; }
  // header train set m (HM_*): word 0 in EnvHdr, word 1 (EnvW) right after it
  SFL_FN unsigned long long &hw0(int m) const {
    EnvHdr *x = h();
    return m == HM_ACTIVE ? x->active_mask : m == HM_MALF ? x->malf_prev_mask : m == HM_DEST ? x->at_dest_mask : x->done_mask;
  }
  SFL_FN unsigned long long *hw1(int m) const { return (unsigned long long *)(hot_ptr(hot) + sizeof(EnvHdr)) + m; }
};
// the environment of a map with more than 64 trains: two words per train set.  A type of its own rather than a third
// template argument of EnvT, so that the types -- and the out-of-line callees named after them -- of the one-word
// kernels stay exactly what they were
template <bool TH, bool SQ_ = false> struct EnvW : EnvT<TH, SQ_> { static const int NW = 2; };
// EVQ ("evaluation table"): the environment of an evaluation context (sfl_config.eval_q), which has no Q region of its own;
// its greedy decisions probe the one read-only table of the launch (eval_action).  A wrapper type, for the same reason as EnvW
template <class Base> struct EnvEval : Base { static const bool EVQ = true; };
template <bool TH, bool SQ, int NW, bool EVQ = false> struct EnvOf { typedef EnvT<TH, SQ> type; };
template <bool TH, bool SQ> struct EnvOf<TH, SQ, 2, false> { typedef EnvW<TH, SQ> type; };
template <bool TH, int NW> struct EnvOf<TH, false, NW, true> { typedef EnvEval<typename EnvOf<TH, false, NW>::type> type; };

// the header's train sets as TSet<Env::NW>
template <class Env> SFL_FN TSet<Env::NW> tset(const Env &e, int m) {
  TSet<Env::NW> s; s.w[0] = e.hw0(m); if (Env::NW > 1) s.w[Env::NW - 1] = *e.hw1(m); return s;
}
template <class Env> SFL_FN void tset_put(const Env &e, int m, const TSet<Env::NW> &s) { e.hw0(m) = s.w[0]; if (Env::NW > 1) *e.hw1(m) = s.w[Env::NW - 1]; }
template <class Env> SFL_FN int tset_any(const Env &e, int m) { return Env::NW == 1 ? e.hw0(m) != 0ull : (e.hw0(m) | *e.hw1(m)) != 0ull; }
template <class Env> SFL_FN int tset_pop(const Env &e, int m) { TSet<Env::NW> s = tset(e, m); const int t = s.pop(); tset_put(e, m, s); return t; }
template <class Env> SFL_FN void tset_add(const Env &e, int m, int t) {
  if (Env::NW > 1 && t >= 64) *e.hw1(m) |= 1ull << (t & 63); else e.hw0(m) |= 1ull << t;
}



// per-group exchange area of one tick (shared memory on the device), sized by T; one 32-bit base, layout
// [tmp 16T | rng 16T | occ T | blk T]:
//   tmp  {src, dst, expected cell, new heading | preprocessed action<<8 | popped action<<16 | flags<<24}
//   rng  the 16 stage-1 malfunction bytes of the current 16-tick block (one Philox call per train and block);
//        replay injects recorded events instead of drawing, so `inj` (durations injected this tick) aliases it
//   occ  train standing on my destination cell, or -1;   blk  movement blocked
struct Scratch {
  const KArgs *kp;
  hot_t base;
  SFL_FN int4 *tmp() const { return (int4 *)hot_ptr(base); }
  SFL_FN int4 *rng() const { return (int4 *)(hot_ptr(base) + 16 * kp->L.T); }
  SFL_FN int *inj() const { return (int *)(hot_ptr(base) + 16 * kp->L.T); }
  SFL_FN int8_t *occ() const { return (int8_t *)(hot_ptr(base) + 32 * kp->L.T); }
  SFL_FN uint8_t *blk() const { return (uint8_t *)(hot_ptr(base) + 33 * kp->L.T); }
};
#if SFL_DEV
__host__
#endif
SFL_FN unsigned scratch_bytes(int T) { return (unsigned)(32 * T + ((2 * T + 15) / 16) * 16); }

// the environment's hyper-parameters (staged next to the hot state on the device): a 32-bit handle, not a pointer
struct Hp {
  hot_t o;
  SFL_FN const sfl_hparams *operator->() const { return (const sfl_hparams *)hot_ptr(o); }
};

// phase clock (instrumented runs of the full kernel only): the first lane charges the cycles since the last mark to a phase
#if SFL_DEV
SFL_FN unsigned long long sm_clock() { return (unsigned long long)clock64(); }
#else
SFL_FN unsigned long long sm_clock() { return 0ull; }
#endif
enum { PH_TICK = 0, PH_OBSERVE = 1, PH_ACT = 2, PH_APPLY = 3, PH_UPDATE = 4, PH_RESET = 5 };
#define SFL_PHASE_START(h) do { if (TRACE && c_ra.phase_clock) (h)->ph_t0 = sm_clock(); } while (0)
#define SFL_PHASE_MARK(h, i) do { if (TRACE && c_ra.phase_clock) { const unsigned long long t_ = sm_clock(); (h)->ph[i] += t_ - (h)->ph_t0; (h)->ph_t0 = t_; } } while (0)

// ------------------------------------------------------------------------------------------------ kernel kinds
// The run mode is a compile-time property of the two production kernels (learn, greedy): with the mode a runtime
// value the replay / step / trace paths stayed in the hot kernels and cost the large-map kernels 8 % (registers and
// instruction fetch at 72 registers).  The third kind carries everything: any mode, traces, the step protocol.
enum { K_LEARN = 0, K_GREEDY = 1, K_FULL = 2 };
template <int KIND> SFL_FN int run_mode(SFL_K) { return KIND == K_LEARN ? (int)SFL_MODE_LEARN : KIND == K_GREEDY ? (int)SFL_MODE_GREEDY : c_ra.mode; }

// ------------------------------------------------------------------------------------------------ Philox4x32-10
struct U4 { unsigned x, y, z, w; };
SFL_FN unsigned mulhi32(unsigned a, unsigned b) { return (unsigned)(((unsigned long long)a * b) >> 32); }
SFL_FN U4 philox4x32(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1) {
  SFL_NU
  for (int i = 0; i < 10; i++) {
    unsigned h0 = mulhi32(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    unsigned h1 = mulhi32(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    unsigned n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  U4 r = {c0, c1, c2, c3};
  return r;
}

// ------------------------------------------------------------------------------------------------ the reference's stream
// SFL_RNG_REFERENCE: numpy's Generator(PCG64) exactly as distr_q.py draws from it -- rng = np.random.default_rng(seed) at
// the start of learn() (:269); per decision rng.random() < epsilon; on exploration Discrete.seed(int(rng.integers(0,
// 2**31 - 1))) and Discrete.sample(mask) = Generator(PCG64(SeedSequence(sd))).choice(where(mask)) (:315-317).  Integer
// arithmetic only (numpy's bit_generator.pyx, _pcg64.pyx, pcg64.h, distributions.c).
struct Pcg {                 // numpy's pcg64_state: 128-bit state and increment, the carried half-word of next_uint32
  unsigned long long s_hi, s_lo, i_hi, i_lo;
  unsigned has32, u32, pad0, pad1;
};
#define SFL_PCG_BYTES 48

SFL_FN void pcg_step(Pcg &g) {        // state = state * 0x2360ED051FC65DA44385DF649FCCF645 + inc  (mod 2^128)
  const unsigned long long M_HI = 0x2360ED051FC65DA4ull, M_LO = 0x4385DF649FCCF645ull;
  const unsigned long long lo = g.s_lo * M_LO;
  const unsigned long long hi = mulhi64(g.s_lo, M_LO) + g.s_lo * M_HI + g.s_hi * M_LO;
  g.s_lo = lo + g.i_lo;
  g.s_hi = hi + g.i_hi + (g.s_lo < lo ? 1ull : 0ull);
}
SFL_FN unsigned long long pcg_next64(Pcg &g) {     // step, then XSL-RR of the new state
  pcg_step(g);
  const unsigned long long x = g.s_hi ^ g.s_lo;
  const unsigned r = (unsigned)(g.s_hi >> 58);
  return (x >> r) | (x << ((64u - r) & 63u));
}
SFL_FN double pcg_double(Pcg &g) { return (double)(pcg_next64(g) >> 11) * (1.0 / 9007199254740992.0); }   // random()
SFL_FN unsigned pcg_next32(Pcg &g) {             // a 64-bit draw serves two calls: low half now, high half carried
  if (g.has32) { g.has32 = 0; return g.u32; }
  const unsigned long long v = pcg_next64(g);
  g.has32 = 1; g.u32 = (unsigned)(v >> 32);
  return (unsigned)v;
}
// Generator.integers(0, ex) for 1 <= ex <= 2^32: random_bounded_uint64_fill, Lemire's method on 32-bit draws
SFL_FN unsigned pcg_bounded(Pcg &g, unsigned long long ex) {
  if (ex <= 1ull) return 0u;                     // one value: no draw
  if (ex == 0x100000000ull) return pcg_next32(g);
  const unsigned e = (unsigned)ex;
  unsigned long long m = (unsigned long long)pcg_next32(g) * e;
  if ((unsigned)m < e) {
    const unsigned threshold = (0u - e) % e;     // (2^32 - ex) mod ex
    SFL_NU
    while ((unsigned)m < threshold) m = (unsigned long long)pcg_next32(g) * e;
  }
  return (unsigned)(m >> 32);
}
// PCG64(SeedSequence(seed)) = np.random.default_rng(seed): the seed's little-endian 32-bit words (one below 2^32) hashed into
// a 4-word pool, cross-mixed, expanded to 8 words = 4 uint64 {initstate hi, lo, initseq hi, lo}; then pcg's srandom
SFL_FN unsigned ss_hashmix(unsigned v, unsigned &hc) { v ^= hc; hc *= 0x931e8875u; v *= hc; return v ^ (v >> 16); }
SFL_FN unsigned ss_mix(unsigned x, unsigned y) { const unsigned r = 0xca01f9ddu * x - 0x4973f715u * y; return r ^ (r >> 16); }
SFL_FN Pcg pcg_seed(unsigned long long seed) {
  unsigned hc = 0x43b0d7e5u, pool[4], w[8];
  pool[0] = ss_hashmix((unsigned)seed, hc);
  pool[1] = ss_hashmix((unsigned)(seed >> 32), hc);   // a seed below 2^32 has one word: the pool is padded with 0 alike
  pool[2] = ss_hashmix(0u, hc);
  pool[3] = ss_hashmix(0u, hc);
  SFL_UA
  for (int s = 0; s < 4; s++) {
    SFL_UA
    for (int d = 0; d < 4; d++) if (s != d) pool[d] = ss_mix(pool[d], ss_hashmix(pool[s], hc));
  }
  hc = 0x8b51f9ddu;
  SFL_UA
  for (int i = 0; i < 8; i++) { unsigned v = pool[i & 3] ^ hc; hc *= 0x58f38dedu; v *= hc; w[i] = v ^ (v >> 16); }
  const unsigned long long v0 = w[0] | (unsigned long long)w[1] << 32, v1 = w[2] | (unsigned long long)w[3] << 32;
  const unsigned long long v2 = w[4] | (unsigned long long)w[5] << 32, v3 = w[6] | (unsigned long long)w[7] << 32;
  Pcg g;
  g.s_hi = 0ull; g.s_lo = 0ull; g.i_hi = (v2 << 1) | (v3 >> 63); g.i_lo = (v3 << 1) | 1ull;     // inc = initseq << 1 | 1
  g.has32 = 0u; g.u32 = 0u; g.pad0 = 0u; g.pad1 = 0u;
  pcg_step(g);
  const unsigned long long lo = g.s_lo + v1;                                                     // state += initstate
  g.s_hi += v0 + (lo < v1 ? 1ull : 0ull); g.s_lo = lo;
  pcg_step(g);
  return g;
}

// decay ** n rounded to nearest: binary exponentiation in double-double (relative error about 2^-100 for n < 2^31, far
// inside half an ulp), the pair rounded by its renormalisation.  The pairs are kept scaled by exact powers of two (2^-er,
// 2^-eb) so that their low words never go subnormal; decay is in [0, 1].
SFL_FN void dd_mul(double &ah, double &al, double bh, double bl) {
  const double p = dmul(ah, bh);
  const double t = dadd(dfma(ah, bh, -p), dadd(dmul(ah, bl), dmul(al, bh)));
  const double s = dadd(p, t);
  al = dadd(t, -dadd(s, -p)); ah = s;
}
SFL_FN void dd_rescale(double &h, double &l, long long &e) {
  if (h < 0x1p-400 && e < 4000) { h = dmul(h, 0x1p400); l = dmul(l, 0x1p400); e += 400; }
}
SFL_FN double pow_dd(double b, int n) {
  if (b == 0.0) return n == 0 ? 1.0 : 0.0;
  double rh = 1.0, rl = 0.0, bh = b, bl = 0.0;
  long long er = 0, eb = 0;
  SFL_NU
  for (; n > 0; n >>= 1) {
    if (n & 1) { dd_mul(rh, rl, bh, bl); er += eb; dd_rescale(rh, rl, er); }
    if (n > 1) { dd_mul(bh, bl, bh, bl); eb = eb < 4000 ? 2 * eb : eb; dd_rescale(bh, bl, eb); }
  }
  return er >= 4000 ? 0.0 : ldexp(rh, -(int)er);
}
// distr_q.py:315 `rng.random() < epsilon * epsilon_decay_rate ** n`.  eps_pow is the kernel's running product of the decay
// (SwS.eps_pow: one rounding per interaction, relative error below (n + 1) 2^-53; pow's is below one ulp): only a draw
// inside that margin of the product recomputes the power exactly -- practically never, but it makes the comparison exact.
SFL_FN int eps_explore(double u, double epsilon, double decay, int n, double eps_pow) {
  const double eps = dmul(epsilon, eps_pow);
  const double tol = dadd(dmul(eps, (double)(n + 4) * 0x1p-52), 0x1p-1000);
  const double gap = dadd(u, -eps);
  if (gap > tol || -gap > tol) return u < eps;
  return u < dmul(epsilon, pow_dd(decay, n));
}
// the exploring branch (distr_q.py:316-317): a new generator from the learner's stream, its choice among the allowed actions
SFL_FN int pcg_explore_action(Pcg &g, int mask) {
  Pcg x = pcg_seed(pcg_bounded(g, 0x7FFFFFFFull));
  unsigned mm = (unsigned)mask;
  SFL_NU
  for (unsigned pick = pcg_bounded(x, (unsigned long long)popc32(mm)); pick > 0; pick--) mm &= mm - 1;
  return ffs64(mm);
}

// ------------------------------------------------------------------------------------------------ flatland's malfunction stream
// SFL_MALF_REFERENCE: numpy's legacy RandomState (MT19937) exactly as flatland draws from it.  rail_env.reset(random_seed=
// seed) creates np_random = RandomState(seed) at every episode (switch_env.py:99); every tick 1 .. max_episode_steps, for
// every train in handle order, ParamMalfunctionGen.generate draws rand() < 1 - exp(-rate) and, on a hit, randint(min,
// max + 1) + 1 steps (SURVEY.md Appendix B, F5).  No draw depends on the actions: the schedule is a function of (seed, rate,
// min, max, T, max_episode_steps), the same in every episode.  Integer arithmetic only (numpy's mt19937.c, _mt19937.pyx
// _legacy_seeding, distributions.c random_bounded_uint64_fill).  The 624 state words and their tempered outputs live in
// memory shared by the G lanes of a group: the group twists together, and every lane walks the same draws (broadcast reads).
#define SFL_MT_N 624
#define SFL_MT_M 397
SFL_FN unsigned mt_temper(unsigned y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9D2C5680u;
  y ^= (y << 15) & 0xEFC60000u;
  return y ^ (y >> 18);
}
// RandomState(seed): init_genrand; numpy accepts only 0 <= seed < 2^32 (returns 0 for any other seed).  The one place that
// turns a seed into the generator's key.
template <int G> SFL_FN int mt_seed(unsigned *key, unsigned long long seed, const Grp<G> &g) {
  if (seed >> 32) return 0;
  if (g.gl == 0) {
    unsigned s = (unsigned)seed;
    SFL_NU
    for (int i = 0; i < SFL_MT_N; i++) { key[i] = s; s = 1812433253u * (s ^ (s >> 30)) + (unsigned)(i + 1); }
  }
  g.sync();
  return 1;
}
// mt19937_gen, G words at a time: new key[i] needs old key[i], old key[i + 1] (new key[0] for i = N - 1) and key[i + M]
// (old) below N - M, key[i - (N - M)] (new: an earlier chunk) from there on -- all read before the chunk writes.  Then
// every word is tempered into out[].
template <int G> SFL_FN void mt_twist(unsigned *key, unsigned *out, const Grp<G> &g) {
  SFL_NU
  for (int base = 0; base < SFL_MT_N; base += G) {
    const int i = base + g.gl;
    unsigned v = 0u;
    if (i < SFL_MT_N) {
      const unsigned y = (key[i] & 0x80000000u) | (key[i + 1 == SFL_MT_N ? 0 : i + 1] & 0x7FFFFFFFu);
      v = key[i < SFL_MT_N - SFL_MT_M ? i + SFL_MT_M : i - (SFL_MT_N - SFL_MT_M)] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908B0DFu);
    }
    g.sync();
    if (i < SFL_MT_N) key[i] = v;
    g.sync();
  }
  for (int i = g.gl; i < SFL_MT_N; i += G) out[i] = mt_temper(key[i]);
  g.sync();
}
template <int G> SFL_FN unsigned mt_next(unsigned *key, unsigned *out, int &pos, const Grp<G> &g) {
  if (pos == SFL_MT_N) { mt_twist(key, out, g); pos = 0; }
  return out[pos++];
}
// RandomState.randint(lo, lo + rng + 1) - lo: masked rejection on 32-bit words, mask = the smallest 2^k - 1 >= rng; rng = 0
// consumes no word
template <int G> SFL_FN unsigned mt_masked(unsigned *key, unsigned *out, int &pos, const Grp<G> &g, unsigned rng) {
  if (!rng) return 0u;
  unsigned mask = rng;
  mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
  unsigned v;
  SFL_NU
  do v = mt_next(key, out, pos, g) & mask; while (v > rng);
  return v;
}
// One environment's schedule: every drawn event (tick, train, duration) in tick order into ev[0 .. ev_cap), -1 after the
// last when there is room.  rand() = ((a >> 5) 2^26 + (b >> 6)) 2^-53 < p is compared in the integers: k < hit_below =
// ceil(p 2^53).  Returns the number of events (also those beyond ev_cap), or -1 for a seed RandomState refuses.
template <int G> SFL_FN int malf_schedule_env(unsigned long long seed, unsigned long long hit_below, int lo, int hi, int T, int steps,
                                              int *ev, int ev_cap, unsigned *key, unsigned *out, const Grp<G> &g) {
  if (!mt_seed(key, seed, g)) return -1;
  int n = 0, pos = SFL_MT_N;
  const unsigned rng = (unsigned)hi - (unsigned)lo;
  SFL_NU
  for (int tick = 1; hit_below && tick <= steps; tick++) {
    SFL_NU
    for (int t = 0; t < T; t++) {
      const unsigned a = mt_next(key, out, pos, g), b = mt_next(key, out, pos, g);
      if ((((unsigned long long)(a >> 5) << 26) | (b >> 6)) >= hit_below) continue;
      const int dur = lo + (int)mt_masked(key, out, pos, g, rng) + 1;
      if (g.gl == 0 && n < ev_cap) { ev[3 * n] = tick; ev[3 * n + 1] = t; ev[3 * n + 2] = dur; }
      n++;
    }
  }
  if (g.gl == 0 && n < ev_cap) ev[3 * n] = -1;
  return n;
}

// ------------------------------------------------------------------------------------------------ F1
// flatland rail.check_action_on_agent (SURVEY.md Appendix B; called switch_env.py:325,450,545, reward_func.py:49)
// through the per-(cell, heading) move table built in sfl_create: entry bits [3a, 3a+3) = valid | new heading << 1
// for RailEnvAction a.  sfl_create rejects maps with a transition into a non-rail cell, so "new cell is rail"
// (the reference's new_cell_valid) is implied by a valid transition.
struct Mv { int cell, dir, valid; };
SFL_FN unsigned mv_entry(SFL_K, int cell, int dir) { return c_m.move[(size_t)cell * 4 + dir]; }
SFL_FN int mv_valid(unsigned e, int action) { return (e >> (3 * action)) & 1; }
SFL_FN Mv mv_apply(SFL_K, unsigned e, int action, int cell) {
  unsigned f = (e >> (3 * action)) & 7u;
  int nd = (int)(f >> 1);
  int delta = (nd & 1) ? (2 - nd) : (nd - 1) * c_m.Wp;
  Mv r;
  r.cell = (e & 0x8000u) ? cell + delta : cell;   // a non-rail cell (only reachable by projecting invalid plans) stays put
  r.dir = nd; r.valid = (int)(f & 1u);
  return r;
}
SFL_FN Mv check_action(SFL_K, int action, int cell, int dir) { return mv_apply(K, mv_entry(K, cell, dir), action, cell); }

SFL_FN int is_moving(int a) { return a >= A_LEFT && a <= A_RIGHT; }

// ------------------------------------------------------------------------------------------------ E4
// extend_semaphores (rail_network.py:229-244) slides every record held by a train that ends a tick STOPPED or MALFUNCTION
// to start at that tick, keeping its length.  The kernel stores only the tick, in the holder's TrB.stop_tick, and every
// reader of a window start takes the later of the two.  Exact, because every writer of a record sets t0 to the current
// tick (transition_semaphore: now; the departure booking: ed - 2 == now; the MALFUNCTION booking: now) and no stamp is
// later than the current tick: a record written after its holder's last stop has t0 >= stop_tick, one written before it
// was slid to exactly that tick.  The reset bookings' t0 = ed - 2 precedes every stop of their holder, and may be
// negative (ed < 2), so the stamp of a train that has not stopped this episode is SFL_NO_STOP, below every t0.
#define SFL_NO_STOP (-0x7FFFFFFF - 1)
SFL_FN int t0_eff(int t0, int stop_tick) { return t0 > stop_tick ? t0 : stop_tick; }
// observer.py:44-151 check_port_blocked.  Every writer of a semaphore record stores dir == map_direction(port)
// (rail_network.py:243,327,337,372,382,396,408; switch_env.py:382,566), so the eight clauses reduce to:
//   rule_next: 'out' -> blocked, 'in' -> blocked iff holder MALFUNCTION;  rule_out: 'in' -> blocked, 'out' -> iff MALFUNCTION.
template <class Env>
SFL_FN int tr_state(Env e, int t) { return (e.tra()[t].y >> 8) & 0xFF; }
template <class Env>
SFL_FN int rule_port(Env e, int port, int me, int now, int blocking_type) {
  int4 r;
  int stamp;
  if (Env::HOT_TAIL) {                                                        // staged table: one shared-memory load
    r = e.sem()[port];
    if (r.z < 0 || r.z == me) return 0;
    stamp = e.stop_tick(r.z);
  } else {                                                              // table in HBM: ask the holder mirror first
    const int holder = e.owner(port);
    if (holder < 0 || holder == me) return 0;
    r = e.sem()[port];
    stamp = e.stop_tick(holder);                                        // shared memory: in flight with the record's load
  }
  if (r.x > now || t0_eff(r.x, stamp) + r.y < now) return 0;           // t0_eff > now iff t0 > now: no stamp is later than now
  if (r.w == blocking_type) return 1;
  return tr_state(e, r.z) == ST_MALF;
}
template <class Env>
SFL_FN int port_blocked(Env e, int next_port, int out_port, int me, int now) {
  if (next_port >= 0) {
    if (rule_port(e, next_port, me, now, SEM_OUT)) return 1;
    return rule_port(e, out_port, me, now, SEM_IN);
  }
  return rule_port(e, out_port, me, now, SEM_OUT);
}

// ------------------------------------------------------------------------------------------------ Q table (Q2, Q6)
// Row = [key+1 as u64 bits | A_max doubles]; open addressing, linear probing, no deletion.  A row is created
// exactly where the reference's __check_entry (distr_q.py:47-57) would insert a dict entry, so the exported
// key set equals the reference's.
// insertion of a new row (rare once the tables are warm): out of line
template <class Env>
SFL_RARE void q_insert(SFL_K, Env e, const Hp hp, unsigned key, double *row) {
  *(unsigned long long *)row = (unsigned long long)key + 1ull;
  e.h()->q_rows++;
  unsigned per_port = (unsigned)(c_L.NT * 48);
  int port = (int)(key / per_port);
  int A = c_m.sw[c_m.port[port].w].y;
  double dq = hp->default_q;
  SFL_NU
  for (int a = 0; a < A; a++) row[1 + a] = dq;
  if (c_ra.q_init_on) {                                   // distr_q.py:81-181 (lazy: same values, created on first touch)
    unsigned rem = key - (unsigned)port * per_port;
    int tgt = (int)(rem / 48u), semb = (int)((rem % 48u) / 3u);
    int qi = c_m.qinit[port * c_L.NT + tgt];
    if (qi >= 0 && semb != 0) row[1 + (qi & 15)] = (qi & 16) ? 1000.0 : 500.0;
  }
}

template <class Env>
SFL_NI double *q_row(SFL_K, Env e, const Hp hp, unsigned key) {
  if (Env::SQ) return c_ra.sq_q + (size_t)key * c_L.a_max;              // shared-table mode: dense, initialised by the host
  unsigned mask = (unsigned)c_L.q_cap - 1u;
  unsigned i = (key * 2654435761u) >> 7;
  SFL_NU
  for (int probe = 0; probe < c_L.q_cap; probe++) {
    i &= mask;
    double *row = e.q() + (size_t)i * c_L.q_stride;
    unsigned long long k = *(unsigned long long *)row;
    if (k == (unsigned long long)key + 1ull) return row + 1;
    if (k == 0ull) {
      if (e.h()->q_rows >= c_L.q_cap - 1) break;
      q_insert(K, e, hp, key, row);
      return row + 1;
    }
    i++;
  }
  e.h()->err |= SFL_ERR_Q_FULL;
  return e.q() + 1;     // keep running on row 0 (flagged)
}

// integer sums: the accumulated step does not depend on the order in which the environments arrive
#if SFL_DEV
SFL_FN void shared_add(long long *d, int *c, long long v) { atomicAdd((unsigned long long *)d, (unsigned long long)v); atomicAdd(c, 1); }
#else
SFL_FN void shared_add(long long *d, int *c, long long v) { *d += v; *c += 1; }
#endif

// lr_decay_rate ** n (distr_q.py:70-79) by binary exponentiation: at most 2 log2(n) roundings (~1e-15 relative, the
// parity bar off the shipped configs is 1e-12; every script uses rate 1.0, which is exact) and none of pow()'s code
SFL_FN double lr_pow(double rate, int n) {
  double r = 1.0, b = rate;
  SFL_NU
  for (; n > 0; n >>= 1) { if (n & 1) r = dmul(r, b); b = dmul(b, b); }
  return r;
}

// distr_q.py:441-447 (fp64, Python operator order, no FMA contraction):
//   bootstrap (successor switch differs): (1 - lr) * Q + lr * (reward + gamma * max_a' Q')    else: (1 - lr) * Q + lr * reward
SFL_FN double td_value(double q, double lr, double reward, double gamma, double mq, int bootstrap) {
  const double one_m = dadd(1.0, -lr);
  return bootstrap ? dadd(dmul(one_m, q), dmul(lr, dadd(reward, dmul(gamma, mq)))) : dadd(dmul(one_m, q), dmul(lr, reward));
}

// distr_q.py:419-447 update
template <class Env>
SFL_NI void q_update(SFL_K, Env e, const Hp hp, unsigned key, int action, double reward,
                     const double *next_row, int prev_sw, int next_sw) {
  double *row = q_row(K, e, hp, key);
  double lr = hp->lr;
  if (hp->lr_decay_rate != 1.0) lr = dmul(lr, lr_pow(hp->lr_decay_rate, e.sws()[prev_sw].ninter));
  const double q = row[action];
  double mq = 0.0;
  if (next_sw != prev_sw && next_row) {                          // distr_q.py:449-466 max_q ignores the mask; max_q(None) = 0
    int A = c_m.sw[next_sw].y;
    mq = next_row[0];
    SFL_NU
    for (int a = 1; a < A; a++) { const double v = next_row[a]; mq = v > mq ? v : mq; }
  }
  const double nq = td_value(q, lr, reward, hp->gamma, mq, next_sw != prev_sw);
  if (Env::SQ) {                                                         // shared table: propose the TD step, leave the table alone
    const size_t i = (size_t)key * c_L.a_max + action;
    shared_add(c_ra.sq_d + i, c_ra.sq_c + i, (long long)llrint((nq - q) * 16777216.0));
    return;
  }
  row[action] = nq;
}

// distr_q.py:468-490 max_action (Row: a plain pointer, or RO<double> for the evaluation table)
template <class Row> SFL_FN int max_action_of(const Row row, int A, int mask) {
  int best = 0, b2 = -1;                       // first maximum over all actions / over the allowed ones (np.argmax)
  double bv = row[0], b2v = 0.0;
  if (mask & 1) { b2 = 0; b2v = bv; }
  SFL_NU
  for (int a = 1; a < A; a++) {
    const double v = row[a];
    if (v > bv) { bv = v; best = a; }
    if (((mask >> a) & 1) && (b2 < 0 || v > b2v)) { b2v = v; b2 = a; }
  }
  return ((mask >> best) & 1) ? best : b2;
}
SFL_FN int max_action(const double *row, int A, int mask) { return max_action_of(row, A, mask); }

// EVQ: the greedy decision on the evaluation table -- the probe of q_row (same hash, linear probing) on the launch's one
// read-only table, loaded through the non-coherent path; nothing is inserted.  A missing row reads as the default row
// (default_q x A): max_action of A equal values is the lowest allowed action, the decision test() makes after inserting
// that row (distr_q.py:482 -> :56-57).  The table always has an empty slot (sfl_set_eval_table: rows < q_cap).
SFL_FN int eval_action(SFL_K, unsigned key, int A, int mask) {
  const unsigned qmask = (unsigned)c_L.q_cap - 1u;
  const unsigned long long want = (unsigned long long)key + 1ull;
  unsigned i = (key * 2654435761u) >> 7;
  SFL_NU
  for (int probe = 0; probe < c_L.q_cap; probe++) {
    i &= qmask;
    const double *row = c_ra.eval_q + (size_t)i * c_L.q_stride;
    const unsigned long long k = ldg((const unsigned long long *)row);
    if (k == want) { RO<double> r; r.p = row + 1; return max_action_of(r, A, mask); }
    if (k == 0ull) break;
    i++;
  }
  return ffs64((unsigned long long)((unsigned)mask & ((1u << A) - 1u)));
}

// ------------------------------------------------------------------------------------------------ E3
template <class Env>
SFL_FN void sem_delete_owned(SFL_K, Env e, int port, int h) {
  int4 sw = c_m.sw[c_m.port[port].w];
  SFL_NU
  for (int k = 0; k < sw.x; k++) {
    int p = sw.z + k;
    if (e.owner(p) == h) e.sem_drop(p);
  }
}

// rail_network.py:303-416 transition_semaphore, step by step.  Its window-start tests `t0 > now` read the stored t0: no stop
// stamp is later than now, so t0_eff(r) > now exactly when t0 > now.
template <class Env>
SFL_FN void transition_semaphore(SFL_K, Env e, int source, int out_port, int target, int h, int now, int st, int old_next, int old_prev) {
  if (st != ST_MALF) {                                                  // :315-323
    sem_delete_owned(K, e, old_next, h);
    if (old_prev >= 0) sem_delete_owned(K, e, old_prev, h);
  }
  if (Env::HOT_TAIL) {                                                        // staged table: load, test, store
    int4 r = e.sem()[out_port];                                           // :326-334
    if (r.z < 0) e.sem()[out_port] = make_int4(now, 3, h, SEM_OUT);
    else if (r.w == SEM_OUT || r.x > now) e.sem()[out_port] = make_int4(now, 3, h, r.w);
    int d_ot = c_m.port[out_port].y;
    r = e.sem()[target];                                                  // :336-344
    if (r.z < 0) e.sem()[target] = make_int4(now, d_ot + 1, h, SEM_IN);
    else if (r.w == SEM_IN || r.x > now) e.sem()[target] = make_int4(now, d_ot + 1, h, r.w);
    int unique = c_m.port[target].z;
    if (unique >= 0) {                                                    // :356 forced path through the next switch
      int4 up = c_m.port[unique];
      int far_port = up.x;
      if (unique != source && unique != out_port && unique != target) {   // :368-378
        r = e.sem()[unique];
        if (r.z < 0 || r.w == SEM_OUT || r.x > now) e.sem()[unique] = make_int4(now, d_ot + 1, h, SEM_OUT);
      }
      r = e.sem()[unique];                                                // :380-388 (the list == 'out' test is never true)
      if (r.z < 0 || r.x > now) e.sem()[unique] = make_int4(now, d_ot, h, SEM_OUT);
      if (far_port != source && far_port != out_port && far_port != unique) {   // :390-402
        r = e.sem()[far_port];
        if (r.z < 0 || r.w == SEM_IN || r.x > now) e.sem()[far_port] = make_int4(now, d_ot + up.y + 1, h, SEM_IN);
      }
    }
    if (target != source && target != out_port) {                         // :404-414 moving edge
      r = e.sem()[target];
      if (r.z < 0 || r.w == SEM_OUT || r.x > now) e.sem()[target] = make_int4(now, d_ot + 1, h, SEM_OUT);
    }
  } else {                                                              // table in HBM: the holder mirror answers "nobody" without a load
    int4 r;                                                             // :326-334
    if (e.owner(out_port) < 0) e.sem_put(out_port, make_int4(now, 3, h, SEM_OUT));
    else { r = e.sem()[out_port]; if (r.w == SEM_OUT || r.x > now) e.sem_put(out_port, make_int4(now, 3, h, r.w)); }
    int d_ot = c_m.port[out_port].y;
    if (e.owner(target) < 0) e.sem_put(target, make_int4(now, d_ot + 1, h, SEM_IN));            // :336-344
    else { r = e.sem()[target]; if (r.w == SEM_IN || r.x > now) e.sem_put(target, make_int4(now, d_ot + 1, h, r.w)); }
    int unique = c_m.port[target].z;
    if (unique >= 0) {                                                  // :356 forced path through the next switch
      int4 up = c_m.port[unique];
      int far_port = up.x;
      if (unique != source && unique != out_port && unique != target) { // :368-378
        r = e.sem()[unique];
        if (e.owner(unique) < 0 || r.w == SEM_OUT || r.x > now) e.sem_put(unique, make_int4(now, d_ot + 1, h, SEM_OUT));
      }
      r = e.sem()[unique];                                              // :380-388 (the list == 'out' test is never true)
      if (e.owner(unique) < 0 || r.x > now) e.sem_put(unique, make_int4(now, d_ot, h, SEM_OUT));
      if (far_port != source && far_port != out_port && far_port != unique) {   // :390-402
        r = e.sem()[far_port];
        if (e.owner(far_port) < 0 || r.w == SEM_IN || r.x > now) e.sem_put(far_port, make_int4(now, d_ot + up.y + 1, h, SEM_IN));
      }
    }
    if (target != source && target != out_port) {                       // :404-414 moving edge
      r = e.sem()[target];
      if (e.owner(target) < 0 || r.w == SEM_OUT || r.x > now) e.sem_put(target, make_int4(now, d_ot + 1, h, SEM_OUT));
    }
  }
}

// ------------------------------------------------------------------------------------------------ decision (first lane)
template <class Env>
SFL_FN int delay_at(SFL_K, Env e, int tgt_index, int cell, int dir, int now, int la) {
  int d = c_m.dist[((size_t)tgt_index * (c_m.Hp * c_m.Wp) + cell) * 4 + dir];
  if (d >= SFL_INF_DIST) { e.h()->err |= SFL_ERR_INF_DISTANCE; d = 0; }     // observer.py:35-36
  return now - la + d;                                                      // observer.py:41
}

// the tail of one iteration of distr_q.py:302-362 that must wait for the train ticks run inside env.step()
// (switch_env.py:648-649): arrival flush (:345-356), interaction counter (:362), truncation (switch_env.py:652-657)
template <int KIND, class Env>
SFL_FN void finish_decision(SFL_K, Env e, const Hp hp, int env_id) {
  const bool TRACE = KIND == K_FULL;
  const int mode = run_mode<KIND>(K);
  EnvHdr *h = e.h();
  SFL_PHASE_START(h);
  if (mode == SFL_MODE_LEARN || mode == SFL_MODE_REPLAY) {
    TSet<Env::NW> fresh = tset(e, HM_DONE).andnot(tset(e, HM_DEST));
    SFL_NU
    while (fresh.any()) {
      int t = fresh.pop();
      tset_add(e, HM_DEST, t);
      int4 b = e.trb()[t];
      int n = (b.y >> 16) & 0xFF;
      SFL_NU
      for (int i = 0; i < n; i++) {
        int2 pe = e.pend()[t * c_L.pend_cap + i];
        q_update(K, e, hp, (unsigned)pe.x, (pe.y >> 24) & 15, 1000.0, nullptr, (pe.y >> 12) & 0xFFF, -1);
      }
      b.y &= 0xFFFF;
      e.trb()[t] = b;
    }
    SwS *ss = e.sws() + h->pending_fin;
    ss->ninter++;
    ss->eps_pow = dmul(ss->eps_pow, hp->epsilon_decay_rate);
  }
  h->pending_fin = -1;
  SFL_PHASE_MARK(h, PH_UPDATE);
  if (h->step_counter > c_ra.max_steps) h->truncated = 1;
  if (TRACE) {
    if (c_ra.trace_dec && h->cur_dec >= 0 && h->cur_dec < c_ra.dec_cap) {
      sfl_dec_rec *rec = c_ra.trace_dec + (size_t)env_id * c_ra.dec_cap + h->cur_dec;
      rec->arrived = h->done_mask; rec->arrived_hi = Env::NW > 1 ? *e.hw1(HM_DONE) : 0ull;
      rec->done = h->terminated | (h->truncated << 1);
      if (c_ra.trace_sem_buf) {
        int4 *dst = c_ra.trace_sem_buf + ((size_t)env_id * c_ra.dec_cap + h->cur_dec) * c_L.NP;
        SFL_NU
        for (int p = 0; p < c_L.NP; p++) {                                                       // traced as {t0, t1, train, type}
          int4 r = e.sem()[p];
          if (r.z >= 0) r.x = t0_eff(r.x, e.stop_tick(r.z));
          r.y += r.x; dst[p] = r;
        }
      }
    }
    h->cur_dec = -1;
  }
}

// The semaphore bits of an observation (observer.py:269-278: check_port_blocked per port of the switch) computed by the
// whole group: item j = port (j & 3); j < 4 the rule on the neighbour ("next") port, j >= 4 the rule on the port itself -- one
// item per lane, so the up to eight semaphore records behind them are fetched at once instead of one after the other; the
// verdicts meet in a vote.  `on`: this group has a decision coming (group-uniform); the vote is the whole warp's.
// Used by the shared-table kernels only: there it is worth +12 %; with private hash tables (every store of a decision goes
// to HBM-resident lines) the two extra warp syncs per decision cost more than the saved round trips (C4 -7 %, C2 -4 %).
template <int G, class Env>
SFL_FN int observe_bits(SFL_K, Env e, const Grp<G> &g, const int on, const int t) {
  const int now = e.h()->elapsed;
  const int s = on ? (e.trb()[t].y & 0xFFFF) : 0;
  const int4 sw = c_m.sw[s];
  unsigned bits = 0;
  SFL_UA
  for (int base = 0; base < 8; base += G) {
    const int j = base + g.gl;
    int b = 0;
    if (on && j < 8 && (j & 3) < sw.x) {
      const int port = sw.z + (j & 3);
      b = (j & 4) ? rule_port(e, port, t, now, SEM_IN) : rule_port(e, c_m.port[port].x, t, now, SEM_OUT);
    }
    bits |= (g.ballot(b) & 0xFFu) << base;
  }
  return (int)(~(bits | (bits >> 4)) & ((1u << sw.x) - 1u));
}

// observation of train t at its active switch (observer.py:246-308 + switch_agents.py:104-134)
struct Obs { int s, P, A, p0, a0, cur, semb, mask, ok; unsigned key; };
template <class Env>
SFL_FN Obs observe(SFL_K, Env e, int t, int now, const int4 ta, const int4 tb, const int semb_pre = -1) {
  Obs ob;
  ob.s = tb.y & 0xFFFF;
  const int4 sw = c_m.sw[ob.s];
  ob.P = sw.x; ob.A = sw.y; ob.p0 = sw.z; ob.a0 = sw.w;
  const int4 tr0 = c_m.train0[t], tr1 = c_m.train1[t];
  const int my_port = (int)((unsigned)ta.w >> 16);
  // compute_delay's distance lookup goes out before the port checks: its latency overlaps with theirs
  const int dist_now = c_m.dist[((size_t)tr0.w * (c_m.Hp * c_m.Wp) + ta.x) * 4 + (ta.y & 0xFF)];
  int semb = semb_pre;
  if (semb_pre < 0) {                                  // not precomputed by the group (observe_bits): port by port
    semb = 0;
    SFL_NU
    for (int k = 0; k < ob.P; k++)
      if (!port_blocked(e, c_m.port[ob.p0 + k].x, ob.p0 + k, t, now)) semb |= 1 << k;
  }
  ob.semb = semb;
  ob.cur = my_port - ob.p0;
  ob.ok = ob.cur >= 0 && ob.cur < ob.P;
  ob.key = 0u; ob.mask = 0;
  if (!ob.ok) return ob;
  int delay = now - tr1.y + dist_now;                                             // observer.py:41
  if (dist_now >= SFL_INF_DIST) { e.h()->err |= SFL_ERR_INF_DISTANCE; delay = now - tr1.y; }     // observer.py:35-36
  int level = delay <= 0 ? 0 : (delay <= (tr1.y - tr1.x) * 20 ? 1 : 2);           // observer.py:239-244
  ob.key = (((unsigned)(ob.p0 + ob.cur) * c_L.NT + tr0.w) * 16u + semb) * 3u + level;
  const int4 px = c_m.pexit[ob.p0 + ob.cur];                                      // switch_agents.py:104-134
  int mask = 1 << (ob.A - 1);
  {
    int ex[3] = {px.y, px.z, px.w};
#if SFL_DEV
#pragma unroll
#endif
    for (int i = 0; i < 3; i++) if (i < px.x && ((semb >> ((ex[i] >> 4) & 3)) & 1)) mask |= 1 << (ex[i] & 15);
  }
  ob.mask = mask;
  return ob;
}

// one switch-agent decision: observe (O1-O3) -> act (Q1) -> apply (E2, E3, R1) -> Q-update (Q2, Q3)
template <int KIND, class Env>
SFL_FN void decide(SFL_K, Env e, const Hp hp, int env_id, int t, const int semb_pre = -1) {
  const bool TRACE = KIND == K_FULL;
  const int mode = run_mode<KIND>(K);
  EnvHdr *h = e.h();
  const int now = h->elapsed;
  SFL_PHASE_START(h);
  int4 ta = e.tra()[t], tb = e.trb()[t];
  // What does not depend on the observation is loaded before it, so that these round trips to HBM overlap with the port
  // checks instead of following them one by one: last()'s reward, epsilon's decay product, the head of the pending list
  const int learning = mode == SFL_MODE_LEARN || mode == SFL_MODE_REPLAY;
  const int s_early = tb.y & 0xFFFF;
  const int reward_in = e.rewards()[s_early * c_L.T + t];                         // last(): _cumulative_rewards[agent][train]
  double eps_pow = 1.0;
  int ninter = 0;
  if (mode == SFL_MODE_LEARN) {
    eps_pow = e.sws()[s_early].eps_pow;
    if (KIND == K_FULL && c_L.off_rng) ninter = e.sws()[s_early].ninter;
  }
  int2 pend0 = make_int2(0, -1);
  if (learning && ((tb.y >> 16) & 0xFF)) pend0 = e.pend()[t * c_L.pend_cap];
  const Obs ob = observe(K, e, t, now, ta, tb, semb_pre);
  if (!ob.ok) {
    // observer.py:294-307: "No train detected at active switch" -- the reference then dies on an unbound current_port
    // (:307).  There is nothing to be faithful to past this point: flag the env, abandon the episode, carry on.
    h->err |= SFL_ERR_NO_TRAIN_AT_SWITCH; h->aborted++; h->truncated = 1;
    return;
  }
  const int s = ob.s, A = ob.A, p0 = ob.p0, a0 = ob.a0, cur = ob.cur, mask = ob.mask;
  const unsigned key = ob.key;
  const int4 tr0 = c_m.train0[t], tr1 = c_m.train1[t];
  const int pos = ta.x, dir = ta.y & 0xFF, st = (ta.y >> 8) & 0xFF;
  const int my_port = (int)((unsigned)ta.w >> 16);
  SFL_PHASE_MARK(h, PH_OBSERVE);
  // ---- act (distr_q.py:312-320 / :211)
  double *my_row = nullptr;
  int action = -1;
  if (mode == SFL_MODE_REPLAY || mode == SFL_MODE_STEP) {
    if (mode == SFL_MODE_STEP) h->act_cursor = 0;              // the host's action for this decision
    int exploited = 0;
    if (h->act_cursor >= c_ra.act_cap) { h->err |= SFL_ERR_REPLAY_UNDERRUN; action = A - 1; }
    else {
      action = c_ra.replay_act[(size_t)env_id * c_ra.act_cap + h->act_cursor++];
      // bit 6 of a recorded action: the learner exploited, i.e. max_action was consulted -- which inserts the row
      // (distr_q.py:318-319, 482); the replay then also checks that the recorded action IS the argmax
      if (mode == SFL_MODE_REPLAY && action >= 0 && (action & 0x40)) { exploited = 1; action &= 0x3F; }
    }
    if (action < 0 || action >= A) { h->err |= SFL_ERR_BAD_ACTION; action = A - 1; }
    if (exploited) {
      my_row = q_row(K, e, hp, key);
      if (max_action(my_row, A, mask) != action) h->err |= SFL_ERR_REPLAY_DIVERGED;
    }
  } else if (KIND == K_FULL && mode == SFL_MODE_LEARN && c_L.off_rng) {
    // the reference's stream: one random() per decision, exploit included; the exploring branch draws its seed from it
    Pcg *gp = (Pcg *)(hot_ptr(e.hot) + c_L.off_rng);
    Pcg g = *gp;
    if (eps_explore(pcg_double(g), hp->epsilon, hp->epsilon_decay_rate, ninter, eps_pow)) action = pcg_explore_action(g, mask);
    *gp = g;
  } else if (mode == SFL_MODE_LEARN) {
    double eps = dmul(hp->epsilon, eps_pow);
    // one Philox4x32-10 block per PAIR of decisions: counter (step_counter >> 1, episode, 0x5F1, 0), key = env seed; the
    // even decision of the pair uses words 0-1, the odd one words 2-3 (kept in the header, so the stream does not depend
    // on how the run is cut into launches)
    const int pair = h->step_counter >> 1;
    unsigned ux, uy;
    if ((h->step_counter & 1) && h->eps_tag == pair) { ux = h->eps_z; uy = h->eps_w; }
    else {
      const U4 u = philox4x32((unsigned)pair, (unsigned)(hp->episode_base + h->episode), 0x5F1u, 0u, (unsigned)hp->seed, (unsigned)(hp->seed >> 32));
      h->eps_tag = pair; h->eps_z = u.z; h->eps_w = u.w;
      if (h->step_counter & 1) { ux = u.z; uy = u.w; } else { ux = u.x; uy = u.y; }
    }
    double u01 = ((double)ux + 0.5) * (1.0 / 4294967296.0);
    if (u01 < eps) {                                       // explore: uniform over the allowed actions
      int pick = (int)(((unsigned long long)uy * (unsigned)popc32((unsigned)mask)) >> 32);
      unsigned mm = (unsigned)mask;
      SFL_NU
      for (; pick > 0; pick--) mm &= mm - 1;
      action = ffs64(mm);
    }
  }
  if (action < 0) {                                        // exploit (distr_q.py:318-319) / test() (:211)
    if (Env::EVQ) action = eval_action(K, key, A, mask);
    else {
      my_row = q_row(K, e, hp, key);
      action = max_action(my_row, A, mask);
    }
  }
  SFL_PHASE_MARK(h, PH_ACT);
  // ---- apply (switch_env.py:203-294, switch_agents.py:136-168)
  int moving = 0, move2 = A_STOP, in_port = my_port, out_port = my_port;
  if (action != A - 1) {
    int4 ac = c_m.act[a0 + action];
    if (ac.x == cur) { moving = 1; move2 = ac.z; in_port = p0 + ac.x; out_port = p0 + ac.y; }
  }
  int next_switch = s, next_port = -1;
  if (moving) {                                                                   // rail_network.py:246-278
    int4 op = c_m.port[out_port];
    next_port = op.x;
    int old_prev = (tb.x & 0xFFFF) == 0xFFFF ? -1 : (tb.x & 0xFFFF);
    transition_semaphore(K, e, in_port, out_port, next_port, t, now, st, my_port, old_prev);
    tb.x = (out_port & 0xFFFF) | (in_port << 16);                                 // prev_port = out, source_port = in
    ta.w = (ta.w & 0xFFFF) | (next_port << 16);
    next_switch = c_m.port[next_port].w;
  }
  unsigned plan = (unsigned)ta.z & 0xFFFFu;
  int pl = ta.z >> 16;
  if (moving && pl > 0) { plan = (plan & 0xFu) | ((unsigned)move2 << 4); pl = 2; }            // :257-266
  else if (!moving) {                                                             // :267-270
    if (pl >= SFL_PLAN_CAP) { h->err |= SFL_ERR_PLAN_FULL; pl = SFL_PLAN_CAP - 1; }
    plan = ((plan << 4) | A_STOP) & 0xFFFFu; pl++;
  } else { plan = A_FWD | ((unsigned)move2 << 4); pl = 2; }                       // :271-272
  ta.z = (int)plan | (pl << 16);
  e.tra()[t] = ta;
  int all_blocked = 1;                                                            // :274-282
  if ((plan & 0xFu) == A_STOP) {                         // only consulted for the stop penalty (reward_func.py:61-76)
    if (moving) all_blocked = port_blocked(e, next_port, out_port, t, now);
    else all_blocked = (mask == (1 << (A - 1)));         // no transition happened: the observe bits still hold
  }
  int cell = pos, d2 = dir;                                                       // reward_func.py:23-78
  {
    unsigned pp = plan;
    SFL_NU
    for (int i = 0; i < pl; i++, pp >>= 4) {
      int a = pp & 0xF;
      if (a != A_STOP) { Mv c = check_action(K, a, cell, d2); cell = c.cell; d2 = c.dir; }
    }
  }
  int curr = delay_at(K, e, tr0.w, cell, d2, now, tr1.y);
  int reward_out = tb.z - curr;
  if (!all_blocked && (plan & 0xFu) == A_STOP) reward_out -= 1300;
  e.rewards()[next_switch * c_L.T + t] = reward_out;                              // switch_env.py:289
  tb.z = curr;                                                                    // switch_env.py:291
  h->step_counter++;
  SFL_PHASE_MARK(h, PH_APPLY);
  // ---- learn (distr_q.py:329-342)
  if (learning) {
    int n = (tb.y >> 16) & 0xFF;
    int2 *pend = e.pend() + t * c_L.pend_cap;
    int hit = -1, same = -1;
    SFL_NU
    for (int i = 0; i < n; i++) {
      int nsw = (i ? pend[i].y : pend0.y) & 0xFFF;
      if (nsw == s && hit < 0) hit = i;
    }
    if (hit >= 0) {
      int2 pe = hit ? pend[hit] : pend0;
      const int prev_sw = (pe.y >> 12) & 0xFFF;
      // max_q creates the successor row (distr_q.py:463-465) -- but only when it is consulted: not for a train that
      // stayed at the same switch (:444-447)
      if (prev_sw != s && !my_row) my_row = q_row(K, e, hp, key);
      q_update(K, e, hp, (unsigned)pe.x, (pe.y >> 24) & 15, (double)reward_in, my_row, prev_sw, s);
      SFL_NU
      for (int j = hit; j + 1 < n; j++) pend[j] = pend[j + 1];
      n--;
    }
    // update_dict[(next_switch, train)] = (obs, action, agent): the same key overwrites in place (:340-342)
    int meta = next_switch | (s << 12) | (action << 24);
    SFL_NU
    for (int i = 0; i < n; i++) if ((pend[i].y & 0xFFF) == next_switch) same = i;
    if (same >= 0) pend[same] = make_int2((int)key, meta);
    else if (n >= c_L.pend_cap) h->err |= SFL_ERR_PEND_FULL;
    else { pend[n] = make_int2((int)key, meta); n++; }
    tb.y = (tb.y & 0xFFFF) | (n << 16);
  }
  e.trb()[t] = tb;
  SFL_PHASE_MARK(h, PH_UPDATE);
  h->cum_reward += (double)reward_in;                                             // distr_q.py:360
  if (TRACE) {
    if (c_ra.trace_dec) {
      h->cur_dec = h->n_dec_logged;
      if (h->n_dec_logged < c_ra.dec_cap) {
        sfl_dec_rec *rec = c_ra.trace_dec + (size_t)env_id * c_ra.dec_cap + h->n_dec_logged;
        rec->ep = h->episode; rec->tick = now; rec->sw = s; rec->train = t; rec->key = key; rec->mask = mask;
        rec->action = action; rec->next_sw = next_switch; rec->reward = reward_in; rec->done = 0; rec->arrived = 0;
        rec->arrived_hi = 0;
      }
      h->n_dec_logged++;
    }
  }
  if (TRACE) h->last_next_sw = next_switch;
  h->decisions++;
  if (mask == (1 << (A - 1))) h->forced_stops++;
  if (action == A - 1) h->stop_actions++;
  h->pending_fin = s;
}

// ------------------------------------------------------------------------------------------------ reset (E1)
// switch_env.py:93-158 with a constant map: state re-init + the precomputed _init_ports table (:507-568)
// (`on`: this group resets; the syncs are the whole warp's)
template <int G, class Env>
SFL_RARE void env_reset(SFL_K, Env e, const Grp<G> &g, int on) {
  EnvHdr *h = e.h();
  const int T = on ? c_L.T : 0, NP = on ? c_L.NP : 0;
  SFL_NU
  for (int t = g.gl; t < T; t += G) {
    int4 tr0 = c_m.train0[t], tr1 = c_m.train1[t];
    e.tra()[t] = make_int4(-1, tr0.y | (ST_WAITING << 8) | (0 << 16) | (A_NONE << 24), 0, (int)((unsigned)tr1.z << 16));
    int4 b = e.trb()[t];
    // prev_port / source_port are NOT cleared: RailNetwork.reset (rail_network.py:135-149) keeps them
    e.trb()[t] = make_int4(b.x, 0xFFFF, c_m.init_delay[t], SFL_NO_STOP);
  }
  SFL_NU
  for (int p = g.gl; p < NP; p += G) e.sem_put(p, make_int4(0, 0, -1, 0));
  SFL_NU
  for (int i = g.gl; i < c_L.S * T; i += G) e.rewards()[i] = 0;
  g.sync();
  if (on && g.gl == 0) {
    SFL_NU
    for (int t = 0; t < T; t++) {                                         // switch_env.py:564-568, train order
      int4 tr1 = c_m.train1[t];
      e.sem_put(tr1.z, make_int4(tr1.x - 2, tr1.w + 2, t, SEM_IN));
    }
    h->elapsed = 0; h->step_counter = 0; h->num_malf = 0; h->terminated = 0; h->truncated = 0; h->need_reset = 0;
    h->pending_fin = -1; h->cur_dec = -1; h->ev_cursor = 0; h->active_mask = 0; h->malf_prev_mask = 0; h->at_dest_mask = 0;
    h->eps_tag = -1;
    h->done_mask = 0; h->cum_reward = 0.0;
    if (Env::NW > 1) { SFL_UA for (int m = 0; m < 4; m++) *e.hw1(m) = 0ull; }
  }
  g.sync();
}

// ------------------------------------------------------------------------------------------------ one tick (E5-E7, F2-F5)
// Group-uniform registers carried across the ticks of a launch (every lane of the group holds the same values);
// the header copy in shared memory is what the decision phase (first lane) reads and writes.
template <int NW> struct TickRegs {
  int elapsed, ended, rng_blk;                 // rng_blk: 16-tick block the cached malfunction bytes belong to (-1: none)
  TSet<NW> active, done;
  unsigned ticks, train_ticks;                 // launch-local (max_ticks * T < 2^32), added to the header at the end
};

// Malfunction draw of train t at tick `now` (row F5), probability thr / 2^32 = 1 - exp(-rate) per (train, tick), in two
// stages so that the common no-event tick costs one byte compare:
//   stage 1  one Philox4x32-10 call per (train, 16-tick block), counter (tick >> 4, train, 0xA11F, 0): 16 bytes, byte
//            tick & 15 is a candidate iff it is below B = ceil(thr / 2^24)                         (probability B / 256)
//   stage 2  candidates only: Philox counter (tick, train, 0xA11E, 0); event iff word 0 < thr2 = floor(thr * 256 / B)
//            (sfl_hparams.malf_thr2; probability thr2 / 2^32, product = thr / 2^32); word 1 gives the duration
//            min + U{0..max-min} + 1.
SFL_FN int malf_stage2(const Hp hp, int now, int t) {
  const U4 u = philox4x32((unsigned)now, (unsigned)t, 0xA11Eu, 0u, (unsigned)hp->seed, (unsigned)(hp->seed >> 32));
  if (u.x >= hp->malf_thr2) return 0;
  return hp->malf_min + (int)(((unsigned long long)u.y * (unsigned)(hp->malf_max - hp->malf_min + 1)) >> 32) + 1;
}

// ONE: every train has its own lane (T <= G), so each per-train phase is a single pass and the train bit-sets are one
// ballot each -- the loops and the 64-bit shifts fold away at compile time (+4 % on C2).
template <int G, int KIND, bool ONE, class Env>
// `live` = this group's environment takes part (not halted, not an idle slot of the last warp); every loop bound and
// branch that contains a collective is warp-uniform, the per-group work inside is predicated.
SFL_FN void env_tick(SFL_K, Env e, Scratch sc, const Hp hp, int env_id, const Grp<G> &g, TickRegs<Env::NW> &R, const int live) {
  const bool TRACE = KIND == K_FULL;
  EnvHdr *h = e.h();
  const int Tw = c_L.T;                                                  // warp-uniform loop bound
  const int T = live ? Tw : 0;
  const int now = R.elapsed + 1;                                         // flatland: _elapsed_steps += 1 first
  const int replay_ev = KIND != K_LEARN && c_ra.replay_ev != 0;          // never in the learn kernel (sfl_run binds events for learn only with the reference stream)
  const unsigned thr = live ? hp->malf_threshold : 0u;
  if (replay_ev) {
    SFL_NU
    for (int t = g.gl; t < T; t += G) sc.inj()[t] = 0;
    g.sync();
    if (live && g.gl == 0) {
      const int *ev = c_ra.replay_ev + (size_t)env_id * c_ra.ev_cap * 3;
      int c = h->ev_cursor;
      SFL_NU
      while (c < c_ra.ev_cap && ev[c * 3] >= 0 && ev[c * 3] <= now) { if (ev[c * 3] == now) sc.inj()[ev[c * 3 + 1]] = ev[c * 3 + 2]; c++; }
      h->ev_cursor = c;
    }
    g.sync();
  }
  const int fresh_rng = !replay_ev && thr && (now >> 4) != R.rng_blk;    // group-uniform
  const unsigned coarse = (thr >> 24) + ((thr & 0xFFFFFFu) ? 1u : 0u);   // stage-1 byte threshold B
  // ---- phase A: per train: plan pop (switch_env.py:304-339) + flatland step part 1 (Appendix B step 2)
  SFL_NU
  for (int t = g.gl, once_ = 1; t < T && (!ONE || once_); t += G, once_ = 0) {
    int4 ta = e.tra()[t];
    const int p = ta.x, d = ta.y & 0xFF, st = (ta.y >> 8) & 0xFF;
    int saved = (ta.y >> 16) & 0xFF, prev_act = (ta.y >> 24) & 0xFF;
    unsigned plan = (unsigned)ta.z & 0xFFFFu;
    int pl = ta.z >> 16, mc = ta.w & 0xFFFF;
    // F5 malfunction draw: every train, every tick; applied only when the counter is 0
    int dur = 0;
    if (replay_ev) dur = sc.inj()[t];
    else if (thr) {
      if (fresh_rng) {
        U4 u = philox4x32((unsigned)(now >> 4), (unsigned)t, 0xA11Fu, 0u, (unsigned)hp->seed, (unsigned)(hp->seed >> 32));
        sc.rng()[t] = make_int4((int)u.x, (int)u.y, (int)u.z, (int)u.w);
      }
      if (((const uint8_t *)&sc.rng()[t])[now & 15] < coarse) dur = malf_stage2(hp, now, t);
    }
    if (mc == 0 && dur > 0) mc = dur;
    int src, dst, ecell = -1, nd = d, act = A_NOTHING, a = A_NOTHING, flags = 0;
    if (st == ST_DONE) { src = dst = -1 - t; }
    else {
      int pp = p, dd = d;
      if (p < 0) { const int4 tr0 = c_m.train0[t]; pp = tr0.x; dd = tr0.y; }
      const unsigned me = mv_entry(K, pp, dd);
      if (pl == 0) a = A_FWD;
      else { a = plan & 0xF; prev_act = a; plan >>= 4; pl--; }
      if (p >= 0) { Mv c = mv_apply(K, me, a, p); ecell = c.valid ? c.cell : p; flags = 1 | (c.valid ? 2 : 0); }
      // action preprocessing (a is never DO_NOTHING here: the reference always sends an action)
      act = a;
      if (st == ST_WAITING) act = A_NOTHING;
      if ((act == A_LEFT || act == A_RIGHT) && !mv_valid(me, act)) act = A_FWD;
      if (is_moving(act) && !mv_valid(me, act)) act = A_STOP;
      if (is_moving(act) && !saved) saved = act;
      const int upd = (mc == 0) && act != A_STOP;
      int ncell = p;
      if (p < 0) { if (saved) { ncell = pp; nd = dd; } }
      else if (saved && upd) { Mv c = mv_apply(K, me, saved, p); if (c.valid) { ncell = c.cell; nd = c.dir; } act = saved; }
      src = p >= 0 ? p : -1 - t;
      dst = ncell >= 0 ? ncell : src;
    }
    ta.y = d | (st << 8) | (saved << 16) | (prev_act << 24);
    ta.z = (int)plan | (pl << 16);
    ta.w = (ta.w & (int)0xFFFF0000) | mc;
    e.tra()[t] = ta;
    sc.tmp()[t] = make_int4(src, dst, ecell, nd | (act << 8) | (a << 16) | (flags << 24));
  }
  if (fresh_rng) R.rng_blk = now >> 4;
  g.sync();
  // ---- phase B: motion check (F3)
  TSet<Env::NW> chain;                        // trains whose destination is occupied by a train that is itself moving
  chain.clear();
  SFL_NU
  for (int base = 0; base < (ONE ? 1 : Tw); base += (ONE ? 1 : G)) {
    const int t = base + g.gl;
    int follows = 0;
    if (t < T) {
      int4 m = sc.tmp()[t];
      int s = m.x, d = m.y;
      int wants = d != s, blocked = !wants, occ = -1;
      if (wants) {
        SFL_NU
        for (int k = 0; k < T; k++) {
          const int2 o = *(const int2 *)&sc.tmp()[k];
          occ = o.x == d ? k : occ;                                      // k != t: my own src differs from my dst
          blocked |= (o.y == d) & (o.y != o.x) & (k < t);                // lowest handle wins a contended cell
        }
        if (occ >= 0) { int2 o = *(const int2 *)&sc.tmp()[occ]; if (o.y == s && o.y != o.x) blocked = 1; }   // swap
      }
      sc.occ()[t] = (int8_t)occ; sc.blk()[t] = (uint8_t)blocked;
      follows = !blocked && occ >= 0;
    }
    chain.or_ballot(g.ballot(follows), base);
  }
  g.sync();
  if (g.wany(chain.any())) {                                               // chains: fixed point (monotone)
    SFL_NU
    for (int iter = 0; iter < Tw; iter++) {
      int changed = 0;
      if (chain.any()) {
        SFL_NU
        for (int t = g.gl, once_ = 1; t < T && (!ONE || once_); t += G, once_ = 0) {
          int occ = sc.occ()[t];
          if (!sc.blk()[t] && occ >= 0 && ((volatile uint8_t *)sc.blk())[occ]) { sc.blk()[t] = 1; changed = 1; }
        }
      }
      g.sync();
      if (!g.wany(changed)) break;
    }
  }
  // ---- phase C: state machine + position update (Appendix B steps 4-5), held-back trains (switch_env.py:353-367),
  //      and _check_active_switch (switch_env.py:427-485), which reads only the train's own new state
  TSet<Env::NW> done_bits, malf_bits, broken_bits, depart_bits, active;      // broken: ended the tick in state MALFUNCTION
  done_bits.clear(); malf_bits.clear(); broken_bits.clear(); depart_bits.clear(); active.clear();
  SFL_NU
  for (int base = 0; base < (ONE ? 1 : Tw); base += (ONE ? 1 : G)) {
    const int t = base + g.gl;
    int f_done = 0, f_malf = 0, f_broken = 0, f_dep = 0, f_act = 0;
    if (t < T) {
      int4 ta = e.tra()[t];
      const int4 m = sc.tmp()[t];
      int p = ta.x, d = ta.y & 0xFF;
      const int st = (ta.y >> 8) & 0xFF;
      int saved = (ta.y >> 16) & 0xFF;
      const int prev_act = (ta.y >> 24) & 0xFF;
      unsigned plan = (unsigned)ta.z & 0xFFFFu;
      int pl = ta.z >> 16, mc = ta.w & 0xFFFF, next_port = (int)((unsigned)ta.w >> 16);
      const int act = (m.w >> 8) & 0xFF, popped = (m.w >> 16) & 0xFF, fl = (m.w >> 24) & 0xFF;
      const int wants = m.y != m.x;
      const int in_malf = mc > 0, allowed = !in_malf && wants && !sc.blk()[t];
      const int4 tr0 = c_m.train0[t];
      const int ed = c_m.train1[t].x;
      const int ed_reached = now >= ed, stop_given = act == A_STOP, valid_move = is_moving(act) && allowed, conflict = !allowed;
      int nxt = st;
      switch (st) {
        case ST_WAITING: if (in_malf) nxt = ST_MALF_OFF; else if (ed_reached) nxt = ST_READY; break;
        case ST_READY: if (in_malf) nxt = ST_MALF_OFF; else if (valid_move) nxt = ST_MOVING; break;
        case ST_MALF_OFF:
          if (!in_malf) { if (ed_reached) nxt = valid_move ? ST_MOVING : ST_STOPPED; else nxt = ST_WAITING; }   // Appendix B step 4
          break;
        case ST_MOVING: if (in_malf) nxt = ST_MALF; else if (stop_given || conflict) nxt = ST_STOPPED; break;
        case ST_STOPPED: if (in_malf) nxt = ST_MALF; else if (valid_move) nxt = ST_MOVING; break;
        case ST_MALF: if (!in_malf && valid_move) nxt = ST_MOVING; else if (!in_malf && (stop_given || conflict)) nxt = ST_STOPPED; break;
        default: break;
      }
      if (nxt >= ST_MOVING && nxt <= ST_MALF) {
        if (st <= ST_MALF_OFF) { p = tr0.x; d = tr0.y; }
        else if (allowed) { p = m.y; d = m.w & 0xFF; if (p == tr0.z) nxt = ST_DONE; }
      }
      if (nxt == ST_DONE) p = -1;
      if (mc > 0) mc--;
      if (p >= 0) saved = 0;
      f_done = nxt == ST_DONE; f_malf = mc != 0; f_broken = nxt == ST_MALF; f_dep = now == ed - 2;
      if (nxt == ST_STOPPED || nxt == ST_MALF) e.trb()[t].w = now;        // extend_semaphores (rail_network.py:229-244): t0_eff
      if (TRACE) {
        if (c_ra.trace_tick && h->n_tick_logged < c_ra.tick_cap) {
          sfl_tick_rec *rec = c_ra.trace_tick + ((size_t)env_id * c_ra.tick_cap + h->n_tick_logged) * T + t;
          rec->pos = p; rec->dir = (int8_t)d; rec->state = (int8_t)nxt; rec->malf = (int16_t)mc;
        }
      }
      // flatland held the train back (switch_env.py:353-367)
      if ((fl & 1) && (fl & 2) && m.z != p && popped != A_STOP) {
        if (pl >= SFL_PLAN_CAP) { h->err |= SFL_ERR_PLAN_FULL; pl = SFL_PLAN_CAP - 1; }
        plan = ((plan << 4) | (unsigned)popped) & 0xFFFFu; pl++;
        if (c_m.cell_switch[m.z] >= 0) {
          int src_port = (int)((unsigned)e.trb()[t].x >> 16);
          if (src_port != 0xFFFF) next_port = src_port;
        }
      }
      // _check_active_switch (switch_env.py:427-485)
      if (p >= 0 && nxt != ST_WAITING) {
        int peek = pl ? (int)(plan & 0xF) : A_FWD;
        Mv c = check_action(K, peek, p, d);
        int s = c_m.cell_switch[c.cell];
        if (s >= 0) {
          int ok = 1;
          if (nxt == ST_MOVING || nxt == ST_READY) { }
          else if ((nxt == ST_STOPPED || nxt == ST_MALF) && prev_act == A_STOP) { }
          else if (nxt == ST_STOPPED || nxt == ST_MALF) s = c_m.port[next_port].w;
          else ok = 0;
          if (ok) { ((uint16_t *)&e.trb()[t].y)[0] = (uint16_t)s; f_act = 1; }
        }
      }
      ta.x = p;
      ta.y = d | (nxt << 8) | (saved << 16) | (prev_act << 24);
      ta.z = (int)plan | (pl << 16);
      ta.w = mc | (next_port << 16);
      e.tra()[t] = ta;
    }
    done_bits.or_ballot(g.ballot(f_done), base);
    malf_bits.or_ballot(g.ballot(f_malf), base);
    broken_bits.or_ballot(g.ballot(f_broken), base);
    depart_bits.or_ballot(g.ballot(f_dep), base);
    active.or_ballot(g.ballot(f_act), base);
  }
  const int ended = live && (done_bits.all(Tw) || now >= c_m.max_episode_steps);   // dones["__all__"] (Appendix B step 6)
  const TSet<Env::NW> prev_done = R.done;
  // ---- phase D2: semaphores of done trains (switch_env.py:370-376); every train counts as done at the end
  const int release = done_bits.andnot(prev_done).any() || ended;
  if (g.wany(release)) {
    const int NP = release ? c_L.NP : 0;
    SFL_NU
    for (int p = g.gl; p < NP; p += G) {
      int tr = e.owner(p);
      if (tr >= 0 && (ended || done_bits.test(tr))) e.sem_drop(p);
    }
  }
  // ---- phase D3: departure bookings (switch_env.py:379-384), then the bookings of extend_semaphores for trains in
  //      MALFUNCTION (rail_network.py:229-244; the slide of the stopped trains' windows is their stop_tick), train order
  if (g.wany(depart_bits.any() || broken_bits.any())) {
    g.sync();
    if (g.gl == 0) {
      TSet<Env::NW> b = depart_bits;
      SFL_NU
      while (b.any()) {
        int t = b.pop();
        int4 tr1 = c_m.train1[t];
        e.sem_put((int)((unsigned)e.tra()[t].w >> 16), make_int4(tr1.x - 2, tr1.w + 2, t, SEM_IN));
      }
      b = broken_bits;
      SFL_NU
      while (b.any()) {
        int t = b.pop();
        int port = (int)((unsigned)e.tra()[t].w >> 16);
        if (e.owner(port) < 0) e.sem_put(port, make_int4(now, c_m.train1[t].w, t, SEM_IN));
      }
    }
  }
  if (live && g.gl == 0) {
    h->elapsed = now;
    const TSet<Env::NW> malf_prev = tset(e, HM_MALF);
    const TSet<Env::NW> new_malf = malf_bits.andnot(malf_prev);
    if (new_malf.any()) h->num_malf += new_malf.popc();                  // switch_env.py:399-401
    if (!(malf_bits == malf_prev)) tset_put(e, HM_MALF, malf_bits);
    if (!(done_bits == prev_done)) tset_put(e, HM_DONE, done_bits);
    if (ended) h->terminated = 1;
    if (active.any()) tset_put(e, HM_ACTIVE, active);                     // the queue is empty whenever a tick runs
    if (TRACE) { if (c_ra.trace_tick) h->n_tick_logged++; }
  }
  R.elapsed = now; R.ended = ended; R.active = active; R.done = done_bits;
  if (live) { R.ticks++; R.train_ticks += (unsigned)(T - prev_done.popc()); }
  g.sync();
}

// ------------------------------------------------------------------------------------------------ episode end
template <class Env>
SFL_RARE void episode_end(SFL_K, Env e, int env_id) {   // first lane
  EnvHdr *h = e.h();
  if (c_ra.ep_log && h->n_ep_logged < c_ra.ep_cap) {
    const TSet<Env::NW> done = tset(e, HM_DONE);
    sfl_ep_rec *rec = c_ra.ep_log + (size_t)env_id * c_ra.ep_cap + h->n_ep_logged;
    rec->cum_reward = h->cum_reward; rec->decisions = h->step_counter; rec->arrived = done.popc();
    rec->num_malfunctions = h->num_malf; rec->ticks = h->elapsed; rec->arrived_mask = done.w[0];
    rec->arrived_mask_hi = Env::NW > 1 ? done.w[Env::NW - 1] : 0ull;
    if (c_ra.ep_delay) {
      int *d = c_ra.ep_delay + ((size_t)env_id * c_ra.ep_cap + h->n_ep_logged) * c_L.T;
      SFL_NU
      for (int t = 0; t < c_L.T; t++) d[t] = e.trb()[t].z;
    }
  }
  h->arrived_trains += (unsigned)tset(e, HM_DONE).popc();
  h->n_ep_logged++;
  h->episode++;
  h->need_reset = 1;
}

// ------------------------------------------------------------------------------------------------ the per-env driver
// Staging area of one group in the CTA's dynamic shared memory, at byte offset `stage`:
// [hot env state (hot_bytes) | sfl_hparams | Scratch].  The host build has no staging: it works on the env block itself.
// One launch = max_ticks iterations; an iteration is one flatland tick preceded by every switch-agent decision that is
// due (and by the end-of-episode bookkeeping + in-place reset when the episode is over).
// ------------------------------------------------------------------------------------------------ SFL_MODE_STEP
// The AEC protocol driven from the host (switch_env.py:616-666): report the waiting decision the way AECEnv.last()
// would, or the end of the episode.  First lane of the group.
template <class Env>
SFL_FN void step_report(SFL_K, Env e, int env_id, int t) {
  EnvHdr *h = e.h();
  sfl_step_rec *o = c_ra.step_out + env_id;
  o->pending = 0; o->sw = -1; o->train = -1; o->key = 0u; o->mask = 0;
  if (t >= 0) {
    const int4 ta = e.tra()[t], tb = e.trb()[t];
    const Obs ob = observe(K, e, t, h->elapsed, ta, tb);
    if (!ob.ok) { h->err |= SFL_ERR_NO_TRAIN_AT_SWITCH; h->aborted++; h->truncated = 1; }    // last() raises in the reference
    else {
      o->pending = 1; o->sw = ob.s; o->train = t; o->key = ob.key; o->mask = ob.mask;
      SFL_NU
      for (int k = 0; k < c_L.T; k++) o->rewards[k] = e.rewards()[ob.s * c_L.T + k];
      h->cur_train = t;
    }
  }
  o->done = h->terminated | (h->truncated << 1);
  o->elapsed = h->elapsed; o->last_next_sw = h->last_next_sw; o->arrived = h->done_mask;
  o->arrived_hi = Env::NW > 1 ? *e.hw1(HM_DONE) : 0ull;
}

template <int G, int KIND, bool TH, bool SQ, bool ONE, int NW = 1, bool EVQ = false>
SFL_FN void env_run(SFL_K, int env_id, unsigned stage, char *host_scratch) {
  const bool TRACE = KIND == K_FULL;
  const Grp<G> g;
  const int valid = env_id < c_ra.n_envs;                                 // idle slots of the last warp keep the warp's rendezvous
  if (!valid) env_id = 0;
  char *gbase = c_ra.state + (size_t)env_id * c_L.env_stride;
  const unsigned hot_bytes = valid ? c_ra.hot_bytes : 0u;
  typename EnvOf<TH, SQ, NW, EVQ>::type e;
  Hp hp;
  Scratch sc;
  e.kp = &K; sc.kp = &K;
  e.gb = gbase;
#if SFL_DEV
  {
    char *smem = g_smem + stage;
    SFL_NU
    for (unsigned o = g.gl * 16u; o < hot_bytes; o += G * 16u) *(int4 *)(smem + o) = *(const int4 *)(gbase + o);
    if (valid) {
      SFL_NU
      for (unsigned o = g.gl * 16u; o < (unsigned)sizeof(sfl_hparams); o += G * 16u)
        *(int4 *)(smem + c_ra.hot_bytes + o) = *(const int4 *)((const char *)(c_ra.hp + env_id) + o);
    }
    g.sync();
    e.hot = stage;
    hp.o = stage + c_ra.hot_bytes;
    sc.base = stage + c_ra.hot_bytes + (unsigned)sizeof(sfl_hparams);
    e.own = sc.base + scratch_bytes(c_L.T);
    if (!TH) {                                                            // holders of the semaphore records, from HBM
      const int NPv = valid ? c_L.NP : 0;
      SFL_NU
      for (int p = g.gl; p < NPv; p += G) e.own_ptr()[p] = (uint8_t)e.sem()[p].z;
      g.sync();
    }
  }
#else
  (void)stage;
  e.hot = gbase;
  e.own = gbase;                                                          // unused: the host build keeps everything "hot"
  hp.o = (char *)(c_ra.hp + env_id);
  sc.base = host_scratch;
#endif
  EnvHdr *h = e.h();
  TickRegs<NW> R;
  R.elapsed = 0; R.ended = 0; R.rng_blk = -1; R.active.clear(); R.done.clear(); R.ticks = 0; R.train_ticks = 0;
  int need_reset = 0, live = 0;
  if (valid) {
    R.elapsed = h->elapsed; R.ended = h->terminated | h->truncated;
    R.active = tset(e, HM_ACTIVE); R.done = tset(e, HM_DONE);
    need_reset = h->need_reset; live = !h->halted;
  }
  const int stepping = TRACE && run_mode<KIND>(K) == SFL_MODE_STEP;
  int paused = 0;                                                         // stepping: a decision waits for the host
  if (stepping) {
    if (live && g.gl == 0) {
      if (h->cur_train >= 0) { decide<KIND>(K, e, hp, env_id, h->cur_train); h->cur_train = -1; }
      else h->last_next_sw = -1;
    }
    g.sync();
    if (live) R.ended = h->terminated | h->truncated;
  }
  int any_reset = g.wany(live && need_reset);                             // warp-uniform; can only change in a decision phase
  SFL_NU
  for (int it = 0; it < c_ra.max_ticks; it++) {
    const int due = live && !paused && (R.active.any() || R.ended);             // something is due before the tick
    const unsigned wf = g.wor((live && !paused ? 1u : 0u) | (due ? 2u : 0u));   // one warp-wide OR: anybody running / due
    if (!(wf & 1u)) break;
    if (wf & 2u) {
      if (due && g.gl == 0 && stepping) {
        if (h->pending_fin >= 0 && (tset_any(e, HM_ACTIVE) || h->terminated)) finish_decision<KIND>(K, e, hp, env_id);
        int t = -1;
        if (!(h->terminated || h->truncated) && tset_any(e, HM_ACTIVE)) t = tset_pop(e, HM_ACTIVE);
        step_report(K, e, env_id, t);
        if (h->terminated || h->truncated) episode_end(K, e, env_id);
      } else if (SQ && !stepping) {
        // shared-table kernels: per decision the first lane closes the previous one and names the next train, the whole
        // group evaluates the port checks of its observation at once (observe_bits), the first lane decides with those bits
        int more = due;
        SFL_NU
        while (g.wany(more)) {
          if (more && g.gl == 0) {
            if (h->pending_fin >= 0 && (tset_any(e, HM_ACTIVE) || h->terminated)) finish_decision<KIND>(K, e, hp, env_id);
            h->dec_go = !(h->terminated || h->truncated || !tset_any(e, HM_ACTIVE));
            if (h->dec_go) h->dec_t = tset_pop(e, HM_ACTIVE);
          }
          g.sync();
          if (more) more = h->dec_go;
          const int t = more ? h->dec_t : 0;
          const int semb = observe_bits(K, e, g, more, t);
          if (more && g.gl == 0) decide<KIND>(K, e, hp, env_id, t, semb);
        }                                                                 // (the sync at the top of the next round orders the first lane's stores)
        if (due && g.gl == 0 && (h->terminated || h->truncated)) episode_end(K, e, env_id);
      } else if (due && g.gl == 0) {
        SFL_NU
        for (;;) {                                                        // agent_iter: FIFO in train-handle order
          if (h->pending_fin >= 0 && (tset_any(e, HM_ACTIVE) || h->terminated)) finish_decision<KIND>(K, e, hp, env_id);
          if (h->terminated || h->truncated || !tset_any(e, HM_ACTIVE)) break;
          const int t = tset_pop(e, HM_ACTIVE);
          decide<KIND>(K, e, hp, env_id, t);
        }
        if (h->terminated || h->truncated) episode_end(K, e, env_id);
      }
      g.sync();
      if (due) { need_reset = h->need_reset; R.active.clear(); if (stepping) paused = h->cur_train >= 0; }
      any_reset = g.wany(live && need_reset);
    }
    if (any_reset) {
      if (live && need_reset && hp->episodes >= 0 && h->episode >= hp->episodes) live = 0;      // halt: need_reset stays set
      const int on = live && need_reset;
      if (on && g.gl == 0) SFL_PHASE_START(h);
      env_reset<G>(K, e, g, on);
      if (on && g.gl == 0) SFL_PHASE_MARK(h, PH_RESET);
      if (on) { need_reset = 0; R.elapsed = 0; R.ended = 0; R.rng_blk = -1; R.active.clear(); R.done.clear(); }
      any_reset = 0;
    }
    if (live && !paused && g.gl == 0) SFL_PHASE_START(h);
    env_tick<G, KIND, ONE>(K, e, sc, hp, env_id, g, R, live && !paused);
    if (live && !paused && g.gl == 0) SFL_PHASE_MARK(h, PH_TICK);
  }
  g.sync();
  if (valid && g.gl == 0) {
    h->halted = !live;
    h->ticks += R.ticks; h->train_ticks += R.train_ticks;
    sfl_env_counters *c = c_ra.counters + env_id;
    c->decisions = h->decisions; c->ticks = h->ticks; c->train_ticks = h->train_ticks; c->episodes = h->episode;
    c->err = h->err; c->q_rows = h->q_rows; c->halted = h->halted; c->n_dec_logged = h->n_dec_logged;
    c->n_tick_logged = h->n_tick_logged; c->n_ep_logged = h->n_ep_logged; c->elapsed = h->elapsed;
    c->aborted = h->aborted; c->reserved = 0;
    c->forced_stops = h->forced_stops; c->stop_actions = h->stop_actions; c->arrived_trains = h->arrived_trains; c->reserved2 = 0;
    SFL_UA
    for (int i = 0; i < 6; i++) c->phase_cycles[i] = h->ph[i];
  }
#if SFL_DEV
  g.sync();
  SFL_NU
  for (unsigned o = g.gl * 16u; o < hot_bytes; o += G * 16u) *(int4 *)(gbase + o) = *(const int4 *)(g_smem + stage + o);
#endif
}

}  // namespace sfl
