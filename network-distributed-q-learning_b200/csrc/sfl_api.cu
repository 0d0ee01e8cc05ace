// sfl_api.cu -- kernels + C-ABI (include/switchfl_b200.h) of the B200 SwitchFL backend.
//
// Product build: nvcc -gencode arch=compute_100a,code=sm_100a (see __graft_entry__.build).  There is no
// CPU path in that build.  tests/emul compiles this same file with g++ -DSFL_HOST_EMUL to unit-test the
// per-environment logic where no GPU exists; that library is never loaded by the product package.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <vector>

#include "sfl_core.cuh"

using namespace sfl;

static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, const char *detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}

// ------------------------------------------------------------------------------------------------ backend glue
#ifndef SFL_HOST_EMUL
#include <cuda_runtime.h>
#define CU(call)                                                               \
  do {                                                                         \
    cudaError_t e_ = (call);                                                   \
    if (e_ != cudaSuccess) return fail(SFL_E_CUDA, "CUDA: %s", cudaGetErrorString(e_)); \
  } while (0)
#define CK(call)                                                               \
  do {                                                                         \
    if (call) return fail(SFL_E_CUDA, "CUDA: %s", cudaGetErrorString(cudaGetLastError())); \
  } while (0)
static int dev_alloc(void **p, size_t n) { return cudaMalloc(p, n) == cudaSuccess ? 0 : 1; }
static void dev_free(void *p) { cudaFree(p); }
static int h2d(void *d, const void *h, size_t n, void *s) { return cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, (cudaStream_t)s) != cudaSuccess; }
static int d2h(void *h, const void *d, size_t n, void *s) {
  if (cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, (cudaStream_t)s) != cudaSuccess) return 1;
  return cudaStreamSynchronize((cudaStream_t)s) != cudaSuccess;
}
static int dev_zero(void *d, size_t n, void *s) { return cudaMemsetAsync(d, 0, n, (cudaStream_t)s) != cudaSuccess; }
#else
#define CU(call) do { if (call) return fail(SFL_E_CUDA, "emul: %s", #call); } while (0)
#define CK(call) CU(call)
static int dev_alloc(void **p, size_t n) { *p = malloc(n ? n : 1); return *p == nullptr; }
static void dev_free(void *p) { free(p); }
static int h2d(void *d, const void *h, size_t n, void *) { memcpy(d, h, n); return 0; }
static int d2h(void *h, const void *d, size_t n, void *) { memcpy(h, d, n); return 0; }
static int dev_zero(void *d, size_t n, void *) { memset(d, 0, n); return 0; }
#endif

// every entry point runs on its context's device and leaves the caller's current device as it found it
struct DeviceGuard {
#ifndef SFL_HOST_EMUL
  int prev;
  explicit DeviceGuard(int dev) : prev(-1) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
#else
  explicit DeviceGuard(int) {}
#endif
};

#ifndef SFL_MINB_BIG
#define SFL_MINB_BIG 7                                 // CTAs per SM the large-map (tail in HBM) kernels are compiled for
#endif
#ifndef SFL_WARPS_PER_CTA
#define SFL_WARPS_PER_CTA 4
#endif
#ifndef SFL_MINB_WIDE
#define SFL_MINB_WIDE 6                                // CTAs per SM the learn / greedy kernels for more than 64 trains (NW = 2) are
#endif                                                 // compiled for: 80 registers; at 7 (72) they spill
#define SFL_CTA_THREADS (32 * SFL_WARPS_PER_CTA)
#define SFL_SMEM_BUDGET (56u * 1024u)                  // per CTA, so that four CTAs share an SM

// ------------------------------------------------------------------------------------------------ kernels
struct InitArgs { Layout L; char *state; const sfl_hparams *hp; int n_envs, keep_q, keep_ninter, no_q; };   // no_q: evaluation context

struct InitEnv {          // the env block in HBM, no staging
  const Layout *L;
  char *b;
  SFL_FN EnvHdr *h() const { return (EnvHdr *)b; }
  SFL_FN int4 *tra() const { return (int4 *)(b + L->off_tra); }
  SFL_FN int4 *trb() const { return (int4 *)(b + L->off_trb); }
  SFL_FN SwS *sws() const { return (SwS *)(b + L->off_sws); }
  SFL_FN double *q() const { return (double *)(b + L->off_q); }
};

SFL_FN void env_init(const InitArgs &ia, int env_id, int lane, int lanes) {
  InitEnv e;
  e.L = &ia.L;
  e.b = ia.state + (size_t)env_id * ia.L.env_stride;
  // RailNetwork.reset (rail_network.py:135-149) never clears _train_prev_port / _train_source_port: a reset that continues
  // a run (keep flags set: the next ep_cap segment of learn(), an exploit pause, test()) keeps them like the in-kernel reset
  const int keep_ports = ia.keep_q || ia.keep_ninter;
  for (int t = lane; t < ia.L.T; t += lanes) {
    const int px = keep_ports ? e.trb()[t].x : -1;
    e.tra()[t] = make_int4(-1, 0, 0, 0); e.trb()[t] = make_int4(px, 0xFFFF, 0, 0);
  }
  if (!ia.keep_ninter) for (int s = lane; s < ia.L.S; s += lanes) { SwS z; z.ninter = 0; z.pad = 0; z.eps_pow = 1.0; e.sws()[s] = z; }
  if (!ia.keep_q && !ia.no_q) {
    size_t n = (size_t)ia.L.q_cap * ia.L.q_stride;
    for (size_t i = lane; i < n; i += lanes) e.q()[i] = 0.0;
  }
  if (lane == 0) {
    int q_rows = ia.keep_q ? e.h()->q_rows : 0;
    EnvHdr z;
    memset(&z, 0, sizeof(z));
    z.need_reset = 1; z.pending_fin = -1; z.cur_dec = -1; z.q_rows = q_rows; z.cur_train = -1; z.last_next_sw = -1; z.eps_tag = -1;
    *e.h() = z;
    if (ia.L.T > 64) for (int m = 0; m < 4; m++) ((unsigned long long *)(e.b + sizeof(EnvHdr)))[m] = 0ull;   // word 1 of the train sets
    // the reference's stream restarts with the interaction counters: np.random.default_rng(seed) at the start of learn() (distr_q.py:269)
    if (ia.L.off_rng && !ia.keep_ninter) *(Pcg *)(e.b + ia.L.off_rng) = pcg_seed(ia.hp[env_id].seed);
  }
}

// distr_q.py:299-300 runs __init_q_table at the first episode of EVERY learn() call and ASSIGNS its rows (:156-158, :179-181):
// rows of optimistic-init states that already exist (an earlier learn(), load() or test() created them) are overwritten with
// the initial values; rows that do not exist yet are materialised lazily with the same values on first touch.
struct ReinitArgs { Layout L; RO<int4> sw, port; RO<int8_t> qinit; char *state; const sfl_hparams *hp; int n_envs, pad; };
SFL_FN void q_reinit_slot(const ReinitArgs &a, int env, int slot) {
  double *row = (double *)(a.state + (size_t)env * a.L.env_stride + a.L.off_q) + (size_t)slot * a.L.q_stride;
  const unsigned long long k = *(const unsigned long long *)row;
  if (!k) return;
  const unsigned key = (unsigned)(k - 1ull), per_port = (unsigned)(a.L.NT * 48);
  const int port = (int)(key / per_port);
  const unsigned rem = key - (unsigned)port * per_port;
  const int tgt = (int)(rem / 48u), semb = (int)((rem % 48u) / 3u);
  const int qi = a.qinit[port * a.L.NT + tgt];
  if (qi < 0 || semb == 0) return;
  const int A = a.sw[a.port[port].w].y;
  const double dq = a.hp[env].default_q;
  for (int x = 0; x < A; x++) row[1 + x] = dq;
  row[1 + (qi & 15)] = (qi & 16) ? 1000.0 : 500.0;
}

// Checkpoint export of many tables at once (sfl_export_q_batch): the occupied rows of environment env_lo + j go to rows
// off[j] .. off[j + 1] - 1 of (keys, vals), in slot order -- the order sfl_export_q gives.  A group walks the table G slots
// at a time: a ballot over the key words marks the occupied slots, and a row's place is the running count plus the popcount
// of the ballot bits below its lane.  No atomics, so the output does not depend on scheduling.  Only key words are read to
// find the rows; values are read for occupied rows only.  Rows past off[j + 1] or cap_rows are counted but not written, so
// a table whose row count disagrees with its q_rows cannot write outside its range: found[j] reports it to the host.
struct CompactArgs { Layout L; const char *state; const unsigned long long *off; uint32_t *keys; double *vals; int *found;
                     unsigned long long cap_rows; int env_lo, n; };
#define SFL_COMPACT_UNROLL 4                           // key loads in flight per lane
template <int G> SFL_FN void q_compact_env(const CompactArgs &a, int j, const Grp<G> &g) {
  const Layout &L = a.L;
  const double *q = (const double *)(a.state + (size_t)(a.env_lo + j) * L.env_stride + L.off_q);
  const unsigned long long row0 = a.off[j], end = a.off[j + 1] < a.cap_rows ? a.off[j + 1] : a.cap_rows;
  const unsigned below = (1u << g.gl) - 1u;
  unsigned long long n = 0;
  SFL_NU
  for (int base = 0; base < L.q_cap; base += G * SFL_COMPACT_UNROLL) {
    unsigned long long k[SFL_COMPACT_UNROLL];
    SFL_UA
    for (int u = 0; u < SFL_COMPACT_UNROLL; u++) {
      const int slot = base + u * G + g.gl;
      k[u] = slot < L.q_cap ? *(const unsigned long long *)(q + (size_t)slot * L.q_stride) : 0ull;
    }
    SFL_UA
    for (int u = 0; u < SFL_COMPACT_UNROLL; u++) {
      const unsigned b = g.ballot(k[u] != 0ull);
      const unsigned long long row = row0 + n + (unsigned)popc32(b & below);
      if (k[u] && row < end) {
        const double *src = q + (size_t)(base + u * G + g.gl) * L.q_stride + 1;
        a.keys[row] = (uint32_t)(k[u] - 1ull);
        for (int x = 0; x < L.a_max; x++) a.vals[row * (unsigned)L.a_max + x] = src[x];
      }
      n += (unsigned)popc32(b);
    }
  }
  if (g.gl == 0) a.found[j] = (int)n;
}

// known-answer hooks of the reference's stream: the kernel's own PCG64 / SeedSequence / epsilon functions on caller operands
SFL_FN void pcg_words(const Pcg &g, uint64_t *o) { o[0] = g.s_hi; o[1] = g.s_lo; o[2] = g.i_hi; o[3] = g.i_lo; o[4] = g.has32; o[5] = g.u32; }
SFL_FN void kat_pcg64_one(const uint64_t *gen, const uint64_t *codes, int n_codes, uint64_t *out) {
  Pcg g;
  if (gen[3] & 1ull) { g.s_hi = gen[0]; g.s_lo = gen[1]; g.i_hi = gen[2]; g.i_lo = gen[3]; g.has32 = (unsigned)gen[4]; g.u32 = (unsigned)gen[5]; g.pad0 = g.pad1 = 0u; }
  else g = pcg_seed(gen[1]);
  pcg_words(g, out);
  for (int k = 0; k < n_codes; k++) {
    const uint64_t c = codes[k];
    uint64_t r;
    if (!c) { const double d = pcg_double(g); memcpy(&r, &d, 8); }
    else if (c >> 63) r = (uint64_t)pcg_explore_action(g, (int)(c & 0xFFFFull));
    else r = pcg_bounded(g, c);
    out[6 + k] = r;
  }
  pcg_words(g, out + 6 + n_codes);
}
SFL_FN int kat_explore_one(const double *r) { return eps_explore(r[0], r[1], r[2], (int)r[3], r[4]); }

// flatland's malfunction schedule of every environment (SFL_MALF_REFERENCE): one group per environment, its MT19937 state
// (2 x 624 words) in shared memory.  result[0]: the largest event count, result[1]: 1 = a seed RandomState refuses,
// 2 = min_duration > max_duration with malfunctions on (randint(min, max + 1) refuses)
struct MalfArgs { const sfl_hparams *hp; const unsigned long long *hit_below; int *ev; int *result; int n_envs, T, steps, ev_cap; };
template <int G> SFL_FN void malf_env(const MalfArgs &a, int env, unsigned *mt, const Grp<G> &g, int &max_n, int &flags) {
  const sfl_hparams &h = a.hp[env];
  const unsigned long long hit = a.hit_below[env];
  if (hit && h.malf_min > h.malf_max) { flags |= 2; return; }
  const int n = malf_schedule_env(h.seed, hit, h.malf_min, h.malf_max, a.T, a.steps, a.ev + (size_t)env * a.ev_cap * 3, a.ev_cap,
                                  mt, mt + SFL_MT_N, g);
  if (n < 0) flags |= 1;
  else if (n > max_n) max_n = n;
}
#define SFL_MALF_WARPS 4

#ifndef SFL_HOST_EMUL
__global__ void k_kat_pcg64(const uint64_t *gens, const uint64_t *codes, int n, int n_codes, uint64_t *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) kat_pcg64_one(gens + 6 * (size_t)i, codes + (size_t)i * n_codes, n_codes, out + (size_t)i * (12 + n_codes));
}
__global__ void k_kat_explore(const double *rows, int n, int *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = kat_explore_one(rows + 5 * (size_t)i);
}

__global__ void __launch_bounds__(32 * SFL_MALF_WARPS) k_malf_schedule(const __grid_constant__ MalfArgs a) {
  __shared__ unsigned s_mt[SFL_MALF_WARPS][2 * SFL_MT_N];
  const int w = threadIdx.x >> 5, env = blockIdx.x * SFL_MALF_WARPS + w;
  if (env >= a.n_envs) return;                         // warp-uniform
  const Grp<32> g;
  int max_n = 0, flags = 0;
  malf_env(a, env, s_mt[w], g, max_n, flags);
  if (g.gl == 0) { if (max_n) atomicMax(&a.result[0], max_n); if (flags) atomicOr(&a.result[1], flags); }
}

__global__ void __launch_bounds__(256) k_q_reinit(const __grid_constant__ ReinitArgs a) {
  const size_t n = (size_t)a.n_envs * a.L.q_cap;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    q_reinit_slot(a, (int)(i / a.L.q_cap), (int)(i % a.L.q_cap));
}

// one warp per environment, one warp per CTA: a checkpoint of a few hundred learners still spreads over every SM
__global__ void __launch_bounds__(32) k_q_compact(const __grid_constant__ CompactArgs a) {
  if ((int)blockIdx.x < a.n) q_compact_env(a, (int)blockIdx.x, Grp<32>());
}

__global__ void __launch_bounds__(SFL_CTA_THREADS) k_init(const __grid_constant__ InitArgs ia) {
  int env_id = blockIdx.x * SFL_WARPS_PER_CTA + (threadIdx.x >> 5);
  if (env_id < ia.n_envs) env_init(ia, env_id, threadIdx.x & 31, 32);
}

// G lanes per environment, 32/G environments per warp, SFL_WARPS_PER_CTA warps per CTA.  Dynamic shared memory per
// environment: [hot env state (hot_bytes) | sfl_hparams | Scratch]; the hot state (header, train records, pending
// lists and -- when they fit -- semaphores, rewards and per-switch counters) is staged once per launch and written
// back at the end, so the tick / decision loops touch HBM only for Q rows.
// ROOMY: compiled for 4 instead of 7 CTAs per SM (about 100 instead of 72 registers, no spills) -- for launches of the
// large-map kernels that do not fill the SMs anyway (C3: 1024 one-environment warps per map, +10 %).
// NW: 64-bit words per train set, 2 for maps with more than 64 trains (tail in HBM, 8 / 16 / 32 lanes, no ONE / ROOMY / SQ);
// The full kernels (traces, replay, step protocol, phase clock, learning on the reference's stream) are compiled for at most
// 5 CTAs per SM: no spills.
template <int G, int KIND, bool TH, bool SQ, bool ONE, bool ROOMY = false, int NW = 1>
__global__ void __launch_bounds__(SFL_CTA_THREADS, KIND == K_FULL ? (TH && G != 32 ? 4 : 5) : NW > 1 ? SFL_MINB_WIDE : TH ? (G == 32 ? 7 : 4) : (ROOMY ? 4 : SFL_MINB_BIG))
k_run(const __grid_constant__ KArgs K) {
  const int slot = threadIdx.x / G;                    // environment slot inside the CTA
  const int env_id = blockIdx.x * (blockDim.x / G) + slot;
  env_run<G, KIND, TH, SQ, ONE, NW>(K, env_id, (unsigned)slot * K.ra.env_smem, nullptr);
}

__global__ void k_sum(const sfl_env_counters *c, int n, unsigned long long *out) {
  unsigned long long d = 0, t = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { d += c[i].decisions; t += c[i].ticks; }
  for (int o = 16; o; o >>= 1) { d += __shfl_down_sync(0xffffffffu, d, o); t += __shfl_down_sync(0xffffffffu, t, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, d); atomicAdd(out + 1, t); }
}

// shared-table mode: fold the mean proposed step into the table, clear the accumulators.  dst = src + mean step; src may be
// dst (in place) or the other table of a double-buffered pair (the overlapped schedule: the kernel of the next step reads
// src while this runs).
__global__ void k_shared_apply(const double *src, double *dst, long long *d, int *c, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = c[i];
    double v = src[i];
    if (k) { v += (double)d[i] / 16777216.0 / (double)k; d[i] = 0; c[i] = 0; }
    if (k || src != dst) dst[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ distance map (row F6 / N1)
// d(cell, o) = 0 on the target cell, else 1 + min over the exits h of (cell, o) of d(cell + step(h), h): unit-cost
// shortest paths, i.e. the reverse BFS of flatland_patch/distance_map.py:88-167, as a monotone relaxation to the fixed
// point.  One CTA per target; the table of the target lives in shared memory when it fits (SMEM), else in the output.
template <bool SMEM>
__global__ void __launch_bounds__(512) k_distance_map(const uint16_t *grid, int H, int W, const int *targets, int *out) {
  extern __shared__ int s_dist[];
  const int n = H * W * 4, target = targets[blockIdx.x];
  int *gd = out + (size_t)blockIdx.x * n;
  int *d = SMEM ? s_dist : gd;
  for (int i = threadIdx.x; i < n; i += blockDim.x) d[i] = (i >> 2) == target ? 0 : SFL_INF_DIST;
  __syncthreads();
  for (;;) {
    int changed = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int cell = i >> 2, o = i & 3;
      if (cell == target) continue;
      const unsigned nib = ((unsigned)grid[cell] >> ((3 - o) * 4)) & 0xFu;       // exits of heading o, bit (3 - h)
      if (!nib) continue;
      const int r = cell / W, c = cell - r * W;
      int best = ((volatile int *)d)[i];
#pragma unroll
      for (int h = 0; h < 4; h++) {
        if (!((nib >> (3 - h)) & 1u)) continue;
        const int nr = r + (h == 0 ? -1 : h == 2 ? 1 : 0), nc = c + (h == 1 ? 1 : h == 3 ? -1 : 0);
        if (nr < 0 || nr >= H || nc < 0 || nc >= W) continue;
        const int v = ((volatile int *)d)[(nr * W + nc) * 4 + h];
        if (v < SFL_INF_DIST && v + 1 < best) best = v + 1;
      }
      if (best < ((volatile int *)d)[i]) { d[i] = best; changed = 1; }
    }
    if (!__syncthreads_or(changed)) break;
  }
  if (SMEM) for (int i = threadIdx.x; i < n; i += blockDim.x) gd[i] = d[i];
}

// known-answer hook: the device's TD arithmetic on caller operands (rows of {q, lr, reward, gamma, max_next, bootstrap})
__global__ void k_kat_q_update(const double *in, int n, double *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = td_value(in[6 * i], in[6 * i + 1], in[6 * i + 2], in[6 * i + 3], in[6 * i + 4], in[6 * i + 5] != 0.0);
}

// Evaluation contexts (sfl_config.eval_q): the greedy kernel on the one read-only table (EVQ), compiled like the greedy
// k_run instantiation it stands in for.  A kernel of its own, so that the names of the k_run instantiations stay as they were.
template <int G, bool TH, bool ONE, int NW = 1>
__global__ void __launch_bounds__(SFL_CTA_THREADS, NW > 1 ? SFL_MINB_WIDE : TH ? (G == 32 ? 7 : 4) : SFL_MINB_BIG)
k_eval(const __grid_constant__ KArgs K) {
  const int slot = threadIdx.x / G;
  const int env_id = blockIdx.x * (blockDim.x / G) + slot;
  env_run<G, K_GREEDY, TH, false, ONE, NW, true>(K, env_id, (unsigned)slot * K.ra.env_smem, nullptr);
}

typedef void (*run_kernel_t)(const KArgs);
// `one`: every train has its own lane (T <= G): the production kernels have a single-pass variant for that; the full and
// the shared-table kernels always run the general chunked loops.
template <int G> static run_kernel_t pick_kernel_g(int kind, int th, int sq, int one, int roomy) {
  if (roomy && !th && !sq && kind == K_LEARN && G >= 16)                                 // the only roomy instantiations
    return one ? k_run<(G >= 16 ? G : 32), K_LEARN, false, false, true, true> : k_run<(G >= 16 ? G : 32), K_LEARN, false, false, false, true>;
  if (sq) {                                                                              // shared-table variants: learn / greedy only
    if (kind == K_GREEDY) return th ? k_run<G, K_GREEDY, true, true, false> : k_run<G, K_GREEDY, false, true, false>;
    return th ? k_run<G, K_LEARN, true, true, false> : k_run<G, K_LEARN, false, true, false>;
  }
  if (kind == K_FULL) return th ? k_run<G, K_FULL, true, false, false> : k_run<G, K_FULL, false, false, false>;
  if (kind == K_GREEDY) return th ? (one ? k_run<G, K_GREEDY, true, false, true> : k_run<G, K_GREEDY, true, false, false>)
                                  : (one ? k_run<G, K_GREEDY, false, false, true> : k_run<G, K_GREEDY, false, false, false>);
  return th ? (one ? k_run<G, K_LEARN, true, false, true> : k_run<G, K_LEARN, true, false, false>)
            : (one ? k_run<G, K_LEARN, false, false, true> : k_run<G, K_LEARN, false, false, false>);
}
// more than 64 trains: the tail stays in HBM (choose_hot) and the groups are 8, 16 or 32 lanes wide (sfl_set_lanes)
template <int G> static run_kernel_t pick_wide_g(int kind) {
  return kind == K_FULL ? k_run<G, K_FULL, false, false, false, false, 2>
       : kind == K_GREEDY ? k_run<G, K_GREEDY, false, false, false, false, 2> : k_run<G, K_LEARN, false, false, false, false, 2>;
}
template <int G> static run_kernel_t pick_eval_g(int th, int one) {
  return th ? (one ? k_eval<G, true, true> : k_eval<G, true, false>) : (one ? k_eval<G, false, true> : k_eval<G, false, false>);
}
static run_kernel_t pick_eval(int G, int th, int one, int nw) {
  if (nw > 1) return G == 8 ? k_eval<8, false, false, 2> : G == 16 ? k_eval<16, false, false, 2> : k_eval<32, false, false, 2>;
  switch (G) {
    case 1: return pick_eval_g<1>(th, one);
    case 2: return pick_eval_g<2>(th, one);
    case 4: return pick_eval_g<4>(th, one);
    case 8: return pick_eval_g<8>(th, one);
    case 16: return pick_eval_g<16>(th, one);
    default: return pick_eval_g<32>(th, one);
  }
}
static run_kernel_t pick_kernel(int G, int kind, int th, int sq, int one, int roomy, int nw) {
  if (nw > 1) return G == 8 ? pick_wide_g<8>(kind) : G == 16 ? pick_wide_g<16>(kind) : pick_wide_g<32>(kind);
  switch (G) {
    case 1: return pick_kernel_g<1>(kind, th, sq, one, roomy);
    case 2: return pick_kernel_g<2>(kind, th, sq, one, roomy);
    case 4: return pick_kernel_g<4>(kind, th, sq, one, roomy);
    case 8: return pick_kernel_g<8>(kind, th, sq, one, roomy);
    case 16: return pick_kernel_g<16>(kind, th, sq, one, roomy);
    default: return pick_kernel_g<32>(kind, th, sq, one, roomy);
  }
}
#endif

// ------------------------------------------------------------------------------------------------ context
struct Ctx {
  DevMap m;
  Layout L;
  sfl_config cfg;
  sfl_buffers bufs;
  int phase_clock;     // per-phase cycle counters: instrumented launches use the full kernel
  int bound, device, q_init_on, lanes, sm_count, cta_warps, roomy;        // roomy: -1 automatic, 0 / 1 forced
  unsigned hot_bytes, env_smem, tail_hot;
  void *blob;          // device block holding every map table
  void *sum_buf;       // 2 x u64
  void *malf_buf;      // SFL_MALF_REFERENCE: n_envs x u64 hit_below, then the 2 x i32 result of k_malf_schedule
};

// ------------------------------------------------------------------------------------------------ launch plan
// Which k_run instantiation a launch of `kind` uses and its launch configuration -- shared by sfl_run and
// sfl_describe_launch, so that tests can pin exactly the instantiations the benchmark times.
struct LaunchPlan { int G, th, one, roomy, nw, threads, grid; size_t smem; };
static int plan_launch(const Ctx *c, int kind, LaunchPlan *lp) {
  const int G = c->lanes;
  // Warps per CTA: the kernels are compiled for at most SFL_WARPS_PER_CTA; small launches use smaller CTAs so that the
  // CTAs spread evenly over the SMs (1024 one-env warps as 256 CTAs leave SMs with 8 or 4 warps; as 1024 CTAs with 7).
  int cta_warps = c->cta_warps;
  const long warps = ((long)c->cfg.n_envs * G + 31) / 32;
  if (cta_warps <= 0) {
    cta_warps = SFL_WARPS_PER_CTA;
    while (cta_warps > 1 && warps / cta_warps < 8L * c->sm_count) cta_warps /= 2;      // fewer than 8 CTAs per SM: halve
  }
  int threads = 32 * cta_warps;                        // then shrink the CTA until its environments fit shared memory
  while (threads > 32 && (size_t)c->env_smem * (threads / G) > SFL_SMEM_BUDGET) threads /= 2;
  const int envs_per_cta = threads / G;
  lp->smem = (size_t)c->env_smem * envs_per_cta;
  if (lp->smem > 227u * 1024u) return fail(SFL_E_ARG, "environment state does not fit shared memory with this many lanes per env: use more lanes%s");
  lp->G = G; lp->threads = threads; lp->grid = (c->cfg.n_envs + envs_per_cta - 1) / envs_per_cta;
  lp->th = (int)c->tail_hot; lp->one = c->L.T <= G && !c->cfg.shared_q && kind != K_FULL;
  lp->nw = c->L.T > 64 ? 2 : 1;
  int roomy = c->roomy >= 0 ? c->roomy : (warps <= 16L * c->sm_count);                   // one wave even at 4 CTAs per SM
  lp->roomy = roomy && !lp->th && !c->cfg.shared_q && kind == K_LEARN && G >= 16 && lp->nw == 1;   // the only roomy instantiations
  return 0;
}


// Shared-memory staging plan for c->lanes lanes per environment: the whole non-Q state (header, train records, pending
// lists, semaphores, rewards, per-switch counters) when that still leaves room for 16 warps per SM,
// else only header + train records + pending lists (semaphores, rewards and counters then stay in HBM / L2).
// More than 64 trains: always the latter -- the whole state fits only for the smallest maps, and the wide kernels are
// built for the tail in HBM only.
static int choose_hot(Ctx *c) {
  const unsigned fixed = (unsigned)sizeof(sfl_hparams) + scratch_bytes(c->L.T);
  const unsigned per_warp = 32u / (unsigned)c->lanes;
  if (c->L.T <= 64 && (size_t)(c->L.off_q + fixed) * per_warp <= 14u * 1024u) { c->tail_hot = 1; c->hot_bytes = c->L.off_q; }   // >= 16 warps per SM
  else { c->tail_hot = 0; c->hot_bytes = c->L.off_pend; }
  c->env_smem = c->hot_bytes + fixed + (c->tail_hot ? 0u : ((unsigned)c->L.NP + 15u) / 16u * 16u);   // + holder bytes of the semaphores
  return (size_t)c->env_smem * per_warp > 227u * 1024u;
}

static unsigned align_up(unsigned v, unsigned a) { return (v + a - 1) / a * a; }

static int make_layout(const sfl_map_desc *map, const sfl_config *cfg, Layout *L, int *a_max_out) {
  if (!map || !cfg) return fail(SFL_E_ARG, "null argument%s");
  if (map->T < 1 || map->T > SFL_MAX_T) return fail(SFL_E_ARG, "T must be in 1..128%s");
  if (map->S < 1 || map->S > 4095) return fail(SFL_E_ARG, "S must be in 1..4095%s");
  if (map->NP > 32767) return fail(SFL_E_ARG, "too many ports%s");
  if ((int64_t)(map->H + 2) * (map->W + 2) >= (1 << 28)) return fail(SFL_E_ARG, "grid too large%s");
  if (cfg->q_cap < 2 || (cfg->q_cap & (cfg->q_cap - 1))) return fail(SFL_E_ARG, "q_cap must be a power of two%s");
  if (cfg->pend_cap < 1 || cfg->pend_cap > 64 || cfg->n_envs < 1) return fail(SFL_E_ARG, "bad pend_cap / n_envs%s");
  int a_max = 0;
  for (int s = 0; s < map->S; s++) { if (map->sw_A[s] > a_max) a_max = map->sw_A[s]; if (map->sw_P[s] > 4) return fail(SFL_E_ARG, "P > 4%s"); }
  if (a_max > 15) return fail(SFL_E_ARG, "A > 15%s");
  if ((uint64_t)map->NP * map->NT * 48ull >= 0xFFFFFFFFull) return fail(SFL_E_ARG, "state index does not fit 32 bits%s");
  if (cfg->rng != SFL_RNG_PHILOX && cfg->rng != SFL_RNG_REFERENCE) return fail(SFL_E_ARG, "rng must be SFL_RNG_PHILOX (0) or SFL_RNG_REFERENCE (1)%s");
  if (cfg->malf_rng != SFL_MALF_PHILOX && cfg->malf_rng != SFL_MALF_REFERENCE)
    return fail(SFL_E_ARG, "malf_rng must be SFL_MALF_PHILOX (0) or SFL_MALF_REFERENCE (1)%s");
  if (cfg->eval_q != 0 && cfg->eval_q != 1) return fail(SFL_E_ARG, "eval_q must be 0 or 1%s");
  memset(L, 0, sizeof(*L));
  L->T = map->T; L->S = map->S; L->NP = map->NP; L->NT = map->NT; L->a_max = a_max; L->q_cap = cfg->q_cap;
  L->q_stride = 1 + a_max; L->pend_cap = cfg->pend_cap;
  unsigned T = (unsigned)map->T;
  unsigned o = (unsigned)sizeof(EnvHdr) + (T > 64 ? 4u * 8u : 0u);                   // + word 1 of the four train sets
  if (cfg->rng == SFL_RNG_REFERENCE) { L->off_rng = o; o += SFL_PCG_BYTES; }          // + the reference's stream (none with Philox)
  o = align_up(o, 16);
#define PUT(field, bytes) L->field = o; o = align_up(o + (unsigned)(bytes), 16)
  PUT(off_tra, 16 * T); PUT(off_trb, 16 * T); PUT(off_pend, 8 * T * cfg->pend_cap);
  PUT(off_sem, 16 * (unsigned)map->NP); PUT(off_rewards, 4 * (unsigned)map->S * T); PUT(off_sws, 16 * (unsigned)map->S);
#undef PUT
  L->off_q = o;
  // an evaluation context has no Q region: q_cap rows are the one table in sfl_buffers.eval_q
  const unsigned long long q_bytes = cfg->eval_q ? 0ull : (unsigned long long)cfg->q_cap * L->q_stride * 8ull;
  L->env_stride = ((unsigned long long)o + q_bytes + 127ull) / 128ull * 128ull;
  *a_max_out = a_max;
  return SFL_OK;
}

// The hash image of a Q table of L.q_cap rows (distr_q.py:510-527 load): row r at the slot the kernels' probe finds key r
// at (q_row / eval_action: same hash, linear probing); a repeated key overwrites its row.  Returns the distinct keys.
// n_rows < q_cap, so that an empty slot ends every probe.
static int q_image(const Layout &L, const uint32_t *keys_host, const double *vals_host, int n_rows, std::vector<double> &img) {
  img.assign((size_t)L.q_cap * L.q_stride, 0.0);
  const unsigned mask = (unsigned)L.q_cap - 1u;
  int distinct = 0;
  for (int r = 0; r < n_rows; r++) {
    unsigned key = keys_host[r];
    unsigned i = (key * 2654435761u) >> 7;
    for (;;) {
      i &= mask;
      unsigned long long k;
      memcpy(&k, &img[(size_t)i * L.q_stride], 8);
      if (k == 0) distinct++;
      if (k == 0 || k == (unsigned long long)key + 1ull) break;
      i++;
    }
    unsigned long long k = (unsigned long long)key + 1ull;
    memcpy(&img[(size_t)i * L.q_stride], &k, 8);
    for (int a = 0; a < L.a_max; a++) img[(size_t)i * L.q_stride + 1 + a] = vals_host[(size_t)r * L.a_max + a];
  }
  return distinct;
}

extern "C" {

int sfl_abi_version(void) { return SFL_ABI_VERSION; }

int sfl_distance_map(const uint16_t *grid, int32_t H, int32_t W, const int32_t *target_cells, int32_t n_targets, int32_t *dist, int device) {
  if (!grid || !target_cells || !dist || H < 1 || W < 1 || n_targets < 0) return fail(SFL_E_ARG, "bad argument%s");
  const size_t n = (size_t)H * W * 4;
  for (int k = 0; k < n_targets; k++) if (target_cells[k] < 0 || target_cells[k] >= H * W) return fail(SFL_E_ARG, "target outside the grid%s");
  if (!n_targets) return SFL_OK;
#ifndef SFL_HOST_EMUL
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SFL_E_CUDA, "no CUDA device: this library has no CPU path%s");
  DeviceGuard guard(device);
  uint16_t *dg = nullptr; int *dt = nullptr, *dd = nullptr;
  if (cudaMalloc(&dg, (size_t)H * W * 2) != cudaSuccess || cudaMalloc(&dt, (size_t)n_targets * 4) != cudaSuccess ||
      cudaMalloc(&dd, n * 4 * n_targets) != cudaSuccess) { cudaFree(dg); cudaFree(dt); cudaFree(dd); return fail(SFL_E_CUDA, "device alloc failed%s"); }
  int rc = SFL_OK;
  do {
    if (cudaMemcpy(dg, grid, (size_t)H * W * 2, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(dt, target_cells, (size_t)n_targets * 4, cudaMemcpyHostToDevice) != cudaSuccess) { rc = fail(SFL_E_CUDA, "upload failed%s"); break; }
    const size_t smem = n * 4;
    if (smem <= 200u * 1024u) {
      if (cudaFuncSetAttribute(k_distance_map<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { rc = fail(SFL_E_CUDA, "smem attribute%s"); break; }
      k_distance_map<true><<<n_targets, 512, smem>>>(dg, H, W, dt, dd);
    } else {
      k_distance_map<false><<<n_targets, 512, 0>>>(dg, H, W, dt, dd);
    }
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(dist, dd, n * 4 * n_targets, cudaMemcpyDeviceToHost) != cudaSuccess) rc = fail(SFL_E_CUDA, "distance map kernel failed%s");
  } while (0);
  cudaFree(dg); cudaFree(dt); cudaFree(dd);
  return rc;
#else
  (void)device;
  for (int k = 0; k < n_targets; k++) {                                  // the same relaxation, one thread
    int *d = dist + (size_t)k * n;
    const int target = target_cells[k];
    for (size_t i = 0; i < n; i++) d[i] = (int)(i >> 2) == target ? 0 : SFL_INF_DIST;
    for (int changed = 1; changed;) {
      changed = 0;
      for (int i = 0; i < (int)n; i++) {
        const int cell = i >> 2, o = i & 3;
        if (cell == target) continue;
        const unsigned nib = ((unsigned)grid[cell] >> ((3 - o) * 4)) & 0xFu;
        const int r = cell / W, c = cell - r * W;
        for (int h = 0; h < 4; h++) {
          if (!((nib >> (3 - h)) & 1u)) continue;
          const int nr = r + (h == 0 ? -1 : h == 2 ? 1 : 0), nc = c + (h == 1 ? 1 : h == 3 ? -1 : 0);
          if (nr < 0 || nr >= H || nc < 0 || nc >= W) continue;
          const int v = d[(nr * W + nc) * 4 + h];
          if (v < SFL_INF_DIST && v + 1 < d[i]) { d[i] = v + 1; changed = 1; }
        }
      }
    }
  }
  return SFL_OK;
#endif
}
const char *sfl_last_error(void) { return g_err; }

int sfl_kat_q_update(const double *operands, int32_t n, double *out, int device) {
  if (!operands || !out || n < 0) return fail(SFL_E_ARG, "bad argument%s");
  if (!n) return SFL_OK;
#ifndef SFL_HOST_EMUL
  int ndev = 0, prev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SFL_E_CUDA, "no CUDA device: this library has no CPU path%s");
  cudaGetDevice(&prev);
  CU(cudaSetDevice(device));
  double *din = nullptr, *dout = nullptr;
  int rc = SFL_OK;
  if (cudaMalloc(&din, (size_t)n * 48) != cudaSuccess || cudaMalloc(&dout, (size_t)n * 8) != cudaSuccess) rc = fail(SFL_E_CUDA, "device alloc failed%s");
  else if (cudaMemcpy(din, operands, (size_t)n * 48, cudaMemcpyHostToDevice) != cudaSuccess) rc = fail(SFL_E_CUDA, "upload failed%s");
  else {
    k_kat_q_update<<<(n + 127) / 128, 128>>>(din, n, dout);
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = fail(SFL_E_CUDA, "kat kernel failed%s");
  }
  cudaFree(din); cudaFree(dout);
  cudaSetDevice(prev);
  return rc;
#else
  (void)device;
  for (int i = 0; i < n; i++) out[i] = td_value(operands[6 * i], operands[6 * i + 1], operands[6 * i + 2], operands[6 * i + 3], operands[6 * i + 4], operands[6 * i + 5] != 0.0);
  return SFL_OK;
#endif
}

// copy in, run the known-answer kernel, copy out (the host build runs the same functions in a loop)
#ifndef SFL_HOST_EMUL
struct KatBufs {
  void *p[3] = {nullptr, nullptr, nullptr};
  ~KatBufs() { for (void *q : p) cudaFree(q); }
};
#endif

int sfl_kat_pcg64(const uint64_t *gens, const uint64_t *codes, int32_t n, int32_t n_codes, uint64_t *out, int device) {
  if (!gens || !out || n < 0 || n_codes < 0 || (n_codes && !codes)) return fail(SFL_E_ARG, "bad argument%s");
  for (size_t i = 0; i < (size_t)n * n_codes; i++)
    if (!(codes[i] >> 63) && codes[i] > 0x100000000ull) return fail(SFL_E_ARG, "a bounded draw's range must be at most 2^32%s");
  if (!n) return SFL_OK;
  const size_t gb = (size_t)n * 48, cb = (size_t)n * n_codes * 8 + 8, ob = (size_t)n * (12 + n_codes) * 8;
#ifndef SFL_HOST_EMUL
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SFL_E_CUDA, "no CUDA device: this library has no CPU path%s");
  DeviceGuard guard(device);
  KatBufs b;
  CU(cudaMalloc(&b.p[0], gb)); CU(cudaMalloc(&b.p[1], cb)); CU(cudaMalloc(&b.p[2], ob));
  CU(cudaMemcpy(b.p[0], gens, gb, cudaMemcpyHostToDevice));
  if (n_codes) CU(cudaMemcpy(b.p[1], codes, cb - 8, cudaMemcpyHostToDevice));
  k_kat_pcg64<<<(n + 127) / 128, 128>>>((const uint64_t *)b.p[0], (const uint64_t *)b.p[1], n, n_codes, (uint64_t *)b.p[2]);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, b.p[2], ob, cudaMemcpyDeviceToHost));
#else
  (void)device; (void)gb; (void)cb; (void)ob;
  for (int i = 0; i < n; i++) kat_pcg64_one(gens + 6 * (size_t)i, codes + (size_t)i * n_codes, n_codes, out + (size_t)i * (12 + n_codes));
#endif
  return SFL_OK;
}

int sfl_kat_explore(const double *rows, int32_t n, int32_t *out, int device) {
  if (!rows || !out || n < 0) return fail(SFL_E_ARG, "bad argument%s");
  for (int i = 0; i < n; i++) if (!(rows[5 * i + 3] >= 0.0 && rows[5 * i + 3] < 2147483648.0)) return fail(SFL_E_ARG, "n must be in 0..2^31-1%s");
  if (!n) return SFL_OK;
#ifndef SFL_HOST_EMUL
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(SFL_E_CUDA, "no CUDA device: this library has no CPU path%s");
  DeviceGuard guard(device);
  KatBufs b;
  CU(cudaMalloc(&b.p[0], (size_t)n * 40)); CU(cudaMalloc(&b.p[1], (size_t)n * 4));
  CU(cudaMemcpy(b.p[0], rows, (size_t)n * 40, cudaMemcpyHostToDevice));
  k_kat_explore<<<(n + 127) / 128, 128>>>((const double *)b.p[0], n, (int *)b.p[1]);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, b.p[1], (size_t)n * 4, cudaMemcpyDeviceToHost));
#else
  (void)device;
  for (int i = 0; i < n; i++) out[i] = kat_explore_one(rows + 5 * (size_t)i);
#endif
  return SFL_OK;
}

int sfl_query_sizes(const sfl_map_desc *map, const sfl_config *cfg, sfl_sizes *out) {
  Layout L; int a_max;
  int rc = make_layout(map, cfg, &L, &a_max);
  if (rc) return rc;
  if (!out) return fail(SFL_E_ARG, "null out%s");
  uint64_t B = (uint64_t)cfg->n_envs;
  out->env_stride = L.env_stride;
  out->state_bytes = B * L.env_stride;
  out->hparams_bytes = B * sizeof(sfl_hparams);
  out->counters_bytes = B * sizeof(sfl_env_counters);
  out->step_out_bytes = B * sizeof(sfl_step_rec);
  const uint64_t cells = cfg->shared_q ? (uint64_t)map->NP * map->NT * 48ull * (uint64_t)a_max : 0;
  out->shared_q_bytes = cells * 8ull; out->shared_d_bytes = cells * 8ull; out->shared_c_bytes = cells * 4ull;
  out->trace_dec_bytes = B * (uint64_t)cfg->dec_cap * sizeof(sfl_dec_rec);
  out->trace_tick_bytes = B * (uint64_t)cfg->tick_cap * map->T * sizeof(sfl_tick_rec);
  out->trace_sem_bytes = cfg->trace_sem ? B * (uint64_t)cfg->dec_cap * map->NP * 16ull : 0;
  out->ep_log_bytes = B * (uint64_t)cfg->ep_cap * sizeof(sfl_ep_rec);
  out->ep_delay_bytes = B * (uint64_t)cfg->ep_cap * map->T * 4ull;
  out->replay_act_bytes = B * (uint64_t)cfg->act_cap;
  out->replay_ev_bytes = B * (uint64_t)cfg->ev_cap * 12ull;
  out->q_stride = L.q_stride;
  out->a_max = a_max;
  out->rng_offset = L.off_rng;
  out->eval_q_bytes = cfg->eval_q ? (uint64_t)cfg->q_cap * L.q_stride * 8ull : 0;
  return SFL_OK;
}

// flatland rail.check_action_on_agent for every (cell, heading, action), SURVEY.md Appendix B (row F1)
static uint16_t move_entry(unsigned v, int dir) {
  if (!v) return 0;
  unsigned nib = (v >> ((3 - dir) * 4)) & 0xFu;
  int n = __builtin_popcount(nib);
  uint16_t e = 0x8000u;
  for (int a = 0; a <= 4; a++) {
    int nd = dir, valid = -1;
    if (a == A_LEFT) { nd = dir - 1; if (n <= 1) valid = 0; }
    else if (a == A_RIGHT) { nd = dir + 1; if (n <= 1) valid = 0; }
    nd &= 3;
    if (a == A_FWD && n == 1) { nd = 3 - (31 - __builtin_clz(nib)); valid = 1; }
    if (valid < 0) valid = (nib >> (3 - nd)) & 1;
    e |= (uint16_t)((valid | (nd << 1)) << (3 * a));
  }
  return e;
}

int sfl_create(const sfl_map_desc *map, const sfl_config *cfg, int device, void **ctx_out) {
  if (!ctx_out) return fail(SFL_E_ARG, "null ctx%s");
  Layout L; int a_max;
  int rc = make_layout(map, cfg, &L, &a_max);
  if (rc) return rc;
  if (cfg->shared_q && map->T > 64) return fail(SFL_E_ARG, "shared-table mode supports at most 64 trains%s");
  if (cfg->shared_q && cfg->rng == SFL_RNG_REFERENCE)
    return fail(SFL_E_ARG, "the reference's random stream (SFL_RNG_REFERENCE) has no shared-table mode: the reference keeps one table and one stream per learner%s");
  if (cfg->malf_rng == SFL_MALF_REFERENCE && cfg->shared_q)
    return fail(SFL_E_ARG, "flatland's malfunction stream (SFL_MALF_REFERENCE) has no shared-table mode%s");
  if (cfg->malf_rng == SFL_MALF_REFERENCE && cfg->ev_cap < 1)
    return fail(SFL_E_ARG, "flatland's malfunction stream (SFL_MALF_REFERENCE) needs ev_cap >= 1: the schedule goes to replay_ev%s");
  if (cfg->eval_q && cfg->shared_q)
    return fail(SFL_E_ARG, "an evaluation context (eval_q) has no shared-table mode: shared-table mode is for learning%s");
  if (cfg->eval_q && cfg->rng == SFL_RNG_REFERENCE)
    return fail(SFL_E_ARG, "an evaluation context (eval_q) runs greedy rollouts only, which draw nothing from the reference's epsilon-greedy stream (SFL_RNG_REFERENCE)%s");
  const int H = map->H, W = map->W, Hp = H + 2, Wp = W + 2, T = map->T, NT = map->NT, S = map->S, NP = map->NP, NA = map->NA;
  // every transition must lead to a rail cell inside the grid (flatland maps are consistent); the device relies on it
  for (int r = 0; r < H; r++) for (int cc = 0; cc < W; cc++) {
    unsigned v = map->grid[r * W + cc];
    for (int x = 0; x < 4; x++) {
      if (!(((v >> 12) | (v >> 8) | (v >> 4) | v) & (8u >> x))) continue;
      int nr = r + (x == 0 ? -1 : x == 2 ? 1 : 0), nc = cc + (x == 1 ? 1 : x == 3 ? -1 : 0);
      if (nr < 0 || nr >= H || nc < 0 || nc >= W || !map->grid[nr * W + nc]) return fail(SFL_E_ARG, "inconsistent map: a transition leads off the rails%s");
    }
  }
  int sm_count = 148;
#ifndef SFL_HOST_EMUL
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(SFL_E_CUDA, "no CUDA device: this library has no CPU path%s");
  if (device < 0 || device >= ndev) return fail(SFL_E_ARG, "no such CUDA device%s");
  CU(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
#endif
  DeviceGuard dg(device);
  Ctx *c = new (std::nothrow) Ctx();
  if (!c) return fail(SFL_E_NOMEM, "host alloc%s");
  c->L = L; c->cfg = *cfg; c->bound = 0; c->device = device; c->q_init_on = 0; c->cta_warps = 0; c->roomy = -1; c->phase_clock = 0; c->blob = nullptr; c->sum_buf = nullptr; c->malf_buf = nullptr; c->sm_count = sm_count;
  memset(&c->bufs, 0, sizeof(c->bufs));
  auto pcell = [&](int cell) { return cell < 0 ? -1 : (cell / W + 1) * Wp + (cell % W + 1); };
  // ---- pack every table into one host image, 16-byte aligned sections
  std::vector<unsigned char> img;
  auto section = [&](size_t bytes) { size_t o = (img.size() + 15) / 16 * 16; img.resize(o + bytes, 0); return o; };
  size_t o_move = section(8ull * Hp * Wp), o_csw = section(2ull * Hp * Wp), o_sw = section(16ull * S), o_port = section(16ull * NP);
  size_t o_pexit = section(16ull * NP), o_act = section(16ull * (NA ? NA : 1)), o_t0 = section(16ull * T), o_t1 = section(16ull * T);
  size_t o_idl = section(4ull * T), o_dist = section(16ull * NT * Hp * Wp), o_qi = section((size_t)NP * NT);
  uint16_t *move = (uint16_t *)&img[o_move]; int16_t *csw = (int16_t *)&img[o_csw];
  for (int i = 0; i < Hp * Wp; i++) csw[i] = -1;
  for (int r = 0; r < H; r++) for (int cc = 0; cc < W; cc++) {
    int pc = (r + 1) * Wp + cc + 1;
    for (int d = 0; d < 4; d++) move[pc * 4 + d] = move_entry(map->grid[r * W + cc], d);
    csw[pc] = (int16_t)map->cell_switch[r * W + cc];
  }
  int4 *sw = (int4 *)&img[o_sw];
  for (int s = 0; s < S; s++) sw[s] = make_int4(map->sw_P[s], map->sw_A[s], map->sw_port0[s], map->sw_act0[s]);
  int4 *port = (int4 *)&img[o_port], *pexit = (int4 *)&img[o_pexit];
  for (int s = 0; s < S; s++)
    for (int p = map->sw_port0[s]; p < map->sw_port0[s + 1]; p++) {
      port[p] = make_int4(map->port_nbr[p], map->port_dist[p], map->port_n_intra[p] == 1 ? map->port_intra0[p] : -1, s);
      int ex[3] = {0, 0, 0}, n = 0;
      for (int a = map->sw_act0[s]; a < map->sw_act0[s + 1]; a++)
        if (map->sw_port0[s] + map->act_in[a] == p) {
          if (n >= 3) { delete c; return fail(SFL_E_ARG, "more than 3 exits from one port%s"); }
          ex[n++] = (a - map->sw_act0[s]) | (map->act_out[a] << 4) | (map->act_move[a] << 8);
        }
      pexit[p] = make_int4(n, ex[0], ex[1], ex[2]);
    }
  int4 *act = (int4 *)&img[o_act];
  for (int a = 0; a < NA; a++) act[a] = make_int4(map->act_in[a], map->act_out[a], map->act_move[a], 0);
  int4 *t0 = (int4 *)&img[o_t0], *t1 = (int4 *)&img[o_t1]; int *idl = (int *)&img[o_idl];
  for (int t = 0; t < T; t++) {
    t0[t] = make_int4(pcell(map->init_cell[t]), map->init_dir[t], pcell(map->target_cell[t]), map->tgt_index[t]);
    t1[t] = make_int4(map->ed[t], map->la[t], map->first_port[t], map->first_dist[t]);
    idl[t] = map->init_delay[t];
  }
  int *dist = (int *)&img[o_dist];
  for (size_t i = 0; i < (size_t)NT * Hp * Wp * 4; i++) dist[i] = SFL_INF_DIST;
  for (int k = 0; k < NT; k++) for (int r = 0; r < H; r++) for (int cc = 0; cc < W; cc++) for (int d = 0; d < 4; d++)
    dist[((size_t)k * Hp * Wp + (r + 1) * Wp + cc + 1) * 4 + d] = map->dist[(((size_t)k * H + r) * W + cc) * 4 + d];
  int8_t *qi = (int8_t *)&img[o_qi];
  for (int i = 0; i < NP * NT; i++) qi[i] = map->qinit_act[i] < 0 ? (int8_t)-1 : (int8_t)(map->qinit_act[i] | (map->qinit_final[i] ? 16 : 0));
  if (dev_alloc(&c->blob, img.size()) || dev_alloc(&c->sum_buf, 16) ||
      (cfg->malf_rng == SFL_MALF_REFERENCE && dev_alloc(&c->malf_buf, (size_t)cfg->n_envs * 8 + 8))) {
    sfl_destroy(c); return fail(SFL_E_CUDA, "device alloc of map constants failed%s");
  }
  if (h2d(c->blob, img.data(), img.size(), nullptr)) { sfl_destroy(c); return fail(SFL_E_CUDA, "upload of map constants failed%s"); }
#ifndef SFL_HOST_EMUL
  if (cudaDeviceSynchronize() != cudaSuccess) { sfl_destroy(c); return fail(SFL_E_CUDA, "upload of map constants failed%s"); }
#endif
  char *b = (char *)c->blob;
  DevMap &m = c->m;
  m.H = H; m.W = W; m.Hp = Hp; m.Wp = Wp; m.S = S; m.NP = NP; m.NA = NA; m.T = T; m.NT = NT; m.max_episode_steps = map->max_episode_steps;
  m.a_max = a_max; m.pad0 = 0;
  m.move.p = (const uint16_t *)(b + o_move); m.cell_switch.p = (const int16_t *)(b + o_csw); m.sw.p = (const int4 *)(b + o_sw);
  m.port.p = (const int4 *)(b + o_port); m.pexit.p = (const int4 *)(b + o_pexit); m.act.p = (const int4 *)(b + o_act);
  m.train0.p = (const int4 *)(b + o_t0); m.train1.p = (const int4 *)(b + o_t1); m.init_delay.p = (const int *)(b + o_idl);
  m.dist.p = (const int *)(b + o_dist); m.qinit.p = (const int8_t *)(b + o_qi);
  c->lanes = 32;
  choose_hot(c);
  // Lanes per environment, from measurements on B200 (DESIGN.md section 4): wide enough that one pass covers the
  // trains (lane = train), and wide enough that the batch still fills ~3.5 warps per SM scheduler -- below that the
  // serial per-environment chains cannot hide their own latency; narrower groups share one instruction stream
  // between the 32/G environments of a warp.
  {
    int g_trains = 1;
    while (g_trains < T && g_trains < 32) g_trains *= 2;
    const long warps_wanted = (long)sm_count * 13;                   // 2048 warps on 148 SMs qualify
    int g_warps = 1;
    while (g_warps < 32 && (long)cfg->n_envs * g_warps / 32 < warps_wanted) g_warps *= 2;
    int G = g_trains > g_warps ? g_trains : g_warps;
    c->lanes = G;
    while (choose_hot(c) && G < 32) { G *= 2; c->lanes = G; }
  }
  *ctx_out = c;
  return SFL_OK;
}

int sfl_destroy(void *ctx) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return SFL_OK;
  DeviceGuard dg(c->device);
  if (c->blob) dev_free(c->blob);
  if (c->sum_buf) dev_free(c->sum_buf);
  if (c->malf_buf) dev_free(c->malf_buf);
  delete c;
  return SFL_OK;
}

int sfl_bind(void *ctx, const sfl_buffers *bufs) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !bufs) return fail(SFL_E_ARG, "null argument%s");
  if (!bufs->state || !bufs->hparams || !bufs->counters) return fail(SFL_E_ARG, "state, hparams and counters are mandatory%s");
  if (c->cfg.dec_cap > 0 && !bufs->trace_dec) return fail(SFL_E_ARG, "dec_cap > 0 needs trace_dec%s");
  if (c->cfg.tick_cap > 0 && !bufs->trace_tick) return fail(SFL_E_ARG, "tick_cap > 0 needs trace_tick%s");
  if (c->cfg.shared_q && (!bufs->shared_q || !bufs->shared_d || !bufs->shared_c)) return fail(SFL_E_ARG, "shared_q needs the three shared buffers%s");
  if (c->cfg.eval_q && !bufs->eval_q) return fail(SFL_E_ARG, "an evaluation context (eval_q) needs the eval_q buffer%s");
  c->bufs = *bufs;
  c->bound = 1;
  return SFL_OK;
}

int sfl_set_lanes(void *ctx, int lanes) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (lanes != 1 && lanes != 2 && lanes != 4 && lanes != 8 && lanes != 16 && lanes != 32) return fail(SFL_E_ARG, "lanes must be 1, 2, 4, 8, 16 or 32%s");
  if (c->L.T > 64 && lanes < 8) return fail(SFL_E_ARG, "maps with more than 64 trains run on 8, 16 or 32 lanes%s");
  int old = c->lanes;
  c->lanes = lanes;
  if (choose_hot(c)) { c->lanes = old; choose_hot(c); return fail(SFL_E_ARG, "one warp of environments does not fit shared memory with this few lanes per env%s"); }
  return SFL_OK;
}

int sfl_set_cta_warps(void *ctx, int warps) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (warps != 0 && warps != 1 && warps != 2 && warps != 4) return fail(SFL_E_ARG, "warps per CTA must be 0 (automatic), 1, 2 or 4%s");
  c->cta_warps = warps;
  return SFL_OK;
}

int sfl_set_roomy(void *ctx, int roomy) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (roomy < -1 || roomy > 1) return fail(SFL_E_ARG, "roomy must be -1 (automatic), 0 or 1%s");
  c->roomy = roomy;
  return SFL_OK;
}

int sfl_set_phase_clock(void *ctx, int on) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (on && c->cfg.shared_q) return fail(SFL_E_ARG, "shared-table mode has no instrumented kernel%s");
  if (on && c->cfg.eval_q) return fail(SFL_E_ARG, "an evaluation context (eval_q) has no instrumented kernel%s");
  c->phase_clock = on ? 1 : 0;
  return SFL_OK;
}

int sfl_describe_launch(void *ctx, int mode, int traced, char *buf, int cap) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !buf || cap < 1) return fail(SFL_E_ARG, "null argument%s");
  const int trace = traced || mode == SFL_MODE_STEP || mode == SFL_MODE_REPLAY || c->phase_clock ||
                    (mode == SFL_MODE_LEARN && (c->cfg.rng || c->cfg.malf_rng));
  const int kind = trace ? K_FULL : (mode == SFL_MODE_GREEDY ? K_GREEDY : K_LEARN);
  LaunchPlan lp;
  if (plan_launch(c, kind, &lp)) return SFL_E_ARG;
  if (c->cfg.eval_q) {                                 // the only kernel of an evaluation context (sfl_run refuses the rest)
    if (kind != K_GREEDY) return fail(SFL_E_ARG, "an evaluation context (eval_q) runs SFL_MODE_GREEDY only, without traces or the phase clock%s");
    snprintf(buf, (size_t)cap, "k_eval<G=%d,KIND=greedy,TH=%d,SQ=0,ONE=%d,ROOMY=0%s,EVQ=1> grid=%d block=%d smem=%zu", lp.G, lp.th, lp.one,
             lp.nw > 1 ? ",NW=2" : "", lp.grid, lp.threads, lp.smem);
    return SFL_OK;
  }
  static const char *kinds[] = {"learn", "greedy", "full"};
  snprintf(buf, (size_t)cap, "k_run<G=%d,KIND=%s,TH=%d,SQ=%d,ONE=%d,ROOMY=%d%s> grid=%d block=%d smem=%zu", lp.G, kinds[kind], lp.th,
           c->cfg.shared_q ? 1 : 0, lp.one, lp.roomy, lp.nw > 1 ? ",NW=2" : "", lp.grid, lp.threads, lp.smem);
  return SFL_OK;
}

int sfl_get_lanes(void *ctx) {
  Ctx *c = (Ctx *)ctx;
  return c ? c->lanes : SFL_E_ARG;
}

int sfl_reset(void *ctx, int keep, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (!c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  InitArgs ia; ia.L = c->L; ia.state = (char *)c->bufs.state; ia.hp = (const sfl_hparams *)c->bufs.hparams; ia.n_envs = c->cfg.n_envs; ia.keep_q = keep & 1; ia.keep_ninter = (keep >> 1) & 1; ia.no_q = c->cfg.eval_q;
  CK(dev_zero(c->bufs.counters, (size_t)c->cfg.n_envs * sizeof(sfl_env_counters), stream));
#ifndef SFL_HOST_EMUL
  int grid = (c->cfg.n_envs + SFL_WARPS_PER_CTA - 1) / SFL_WARPS_PER_CTA;
  k_init<<<grid, SFL_CTA_THREADS, 0, (cudaStream_t)stream>>>(ia);
  CU(cudaGetLastError());
#else
  for (int i = 0; i < c->cfg.n_envs; i++) env_init(ia, i, 0, 1);
#endif
  return SFL_OK;
}

int sfl_reapply_q_init(void *ctx, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (!c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  if (c->cfg.shared_q) return fail(SFL_E_STATE, "shared-table mode keeps no per-environment tables%s");
  if (c->cfg.eval_q) return fail(SFL_E_STATE, "an evaluation context (eval_q) keeps no per-environment tables: put the optimistic rows into the evaluation table%s");
  DeviceGuard dg(c->device);
  ReinitArgs a;
  a.L = c->L; a.sw = c->m.sw; a.port = c->m.port; a.qinit = c->m.qinit; a.state = (char *)c->bufs.state;
  a.hp = (const sfl_hparams *)c->bufs.hparams; a.n_envs = c->cfg.n_envs; a.pad = 0;
#ifndef SFL_HOST_EMUL
  k_q_reinit<<<c->sm_count * 8, 256, 0, (cudaStream_t)stream>>>(a);
  CU(cudaGetLastError());
#else
  (void)stream;
  for (int e = 0; e < a.n_envs; e++) for (int i = 0; i < a.L.q_cap; i++) q_reinit_slot(a, e, i);
#endif
  return SFL_OK;
}

int sfl_enable_q_init(void *ctx, int on) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  c->q_init_on = on ? 1 : 0;
  return SFL_OK;
}

int sfl_run(void *ctx, int mode, int max_ticks, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c) return fail(SFL_E_ARG, "null ctx%s");
  if (!c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  if (mode < SFL_MODE_LEARN || mode > SFL_MODE_STEP || max_ticks < 0 || max_ticks > (1 << 25)) return fail(SFL_E_ARG, "bad mode / max_ticks (at most 2^25 ticks per launch)%s");
  if ((mode == SFL_MODE_REPLAY || mode == SFL_MODE_STEP) && (!c->bufs.replay_act || c->cfg.act_cap < 1))
    return fail(SFL_E_ARG, "replay / step mode needs replay_act (act_cap >= 1)%s");
  if (mode == SFL_MODE_STEP && !c->bufs.step_out) return fail(SFL_E_ARG, "step mode needs step_out%s");
  if (c->cfg.eval_q) {
    if (mode != SFL_MODE_GREEDY)
      return fail(SFL_E_ARG, "an evaluation context (eval_q) runs SFL_MODE_GREEDY only: learn, replay and step mode need per-environment tables%s");
    if (c->cfg.dec_cap > 0 || c->cfg.tick_cap > 0 || c->phase_clock)
      return fail(SFL_E_ARG, "an evaluation context (eval_q) has no traced or instrumented kernel (dec_cap, tick_cap, phase clock)%s");
  }
  DeviceGuard dg(c->device);
  KArgs K;
  memset(&K, 0, sizeof(K));
  K.m = c->m; K.L = c->L;
  RunArgs &ra = K.ra;
  ra.mode = mode; ra.max_ticks = max_ticks; ra.n_envs = c->cfg.n_envs; ra.trace_sem = c->cfg.trace_sem;
  ra.dec_cap = c->cfg.dec_cap; ra.tick_cap = c->cfg.tick_cap; ra.ep_cap = c->cfg.ep_cap; ra.act_cap = c->cfg.act_cap;
  ra.ev_cap = c->cfg.ev_cap; ra.max_steps = c->cfg.max_steps; ra.q_init_on = c->q_init_on;
  ra.hot_bytes = c->hot_bytes; ra.env_smem = c->env_smem; ra.tail_hot = c->tail_hot;
  ra.state = (char *)c->bufs.state; ra.hp = (const sfl_hparams *)c->bufs.hparams; ra.counters = (sfl_env_counters *)c->bufs.counters;
  ra.trace_dec = c->cfg.dec_cap > 0 ? (sfl_dec_rec *)c->bufs.trace_dec : nullptr;
  ra.trace_tick = c->cfg.tick_cap > 0 ? (sfl_tick_rec *)c->bufs.trace_tick : nullptr;
  ra.trace_sem_buf = (c->cfg.trace_sem && c->cfg.dec_cap > 0) ? (int4 *)c->bufs.trace_sem : nullptr;
  ra.ep_log = c->cfg.ep_cap > 0 ? (sfl_ep_rec *)c->bufs.ep_log : nullptr;
  ra.ep_delay = c->cfg.ep_cap > 0 ? (int *)c->bufs.ep_delay : nullptr;
  ra.replay_act = (const int8_t *)c->bufs.replay_act;
  ra.step_out = (sfl_step_rec *)c->bufs.step_out;
  if (c->cfg.shared_q) { ra.sq_q = (double *)c->bufs.shared_q; ra.sq_d = (long long *)c->bufs.shared_d; ra.sq_c = (int *)c->bufs.shared_c; }
  if (c->cfg.eval_q) ra.eval_q = (const double *)c->bufs.eval_q;
  // recorded malfunction events replace the Philox draws in replay mode, and in greedy / step mode when a schedule was bound (ev_cap > 0)
  // -- and in learn mode with the reference's stream or flatland's malfunction schedule, whose learn runs use the full kernel
  const int ref_learn = mode == SFL_MODE_LEARN && (c->cfg.rng == SFL_RNG_REFERENCE || c->cfg.malf_rng == SFL_MALF_REFERENCE);
  ra.replay_ev = ((mode != SFL_MODE_LEARN || ref_learn) && c->cfg.ev_cap > 0) ? (const int *)c->bufs.replay_ev : nullptr;
  // learn and greedy without traces run the two specialised kernels; replay, step, traced runs and learning on the
  // reference's streams the full one
  ra.phase_clock = c->phase_clock;
  const int trace = ra.trace_dec || ra.trace_tick || mode == SFL_MODE_STEP || mode == SFL_MODE_REPLAY || c->phase_clock || ref_learn;
  const int kind = trace ? K_FULL : (mode == SFL_MODE_GREEDY ? K_GREEDY : K_LEARN);
#ifndef SFL_HOST_EMUL
  LaunchPlan lp;
  if (plan_launch(c, kind, &lp)) return SFL_E_ARG;
  if (c->cfg.shared_q && trace) return fail(SFL_E_ARG, "shared-table mode has no trace / step variants%s");
  const int grid = lp.grid, threads = lp.threads;
  const size_t smem = lp.smem;
  run_kernel_t k = c->cfg.eval_q ? pick_eval(lp.G, lp.th, lp.one, lp.nw) : pick_kernel(lp.G, kind, lp.th, c->cfg.shared_q, lp.one, lp.roomy, lp.nw);
  CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, threads, smem, (cudaStream_t)stream>>>(K);
  CU(cudaGetLastError());
#else
  static thread_local char host_scratch[32 * SFL_MAX_T + 2 * SFL_MAX_T + 64];
  for (int i = 0; i < c->cfg.n_envs; i++) {
    if (c->cfg.eval_q) {
      if (c->L.T > 64) env_run<1, K_GREEDY, true, false, false, 2, true>(K, i, 0u, host_scratch);
      else env_run<1, K_GREEDY, true, false, false, 1, true>(K, i, 0u, host_scratch);
    } else if (c->cfg.shared_q) {
      if (trace) return fail(SFL_E_ARG, "shared-table mode has no trace / step variants%s");
      if (kind == K_GREEDY) env_run<1, K_GREEDY, true, true, false>(K, i, 0u, host_scratch); else env_run<1, K_LEARN, true, true, false>(K, i, 0u, host_scratch);
    } else if (c->L.T > 64) {
      if (kind == K_FULL) env_run<1, K_FULL, true, false, false, 2>(K, i, 0u, host_scratch);
      else if (kind == K_GREEDY) env_run<1, K_GREEDY, true, false, false, 2>(K, i, 0u, host_scratch);
      else env_run<1, K_LEARN, true, false, false, 2>(K, i, 0u, host_scratch);
    } else if (kind == K_FULL) env_run<1, K_FULL, true, false, false>(K, i, 0u, host_scratch);
    else if (kind == K_GREEDY) env_run<1, K_GREEDY, true, false, false>(K, i, 0u, host_scratch);
    else env_run<1, K_LEARN, true, false, false>(K, i, 0u, host_scratch);
  }
#endif
  return SFL_OK;
}

int sfl_malf_schedule(void *ctx, const uint64_t *hit_below, int32_t *max_events, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !hit_below || !max_events) return fail(SFL_E_ARG, "null argument%s");
  if (c->cfg.malf_rng != SFL_MALF_REFERENCE) return fail(SFL_E_STATE, "the context was not created with SFL_MALF_REFERENCE%s");
  if (!c->bound || !c->bufs.replay_ev) return fail(SFL_E_STATE, "sfl_bind first, with replay_ev%s");
  const int n = c->cfg.n_envs;
  for (int i = 0; i < n; i++) if (hit_below[i] > (1ull << 53)) return fail(SFL_E_ARG, "hit_below must be at most 2^53%s");
  DeviceGuard dg(c->device);
  MalfArgs a;
  a.hp = (const sfl_hparams *)c->bufs.hparams; a.hit_below = (const unsigned long long *)c->malf_buf; a.ev = (int *)c->bufs.replay_ev;
  a.result = (int *)((char *)c->malf_buf + (size_t)n * 8); a.n_envs = n; a.T = c->L.T; a.steps = c->m.max_episode_steps; a.ev_cap = c->cfg.ev_cap;
  int res[2] = {0, 0};
  CK(h2d(c->malf_buf, hit_below, (size_t)n * 8, stream));
#ifndef SFL_HOST_EMUL
  CK(dev_zero(a.result, 8, stream));
  k_malf_schedule<<<(n + SFL_MALF_WARPS - 1) / SFL_MALF_WARPS, 32 * SFL_MALF_WARPS, 0, (cudaStream_t)stream>>>(a);
  CU(cudaGetLastError());
  CK(d2h(res, a.result, 8, stream));
#else
  static thread_local unsigned mt[2 * SFL_MT_N];
  for (int i = 0; i < n; i++) malf_env(a, i, mt, Grp<1>(), res[0], res[1]);
#endif
  *max_events = res[0];
  if (res[1] & 1) return fail(SFL_E_ARG, "Seed must be between 0 and 2**32 - 1%s");
  if (res[1] & 2) return fail(SFL_E_ARG, "min_duration > max_duration: randint(min_duration, max_duration + 1) has low >= high%s");
  if (res[0] > c->cfg.ev_cap) {
    char detail[96];
    snprintf(detail, sizeof(detail), "%d events, ev_cap is %d", res[0], c->cfg.ev_cap);
    return fail(SFL_E_NOMEM, "the malfunction schedule does not fit replay_ev: %s", detail);
  }
  return SFL_OK;
}

static int shared_apply(Ctx *c, const double *src, double *dst, long long *d, int *cn, void *stream) {
  const size_t n = (size_t)c->m.NP * c->m.NT * 48u * (size_t)c->L.a_max;
#ifndef SFL_HOST_EMUL
  k_shared_apply<<<c->sm_count * 8, 256, 0, (cudaStream_t)stream>>>(src, dst, d, cn, n);
  CU(cudaGetLastError());
#else
  (void)stream;
  for (size_t i = 0; i < n; i++) {
    double v = src[i];
    if (cn[i]) { v += (double)d[i] / 16777216.0 / (double)cn[i]; d[i] = 0; cn[i] = 0; }
    dst[i] = v;
  }
#endif
  return SFL_OK;
}

int sfl_shared_q_apply(void *ctx, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  if (!c->cfg.shared_q) return fail(SFL_E_STATE, "context was not created in shared-table mode%s");
  return shared_apply(c, (const double *)c->bufs.shared_q, (double *)c->bufs.shared_q, (long long *)c->bufs.shared_d, (int *)c->bufs.shared_c, stream);
}

int sfl_shared_q_apply_to(void *ctx, const void *q_src, void *q_dst, void *d, void *cnt, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !q_src || !q_dst || !d || !cnt) return fail(SFL_E_ARG, "null argument%s");
  if (!c->cfg.shared_q) return fail(SFL_E_STATE, "context was not created in shared-table mode%s");
  DeviceGuard dg(c->device);
  return shared_apply(c, (const double *)q_src, (double *)q_dst, (long long *)d, (int *)cnt, stream);
}

int sfl_total_decisions(void *ctx, uint64_t *decisions, uint64_t *ticks, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  unsigned long long out[2] = {0, 0};
#ifndef SFL_HOST_EMUL
  CK(dev_zero(c->sum_buf, 16, stream));
  k_sum<<<c->sm_count, 256, 0, (cudaStream_t)stream>>>((const sfl_env_counters *)c->bufs.counters, c->cfg.n_envs, (unsigned long long *)c->sum_buf);
  CU(cudaGetLastError());
  CK(d2h(out, c->sum_buf, 16, stream));
#else
  const sfl_env_counters *cn = (const sfl_env_counters *)c->bufs.counters;
  for (int i = 0; i < c->cfg.n_envs; i++) { out[0] += cn[i].decisions; out[1] += cn[i].ticks; }
#endif
  if (decisions) *decisions = out[0];
  if (ticks) *ticks = out[1];
  return SFL_OK;
}

int sfl_export_q(void *ctx, int env, uint32_t *keys_host, double *vals_host, int cap_rows, int *n_rows, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  if (c->cfg.eval_q) return fail(SFL_E_STATE, "an evaluation context (eval_q) keeps no per-environment tables%s");
  if (env < 0 || env >= c->cfg.n_envs || !n_rows) return fail(SFL_E_ARG, "bad env / n_rows%s");
  const Layout &L = c->L;
  size_t n = (size_t)L.q_cap * L.q_stride;
  std::vector<double> img(n);
  CK(d2h(img.data(), (char *)c->bufs.state + (size_t)env * L.env_stride + L.off_q, n * 8, stream));
  int rows = 0;
  for (int i = 0; i < L.q_cap; i++) {
    unsigned long long k;
    memcpy(&k, &img[(size_t)i * L.q_stride], 8);
    if (!k) continue;
    if (rows < cap_rows && keys_host && vals_host) {
      keys_host[rows] = (uint32_t)(k - 1);
      for (int a = 0; a < L.a_max; a++) vals_host[(size_t)rows * L.a_max + a] = img[(size_t)i * L.q_stride + 1 + a];
    }
    rows++;
  }
  *n_rows = rows;
  return rows > cap_rows && keys_host ? fail(SFL_E_NOMEM, "export buffer too small%s") : SFL_OK;
}

int sfl_export_q_batch(void *ctx, int env_lo, int env_hi, const uint64_t *row_offsets, uint32_t *keys, double *vals, uint64_t cap_rows,
                       int32_t *rows_found, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  if (c->cfg.eval_q) return fail(SFL_E_STATE, "an evaluation context (eval_q) keeps no per-environment tables%s");
  if (env_lo < 0 || env_hi > c->cfg.n_envs || env_lo > env_hi) return fail(SFL_E_ARG, "bad environment range: need 0 <= env_lo <= env_hi <= n_envs%s");
  if (!row_offsets || !keys || !vals || !rows_found) return fail(SFL_E_ARG, "null argument%s");
  const int n = env_hi - env_lo;
  uint64_t last = 0;
  CK(d2h(&last, row_offsets + n, 8, stream));
  if (last > cap_rows) {
    char detail[96];
    snprintf(detail, sizeof(detail), "%llu rows, cap_rows is %llu", (unsigned long long)last, (unsigned long long)cap_rows);
    return fail(SFL_E_NOMEM, "the export buffers are smaller than the last row offset: %s", detail);
  }
  if (!n) return SFL_OK;
  CompactArgs a;
  a.L = c->L; a.state = (const char *)c->bufs.state; a.off = (const unsigned long long *)row_offsets; a.keys = keys; a.vals = vals;
  a.found = rows_found; a.cap_rows = cap_rows; a.env_lo = env_lo; a.n = n;
#ifndef SFL_HOST_EMUL
  k_q_compact<<<n, 32, 0, (cudaStream_t)stream>>>(a);
  CU(cudaGetLastError());
#else
  for (int j = 0; j < n; j++) q_compact_env(a, j, Grp<1>());
#endif
  return SFL_OK;
}

int sfl_import_q(void *ctx, int env, const uint32_t *keys_host, const double *vals_host, int n_rows, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  DeviceGuard dg(c->device);
  if (c->cfg.eval_q) return fail(SFL_E_STATE, "an evaluation context (eval_q) keeps no per-environment tables: use sfl_set_eval_table%s");
  if (env < 0 || env >= c->cfg.n_envs || n_rows < 0 || n_rows >= c->cfg.q_cap) return fail(SFL_E_ARG, "bad env / n_rows%s");
  const Layout &L = c->L;
  std::vector<double> img;
  int q_rows = q_image(L, keys_host, vals_host, n_rows, img);     // repeated keys overwrite their row
  char *base = (char *)c->bufs.state + (size_t)env * L.env_stride;
  CK(h2d(base + L.off_q, img.data(), img.size() * 8, stream));
  CK(h2d(base + offsetof(EnvHdr, q_rows), &q_rows, 4, stream));
#ifndef SFL_HOST_EMUL
  CU(cudaStreamSynchronize((cudaStream_t)stream));
#endif
  return SFL_OK;
}

int sfl_set_eval_table(void *ctx, const uint32_t *keys_host, const double *vals_host, int n_rows, void *stream) {
  Ctx *c = (Ctx *)ctx;
  if (!c || !c->bound) return fail(SFL_E_STATE, "sfl_bind first%s");
  if (!c->cfg.eval_q) return fail(SFL_E_STATE, "the context was not created as an evaluation context (eval_q)%s");
  if (n_rows < 0 || (n_rows && (!keys_host || !vals_host))) return fail(SFL_E_ARG, "bad keys / values / n_rows%s");
  if (n_rows >= c->cfg.q_cap) {
    char detail[96];
    snprintf(detail, sizeof(detail), "%d rows, q_cap is %d", n_rows, c->cfg.q_cap);
    return fail(SFL_E_NOMEM, "the evaluation table needs q_cap above its row count (a power of two; an empty slot ends every probe): %s", detail);
  }
  DeviceGuard dg(c->device);
  std::vector<double> img;
  q_image(c->L, keys_host, vals_host, n_rows, img);
  CK(h2d(c->bufs.eval_q, img.data(), img.size() * 8, stream));
#ifndef SFL_HOST_EMUL
  CU(cudaStreamSynchronize((cudaStream_t)stream));
#endif
  return SFL_OK;
}

}  // extern "C"
