// nbody_b200.cu — C-ABI implementation: parameter layouts, launch sequencing of the EGNO / SEGNO
// forward and backward, and the exported building blocks.  See include/nbody_b200.h.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "nb_common.cuh"
#include "nb_node.cuh"
#include "nb_spectral.cuh"
#include "nb_rollout.cuh"
#include "nb_sim.cuh"
#include "nb_edge.cuh"
#include "nb_tc.cuh"
#include "nb_edge_sel.cuh"
#include "nb_node_tc.cuh"
#include "nb_segno_fused.cuh"
#include "nb_merge.cuh"
#include "nb_egno_node.cuh"
#include <cstdlib>
#include <initializer_list>

// every kernel launch of this library is counted (bench.py reports it as gpu_launches)
#define NB_LAUNCH_COUNTED(...)                             \
  do {                                                     \
    __atomic_fetch_add(&g_launches, 1LL, __ATOMIC_RELAXED); \
    NB_LAUNCH(__VA_ARGS__);                                \
  } while (0)
static long long g_launches = 0;

// NVTX ranges around every compute entry point of the C ABI (header-only NVTX3: a no-op unless a profiler injects itself)
#ifndef NB_EMU
#include <nvtx3/nvToolsExt.h>
struct NbRange {
  explicit NbRange(const char* name) { nvtxRangePushA(name); }
  ~NbRange() { nvtxRangePop(); }
};
#define NB_RANGE(name) NbRange nb_range_guard_(name)
#else
#define NB_RANGE(name)
#endif

int nb_pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("NB_B200_PDL");   // opt-in: measured neutral in this form (see nb_common.cuh)
    on = (e && e[0] == '1') ? 1 : 0;
  }
  return on;
}

// ============================================================================= side stream
// Independent kernels of a call (EGNO: the 2-channel (x - mean, v) temporal convolution next to the 64-channel one) run on
// a library-owned second stream between a fork and a join event, so they overlap on the SMs instead of queueing behind
// each other.  The caller still sees ONE stream: everything forked is joined before the entry point returns, and under
// stream capture the side stream joins the caller's capture through the events (a fork / join pair in the graph).
// Created once per device at the first call (never while a capture is open: GraphedStep warms up eagerly first).
#ifndef NB_EMU
struct NbSide {
  cudaStream_t s;
  cudaEvent_t fork, join;
  cudaStream_t s2;               // deferred weight-gradient reductions of the EGNO backward (defer_flush)
  cudaEvent_t fork2, done2[2];
  bool ok;
};
static NbSide* side_get() {
  static NbSide tab[64];
  static bool tried[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  NbSide& x = tab[dev];
  if (!tried[dev]) {
    tried[dev] = true;
    x.ok = cudaStreamCreateWithFlags(&x.s, cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&x.fork, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&x.join, cudaEventDisableTiming) == cudaSuccess &&
           cudaStreamCreateWithFlags(&x.s2, cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&x.fork2, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&x.done2[0], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&x.done2[1], cudaEventDisableTiming) == cudaSuccess;
    if (!x.ok) cudaGetLastError();
  }
  return x.ok ? &x : nullptr;
}
// fork: returns the stream to launch the independent work on (the caller's own stream when there is no side stream)
static void* side_fork(void* main_st) {
  NbSide* x = side_get();
  if (!x) return main_st;
  cudaEventRecord(x->fork, (cudaStream_t)main_st);
  cudaStreamWaitEvent(x->s, x->fork, 0);
  return (void*)x->s;
}
static void side_join(void* side_st, void* main_st) {
  if (side_st == main_st) return;
  NbSide* x = side_get();
  cudaEventRecord(x->join, (cudaStream_t)side_st);
  cudaStreamWaitEvent((cudaStream_t)main_st, x->join, 0);
}
// the second side stream (deferred reductions, only with defer_available()): fork, completion slot i, wait for slot i
static void* side2_fork(void* main_st) {
  NbSide* x = side_get();
  cudaEventRecord(x->fork2, (cudaStream_t)main_st);
  cudaStreamWaitEvent(x->s2, x->fork2, 0);
  return (void*)x->s2;
}
static void side2_done(int i) { cudaEventRecord(side_get()->done2[i], side_get()->s2); }
static void side2_wait(void* main_st, int i) { cudaStreamWaitEvent((cudaStream_t)main_st, side_get()->done2[i], 0); }
#else
static void* side_fork(void* main_st) { return main_st; }
static void side_join(void*, void*) {}
static void* side2_fork(void* main_st) { return main_st; }
static void side2_done(int) {}
static void side2_wait(void*, int) {}
#endif

// ============================================================================= errors / device info
static thread_local char g_err[512] = "";

void nb_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int nb_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    nb_set_error("CUDA error reported after %s (it may stem from earlier asynchronous work on this device): %s", what,
                 cudaGetErrorString(e));
    return NB_ERR_CUDA;
  }
  return NB_OK;
}

int nb_num_sms() {
#ifdef NB_EMU
  return 3;
#else
  // cached per device ordinal: a thread may drive different GPUs over its lifetime
  static int cached[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  int n = cached[dev];
  if (!n) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    n = n > 0 ? n : 148;
    cached[dev] = n;   // benign race: every writer stores the same value
  }
  return n;
#endif
}

// ---- launch accounting and optional per-kernel CUDA-event timing (used by bench.py for the roofline)
#define NB_PROF_CATS 8  /* 0 edge_fwd, 1 edge_bwd, 2 node GEMMs / pair / SEGNO chain, 3 wgrad64, 4 temporal conv, 5 fused SEGNO forward,
                           6 k_egno_node_fwd, 7 k_egno_node_bwd */
#define NB_PROF_MAX 8192
#ifndef NB_EMU
static int g_prof_on = 0;
static cudaEvent_t g_prof_ev[NB_PROF_CATS][NB_PROF_MAX][2];
static int g_prof_made[NB_PROF_CATS] = {0};
static int g_prof_n[NB_PROF_CATS] = {0};
static int prof_begin(int cat, void* st) {
  if (!g_prof_on || g_prof_n[cat] >= NB_PROF_MAX) return -1;
  int i = g_prof_n[cat];
  if (i >= g_prof_made[cat]) {
    cudaEventCreate(&g_prof_ev[cat][i][0]);
    cudaEventCreate(&g_prof_ev[cat][i][1]);
    g_prof_made[cat] = i + 1;
  }
  cudaEventRecord(g_prof_ev[cat][i][0], (cudaStream_t)st);
  return i;
}
static void prof_end(int cat, int i, void* st) {
  if (i < 0) return;
  cudaEventRecord(g_prof_ev[cat][i][1], (cudaStream_t)st);
  g_prof_n[cat] = i + 1;
}
#else
static int prof_begin(int, void*) { return -1; }
static void prof_end(int, int, void*) {}
#endif

extern "C" long long nb_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

// enable != 0: start timing the dominant kernels with CUDA events on their launch stream (counters reset)
#ifdef NB_STAGE_CLOCKS
// profiling builds only (tools/stage_clocks.py): per-stage cycle totals of CTA 0 of k_edge_bwd_sel since the last reset
extern "C" int nb_debug_stage_clocks(long long* out, int reset) {
  cudaDeviceSynchronize();
  if (out) cudaMemcpyFromSymbol(out, nb_dbg_clk, sizeof(long long) * 32);
  if (reset) {
    long long z[32] = {0};
    cudaMemcpyToSymbol(nb_dbg_clk, z, sizeof(z));
  }
  return 0;
}
// the same for k_gemm64_tc (CTA (0, 0), thread 0): out[0] = launches, out[1..12] = cycles per stage (NB_GCLK)
extern "C" int nb_debug_gemm_clocks(long long* out, int reset) {
  cudaDeviceSynchronize();
  if (out) cudaMemcpyFromSymbol(out, nb_dbg_clk_gemm, sizeof(long long) * 16);
  if (reset) {
    long long z[16] = {0};
    cudaMemcpyToSymbol(nb_dbg_clk_gemm, z, sizeof(z));
  }
  return 0;
}
#endif

extern "C" int nb_profile_enable(int enable) {
#ifndef NB_EMU
  g_prof_on = enable;
  for (int c = 0; c < NB_PROF_CATS; ++c) g_prof_n[c] = 0;
#else
  (void)enable;
#endif
  return NB_OK;
}

// total milliseconds and launch counts per category since nb_profile_enable(1); synchronises the events
extern "C" int nb_profile_read(double* ms, long long* counts) {
  for (int c = 0; c < NB_PROF_CATS; ++c) { ms[c] = 0.0; counts[c] = 0; }
#ifndef NB_EMU
  for (int c = 0; c < NB_PROF_CATS; ++c) {
    for (int i = 0; i < g_prof_n[c]; ++i) {
      float t = 0.f;
      cudaEventSynchronize(g_prof_ev[c][i][1]);
      if (cudaEventElapsedTime(&t, g_prof_ev[c][i][0], g_prof_ev[c][i][1]) == cudaSuccess) ms[c] += t;
    }
    counts[c] = g_prof_n[c];
  }
#endif
  return nb_check_launch("nb_profile_read");
}

extern "C" int nb_version(void) { return 1; }
extern "C" const char* nb_last_error(void) { return g_err; }

#define NB_TRY(expr)          \
  do {                        \
    int _rc = (expr);         \
    if (_rc != NB_OK) return _rc; \
  } while (0)

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int imin(int64_t a, int64_t b) { return (int)(a < b ? a : b); }

// partial-sum scratch shared by all reducing kernels (floats)
#define NB_PARTIAL_FLOATS ((int64_t)8 * 1024 * 1024)
static inline int wgrad_grid_cap() { return imin(nb_num_sms(), 160); }
static inline int edge_bwd_grid_cap() { return imin(nb_num_sms(), 320); }

// node-level GEMMs / weight-gradient reductions: 1 = tcgen05 kernels (nb_node_tc.cuh, product path), 0 = fp32 SIMT
#ifdef NB_EMU
static int g_node_impl = 0;
#else
static int g_node_impl = 1;
#endif
extern "C" int nb_set_node_impl(int impl) {
#ifdef NB_EMU
  if (impl != 0) { nb_set_error("the host emulator only runs the SIMT node kernels"); return NB_ERR_INVALID; }
#endif
  if (impl != 0 && impl != 1) { nb_set_error("node impl must be 0 (SIMT) or 1 (tcgen05)"); return NB_ERR_INVALID; }
  g_node_impl = impl;
  return NB_OK;
}
extern "C" int nb_get_node_impl(void) { return g_node_impl; }
// EGNO: 1 = one node kernel per layer and direction (nb_egno_node.cuh; needs the tcgen05 node kernels), 0 = the generic
// GEMM launches + coordinate-update kernels they replaced (the cross-check)
static int g_node_fused = 1;
extern "C" int nb_set_node_fused(int on) { g_node_fused = on ? 1 : 0; return NB_OK; }
extern "C" int nb_get_node_fused(void) { return g_node_fused; }

// SEGNO: 1 = forward with all T sub-steps in one kernel, the node state resident in shared memory (nb_segno_fused.cuh;
// needs the tcgen05 variants and N <= 27), and backward with the node-level chain between two edge sweeps as one kernel
// (k_segno_node_bwd); 0 = one kernel sequence per sub-step in both directions (the cross-check)
#ifdef NB_EMU
static int g_segno_fused = 0;
#else
static int g_segno_fused = 1;
#endif
extern "C" int nb_set_segno_fused(int on) {
#ifdef NB_EMU
  if (on) { nb_set_error("the host emulator runs SEGNO one sub-step at a time"); return NB_ERR_INVALID; }
#endif
  g_segno_fused = on ? 1 : 0;
  return NB_OK;
}
extern "C" int nb_get_segno_fused(void) { return g_segno_fused; }

// ============================================================================= launch helpers
// exact_fp32: run the fp32 SIMT kernel even when the tcgen05 node kernels are selected.  Used for the spectral mode
// mixing, whose result feeds LeakyReLU: split-bf16 rounding (1e-5) would flip the kink for ~1e-5 of the elements and
// move the weight gradients by O(1/rows) per flip; fp32 keeps the forward mask and its backward recompute identical
// to the reference's.  These GEMMs have T times fewer rows than every other node GEMM.
#define EGNO_WIMG_PER_LAYER 6
// ---- weight images of the current forward / backward call (tcgen05 node GEMMs): registered once per call by
// wimg_prepare(), looked up by the weight block's address when a job is launched; a guard object clears the table when
// the call returns.  Sources whose weights are not registered (odd shapes, scaled operands) stage them element-wise.
#ifndef NB_EMU
struct WimgTable {
  const float* W[NB_MAX_WIMG];
  int ld[NB_MAX_WIMG];
  const unsigned char* img[NB_MAX_WIMG];
  int n;
};
static thread_local WimgTable g_wimg = {{nullptr}, {0}, {nullptr}, 0};
struct WimgGuard {
  ~WimgGuard() { g_wimg.n = 0; }
};
static inline int64_t wimg_floats(int nblocks) { return ((int64_t)nblocks * 2 * NB_TC_TILE_BYTES(64) / 4 + 63) / 64 * 64; }
// blocks: (address of element [0][0], leading dimension) of every 64 x 64 weight block the call's GEMMs multiply with
static int wimg_prepare(const float* const* W, const int* ld, int n, float* scratch, void* st) {
  g_wimg.n = 0;
  if (g_node_impl != 1 || n <= 0) return NB_OK;
  if (n > NB_MAX_WIMG) n = NB_MAX_WIMG;
  NbWimgBatch b;
  memset(&b, 0, sizeof(b));
  b.out = reinterpret_cast<unsigned char*>(scratch);
  for (int i = 0; i < n; ++i) {
    b.W[i] = W[i]; b.ld[i] = ld[i];
    g_wimg.W[i] = W[i]; g_wimg.ld[i] = ld[i]; g_wimg.img[i] = b.out + (size_t)i * 2 * NB_TC_TILE_BYTES(64);
  }
  g_wimg.n = n;
  NB_LAUNCH_COUNTED(k_weight_images, (unsigned)n, 256, 0, st, b);
  return nb_check_launch("k_weight_images");
}
static void wimg_attach(NbGemmArgs& a) {
  for (int s = 0; s < a.nsrc; ++s) {
    NbGemmSrc& src = a.src[s];
    src.img = nullptr; src.img_mn = 0;
    if (src.scale != 1.f || src.kmax != NB_H) continue;
    for (int i = 0; i < g_wimg.n; ++i) {
      if (g_wimg.W[i] != src.W) continue;
      if (src.sk == 1 && src.sn == g_wimg.ld[i]) { src.img = g_wimg.img[i]; src.img_mn = 0; }        // y = x W^T
      else if (src.sn == 1 && src.sk == g_wimg.ld[i]) { src.img = g_wimg.img[i]; src.img_mn = 1; }   // g = g' W
      break;
    }
  }
}
#else
struct WimgGuard {};
static inline int64_t wimg_floats(int) { return 0; }
static int wimg_prepare(const float* const*, const int*, int, float*, void*) { return NB_OK; }
#endif

static int launch_gemm_batch(const NbGemmArgs* jobs, int n, void* st, bool exact_fp32 = false) {
  int i = 0;
  while (i < n) {
    NbGemmBatch b;
    memset(&b, 0, sizeof(b));
    int maxrows = 0;
    while (i < n && b.njobs < NB_MAX_GEMM_JOBS) {
      if (jobs[i].rows > 0) {
        b.job[b.njobs++] = jobs[i];
        if (jobs[i].rows > maxrows) maxrows = jobs[i].rows;
      }
      ++i;
    }
    if (b.njobs == 0) continue;
#ifndef NB_EMU
    if (g_node_impl == 1 && !exact_fp32) {
      int nsrc_max = 1;
      for (int j = 0; j < b.njobs; ++j) {
        if (b.job[j].nsrc > nsrc_max) nsrc_max = b.job[j].nsrc;
        wimg_attach(b.job[j]);
      }
      const size_t smem_tc = NB_GEMM_TC_SMEM(nsrc_max);
      NB_SET_SMEM(k_gemm64_tc, NB_GEMM_TC_SMEM(2));
      // persistent CTAs: the two co-resident CTAs per SM (128 registers each) shared by the jobs of the batch, each
      // pipelined over its tiles (next tile's rows in flight under the current tile's MMAs and epilogue)
      int per_job = 2 * nb_num_sms() / b.njobs;
      if (per_job < 1) per_job = 1;
      const int gx = imin(cdiv(maxrows, NB_TILE), per_job);
      int pi_tc = prof_begin(2, st);
      NB_LAUNCH_COUNTED(k_gemm64_tc, dim3((unsigned)gx, (unsigned)b.njobs), NB_THREADS, smem_tc, st, b, nsrc_max);
      prof_end(2, pi_tc, st);
      NB_TRY(nb_check_launch("k_gemm64_tc"));
      continue;
    }
#endif
    const size_t smem = (NB_TILE * NB_LDA + NB_H * NB_H) * sizeof(float);
    NB_SET_SMEM(k_gemm64, smem);
    int pi = prof_begin(2, st);
    NB_LAUNCH_COUNTED(k_gemm64, dim3((unsigned)cdiv(maxrows, NB_TILE), (unsigned)b.njobs), NB_THREADS, smem, st, b);
    prof_end(2, pi, st);
    NB_TRY(nb_check_launch("k_gemm64"));
  }
  return NB_OK;
}
static int launch_gemm(const NbGemmArgs& a, void* st) { return launch_gemm_batch(&a, 1, st); }

static NbGemmSrc gsrc(const float* A, int lda, int a_silu, const float* W, int64_t sk, int64_t sn, float scale = 1.f) {
  NbGemmSrc s;
  s.A = A; s.lda = lda; s.a_silu = a_silu; s.W = W; s.sk = sk; s.sn = sn; s.scale = scale; s.kmax = NB_H;
  s.img = nullptr; s.img_mn = 0; s.seg_rows = 0; s.seg_a = 0;
  return s;
}

static NbGemmArgs gemm_args(int rows) {
  NbGemmArgs a;
  memset(&a, 0, sizeof(a));
  a.rows = rows;
  a.ldu = a.ldr = a.ldo = a.ldp = NB_H;
  return a;
}

static NbFinSeg fseg(int start, int count, int inner, int64_t dst_off, int64_t so, int64_t si) {
  NbFinSeg s;
  s.start = start; s.count = count; s.inner = inner; s.dst_off = dst_off; s.so = so; s.si = si; s.klimit = 0;
  return s;
}

// ---- deferred reductions: weight-gradient GEMMs and partial-sum finalisations are queued and launched in batches
// (one k_wgrad64 + one k_finalize launch per layer / iteration instead of one pair per parameter tensor).
// Jobs of one batch must target disjoint destination elements; q_flush() separates dependent batches.
struct WgradFin {
  int64_t w_off, so, si, b_off;
  float* dst;
  int accumulate;
  int klimit;
};
struct LaunchQueue {
  float* pbase;
  int64_t pcap, pused;
  NbWgradBatch wb;
  WgradFin wfin[NB_MAX_WGRAD_JOBS];
  NbFinBatch fb;
};
static thread_local LaunchQueue g_q;

static void q_begin(float* partial_base, int64_t cap) {
  g_q.pbase = partial_base;
  g_q.pcap = cap;
  g_q.pused = 0;
  g_q.wb.njobs = 0;
  g_q.fb.njobs = 0;
}
static int q_flush(void* st);
static int q_flush_fin(void* st, bool release_scratch = true) {
  if (g_q.fb.njobs == 0) {
    if (release_scratch) g_q.pused = 0;
    return NB_OK;
  }
  int maxtotal = 0;
  for (int j = 0; j < g_q.fb.njobs; ++j)
    if (g_q.fb.job[j].total > maxtotal) maxtotal = g_q.fb.job[j].total;
  NB_LAUNCH_COUNTED(k_finalize, dim3((unsigned)cdiv(maxtotal, 32), (unsigned)g_q.fb.njobs), 256, 0, st, g_q.fb);
  g_q.fb.njobs = 0;
  // stream order: the finalisation has consumed every partial slice whose reduction was queued; the caller keeps
  // the scratch when a slice has been handed out but its reduction is not queued yet
  if (release_scratch) g_q.pused = 0;
  return nb_check_launch("k_finalize");
}
// partial-sum scratch for a kernel launched now and finalised at the next flush
static float* q_alloc(int64_t nfloats, void* st) {
  nfloats = (nfloats + 63) / 64 * 64;
  if (g_q.pused + nfloats > g_q.pcap) {
    if (q_flush(st) != NB_OK || nfloats > g_q.pcap) return nullptr;
  }
  float* p = g_q.pbase + g_q.pused;
  g_q.pused += nfloats;
  return p;
}
static int q_partial(float** p, int64_t nfloats, void* st) {
  *p = q_alloc(nfloats, st);
  if (!*p) { nb_set_error("partial-sum workspace too small"); return NB_ERR_INVALID; }
  return NB_OK;
}
static int launch_finalize(NbFinArgs& f, void* st) {
  int total = 0;
  for (int s = 0; s < f.nseg; ++s) total += f.seg[s].count;
  f.total = total;
  if (g_q.fb.njobs == NB_MAX_FIN_JOBS) NB_TRY(q_flush_fin(st, false));
  g_q.fb.job[g_q.fb.njobs++] = f;
  return NB_OK;
}
// queues the reduction of `nparts` partial slices of `plen` floats into dst at the given segments
static int q_finalize(const float* partial, int nparts, int plen, float* dst, int accumulate,
                      std::initializer_list<NbFinSeg> segs, void* st) {
  NbFinArgs f;
  memset(&f, 0, sizeof(f));
  f.partial = partial; f.nparts = nparts; f.plen = plen; f.dst = dst; f.accumulate = accumulate;
  for (const NbFinSeg& s : segs) f.seg[f.nseg++] = s;
  return launch_finalize(f, st);
}
static int q_flush_wgrad(void* st) {
  NbWgradBatch& wb = g_q.wb;
  if (wb.njobs == 0) return NB_OK;
  int maxrows = 0;
  for (int j = 0; j < wb.njobs; ++j)
    if (wb.job[j].rows > maxrows) maxrows = wb.job[j].rows;
  int grid = imin(cdiv(maxrows, NB_TILE), wgrad_grid_cap());
#ifndef NB_EMU
  if (g_node_impl == 1) {
    // CTAs per SM over all jobs of the batch.  Three fit (and were the choice while the launch had the GPU to itself); on
    // the second stream, sharing the SMs with the next layer's kernels, two measured better (same box, alternating:
    // 3.241 / 3.241 ms per EGNO step with 3, 3.207 / 3.225 with 2, 3.277 with 1).
    const int ctas = 2;
    int per_job = ctas * nb_num_sms() / wb.njobs;
    if (per_job < 16) per_job = 16;
    if (per_job > nb_num_sms()) per_job = nb_num_sms();
    grid = imin(cdiv(maxrows, NB_TILE), per_job);
  }
#endif
  const int64_t need = (int64_t)wb.njobs * grid * NB_WGRAD_PLEN;
  if (g_q.pused + need > g_q.pcap) NB_TRY(q_flush_fin(st));
  if (need > g_q.pcap) { nb_set_error("partial-sum workspace too small"); return NB_ERR_INVALID; }
  for (int j = 0; j < wb.njobs; ++j) {
    wb.job[j].partial = g_q.pbase + g_q.pused;
    g_q.pused += (int64_t)grid * NB_WGRAD_PLEN;
  }
  bool wdone = false;
#ifndef NB_EMU
  if (g_node_impl == 1) {
    const size_t smem_tc = NB_WT_SMEM;
    NB_SET_SMEM(k_wgrad64_tc, smem_tc);
    int pi_tc = prof_begin(3, st);
    NB_LAUNCH_COUNTED(k_wgrad64_tc, dim3((unsigned)grid, (unsigned)wb.njobs), NB_THREADS, smem_tc, st, wb);
    prof_end(3, pi_tc, st);
    NB_TRY(nb_check_launch("k_wgrad64_tc"));
    wdone = true;
  }
#endif
  if (!wdone) {
    const size_t smem = 2 * NB_TILE * NB_LDA * sizeof(float);
    NB_SET_SMEM(k_wgrad64, smem);
    int pi = prof_begin(3, st);
    NB_LAUNCH_COUNTED(k_wgrad64, dim3((unsigned)grid, (unsigned)wb.njobs), NB_THREADS, smem, st, wb);
    prof_end(3, pi, st);
    NB_TRY(nb_check_launch("k_wgrad64"));
  }
  const int n = wb.njobs;
  wb.njobs = 0;
  for (int j = 0; j < n; ++j) {
    const WgradFin& wf = g_q.wfin[j];
    NbFinSeg w = fseg(0, NB_H * NB_H, NB_H, wf.w_off, wf.so, wf.si), b = fseg(NB_H * NB_H, NB_H, NB_H, wf.b_off, 0, 1);
    w.klimit = wf.klimit;
    if (wf.b_off >= 0) NB_TRY(q_finalize(wb.job[j].partial, grid, NB_WGRAD_PLEN, wf.dst, wf.accumulate, {w, b}, st));
    else NB_TRY(q_finalize(wb.job[j].partial, grid, NB_WGRAD_PLEN, wf.dst, wf.accumulate, {w}, st));
  }
  return NB_OK;
}
static int q_flush(void* st) {
  NB_TRY(q_flush_wgrad(st));
  return q_flush_fin(st);
}

// ---- deferred flush (EGNO backward).  The weight-gradient GEMMs and partial-sum finalisations of a layer feed nothing
// but the optimizer, yet launched on the caller's stream they sit between two layers of the dependent chain (one
// k_wgrad64_tc + one k_finalize per layer, ~50 us of a 3.3 ms step each).  Here a flush runs on a library-owned second
// stream (NbSide::s2), forked after the kernels that produced its operands, underneath the NEXT layer's backward.  What
// makes that legal: every buffer a queued job reads and a later layer rewrites exists twice (gh, GU5, GUV, gP, gQ, the
// spectral planes, the partial-sum arena), layer l uses set l & 1, and the caller's stream waits for flush k - 1 before
// it goes on past flush k — so a set is rewritten only after the flush that read it has completed.  The side stream is
// in order, the destinations are the same as before and every reduction keeps its fixed order: results are bitwise
// those of the synchronous flush.  Joined before the entry point returns; under stream capture fork / done events become
// graph edges.  NB_B200_WGRAD_DEFER=0 keeps the synchronous flush (A/B switch).
struct DeferState {
  bool on;
  int k;                     // flushes issued so far
  float* const* arena;       // the two partial-sum arenas, NB_PARTIAL_FLOATS each
};
static bool defer_available() {
#ifndef NB_EMU
  static int off = -1;
  if (off < 0) { const char* e = getenv("NB_B200_WGRAD_DEFER"); off = (e && e[0] == '0') ? 1 : 0; }
  return !off && side_get() != nullptr;
#else
  return false;
#endif
}
static int defer_flush(DeferState& D, void* main_st) {
  if (!D.on) return q_flush(main_st);
  NB_TRY(q_flush(side2_fork(main_st)));
  side2_done(D.k & 1);
  if (D.k > 0) side2_wait(main_st, (D.k - 1) & 1);   // set (k + 1) & 1 is free again
  ++D.k;
  g_q.pbase = D.arena[D.k & 1];
  g_q.pused = 0;
  return nb_check_launch("deferred flush");
}
static void defer_join(DeferState& D, void* main_st) {
  if (D.on && D.k > 0) side2_wait(main_st, (D.k - 1) & 1);
}

// dst[w_off + o*so + k*si] (+)= sum_rows sum_p scale_p G_p[r][o] A_p[r][k];  dst[b_off + o] (+)= colsum(G_0) if b_off >= 0
// (queued; executed at the next q_flush)
static int wgrad_to(int rows, int npair, NbWgradPair p0, NbWgradPair p1, float* dst, int64_t w_off, int64_t so,
                    int64_t si, int64_t b_off, int accumulate, void* st, int klimit = 0) {
  if (rows <= 0) return NB_OK;
  if (g_q.wb.njobs == NB_MAX_WGRAD_JOBS) NB_TRY(q_flush_wgrad(st));
  NbWgradArgs a;
  memset(&a, 0, sizeof(a));
  a.rows = rows; a.npair = npair; a.pair[0] = p0; a.pair[1] = p1; a.colsum = b_off >= 0;
  WgradFin wf;
  wf.w_off = w_off; wf.so = so; wf.si = si; wf.b_off = b_off; wf.dst = dst; wf.accumulate = accumulate; wf.klimit = klimit;
  g_q.wfin[g_q.wb.njobs] = wf;
  g_q.wb.job[g_q.wb.njobs++] = a;
  return NB_OK;
}

static NbWgradPair wpair(const float* G, const float* A, int a_silu = 0, float scale = 1.f) {
  NbWgradPair p;
  p.G = G; p.ldg = NB_H; p.A = A; p.lda = NB_H; p.a_silu = a_silu; p.scale = scale;
  p.seg_rows = 0; p.seg_g = p.seg_a = 0;
  return p;
}
// the same tensors of `nseg` consecutive blocks (seg_rows rows each, seg_g / seg_a floats apart): rows = nseg * seg_rows
static NbWgradPair wpair_seg(const float* G, const float* A, int a_silu, int seg_rows, int64_t seg_g, int64_t seg_a) {
  NbWgradPair p = wpair(G, A, a_silu);
  p.seg_rows = seg_rows; p.seg_g = seg_g; p.seg_a = seg_a;
  return p;
}
static int wgrad_to(int rows, NbWgradPair p, float* dst, int64_t w_off, int64_t so, int64_t si, int64_t b_off,
                    int accumulate, void* st, int klimit = 0) {
  return wgrad_to(rows, 1, p, wpair(nullptr, nullptr), dst, w_off, so, si, b_off, accumulate, st, klimit);
}

static int ew_grid(int64_t n) { return imin(cdiv(n, 256), 8 * nb_num_sms()); }

// ============================================================================= edge tile launches
static NbEdgeGeom edge_geom(int n_gt, int B, int N, int nef, int clamp_edge) {
  NbEdgeGeom g;
  memset(&g, 0, sizeof(g));
  g.N = N; g.EPG = N * (N - 1); g.NGT = n_gt; g.B = B; g.nef = nef; g.clamp_edge = clamp_edge;
  int G = NB_TILE / g.EPG;            // pack small graphs so a tile is (nearly) full
  if (G < 1) G = 1;
  if (G * N > 128) G = 128 / N;
  if (G < 1) G = 1;
  g.G = G;
  g.n_units = (int)cdiv(n_gt, G);
  return g;
}

// 2 = tcgen05 edge tiles with tensor-core gathers / scatters (nb_edge_sel.cuh; product path on sm_100a, whole-graph
//     units for N <= 27 and the blocked walk up to N = 255), 0 = fp32 SIMT tiles (cross-check; the only variant the
//     host emulator can run)
#ifdef NB_EMU
static int g_edge_impl = 0;
#else
static int g_edge_impl = 2;
#endif
extern "C" int nb_set_edge_impl(int impl) {
#ifdef NB_EMU
  if (impl != 0) { nb_set_error("the host emulator only runs the SIMT edge tiles"); return NB_ERR_INVALID; }
#endif
  if (impl != 0 && impl != 2) { nb_set_error("edge impl must be 0 (SIMT) or 2 (tcgen05 + selector MMAs)"); return NB_ERR_INVALID; }
  g_edge_impl = impl;
  return NB_OK;
}
extern "C" int nb_get_edge_impl(void) { return g_edge_impl; }
// edge impl 2, forward: 1 = whole-graph units of three or more tiles run k_edge_fwd_sel3 (three tiles in flight per SM),
// 0 = every shape runs k_edge_fwd_sel (the cross-check; both give bitwise equal results)
static int g_edge_fwd3 = 1;
extern "C" int nb_set_edge_fwd3(int on) { g_edge_fwd3 = on ? 1 : 0; return NB_OK; }
extern "C" int nb_get_edge_fwd3(void) { return g_edge_fwd3; }

#ifndef NB_EMU
// unit geometry of the selector kernels: G graph-instances with G*N <= 27 nodes and (for G > 1) at most 128 rows
static bool sel_geom(NbEdgeGeom& g) {
  if (g.N > NB_SEL_MAX_GN) {  // blocked walk: (8 receivers) x (16 senders) per tile, one CTA per graph-instance
    if (g.N > 255) return false;
    g.blk = 1;
    // receivers x senders per tile: IB * JB <= 128 rows, IB + JB <= 54 selector columns, IB <= 32 (position slots);
    // fewest tiles per graph wins
    int best = 1 << 30;
    for (int ib = 1; ib <= 32; ++ib) {
      int jb = NB_TILE / ib;
      if (jb > 32) jb = 32;
      if (jb > g.N) jb = g.N;
      if (ib + jb > NB_SEL_XC0 || jb < 1) continue;
      const int tiles = (int)(cdiv(g.N, ib) * cdiv(g.N, jb));
      if (tiles < best) { best = tiles; g.IB = ib; g.JB = jb; }
    }
    g.nI = (int)cdiv(g.N, g.IB);
    g.nJ = (int)cdiv(g.N, g.JB);
    g.G = 1;
    g.n_units = g.NGT;
    return true;
  }
  g.blk = 0; g.nI = g.nJ = g.IB = g.JB = 0;
  int G = NB_TILE / g.EPG;
  if (G > NB_SEL_MAX_GN / g.N) G = NB_SEL_MAX_GN / g.N;
  if (G < 1) G = 1;
  g.G = G;
  g.n_units = (int)cdiv(g.NGT, G);
  return true;
}
#endif

static int launch_edge_fwd(NbEdgeFwdArgs& a, void* st) {
#ifndef NB_EMU
  if (g_edge_impl == 2) {
    // no silent switch to another variant: a shape the selector kernels cannot walk is an error
    if (!sel_geom(a.g)) { nb_set_error("selector edge kernels support at most 255 nodes per graph (N=%d)", a.g.N); return NB_ERR_INVALID; }
    // one graph-instance of at least three tiles per unit (N = 17 .. 27): every warp group of k_edge_fwd_sel3 has a tile
    // in every unit.  Smaller units (two tiles at N = 12 .. 16, packed graphs below) and the blocked walk keep the
    // two-CTA kernel.
    if (g_edge_fwd3 && !a.g.blk && a.g.G == 1 && a.g.EPG > 2 * NB_TILE) {
      const size_t smem3 = NB_EDGE_FWD_SEL3_SMEM(a.g.EPG);
      const int grid3 = imin(a.g.n_units, nb_num_sms());
      int pi3 = prof_begin(0, st);
      NB_SET_SMEM(k_edge_fwd_sel3, smem3);
      NB_LAUNCH_COUNTED(k_edge_fwd_sel3, (unsigned)grid3, NB_F3_THREADS, smem3, st, a);
      prof_end(0, pi3, st);
      return nb_check_launch("k_edge_fwd_sel3");
    }
    const size_t smem_sel = NB_EDGE_FWD_SEL_SMEM(a.g.blk ? 0 : a.g.G * a.g.EPG);
    int grid_sel = imin(a.g.n_units, 2 * nb_num_sms());
    int pi_sel = prof_begin(0, st);
    if (a.g.blk) {
      NB_SET_SMEM(k_edge_fwd_sel<true>, smem_sel);
      NB_LAUNCH_COUNTED(k_edge_fwd_sel<true>, (unsigned)grid_sel, NB_THREADS, smem_sel, st, a);
    } else {
      NB_SET_SMEM(k_edge_fwd_sel<false>, smem_sel);
      NB_LAUNCH_COUNTED(k_edge_fwd_sel<false>, (unsigned)grid_sel, NB_THREADS, smem_sel, st, a);
    }
    prof_end(0, pi_sel, st);
    return nb_check_launch("k_edge_fwd_sel");
  }
#endif
  const size_t smem = NB_EDGE_FWD_SMEM_FLOATS * sizeof(float);
  NB_SET_SMEM(k_edge_fwd, smem);
  int grid = imin(a.g.n_units, 3 * nb_num_sms());
  int pi = prof_begin(0, st);
  NB_LAUNCH_COUNTED(k_edge_fwd, (unsigned)grid, NB_THREADS, smem, st, a);
  prof_end(0, pi, st);
  return nb_check_launch("k_edge_fwd");
}

// grads of the edge-tile weights go to `dst` (parameter-gradient buffer) at the given offsets
struct EdgeGradDst {
  int64_t w1, b_unused, W2, b2, W3, b3, w4, b4;
  int ldw1, col_rad, col_ef;
};

// reduction of `nparts` per-CTA partial slices of the edge backward kernel(s) into the parameter gradients
static int edge_bwd_finalize(float* partial, int nparts, int nef, float* dst, const EdgeGradDst& d, int accumulate, void* st) {
  return q_finalize(partial, nparts, NB_EB_PLEN, dst, accumulate,
                    {fseg(NB_EB_GW2, NB_H * NB_H, NB_H, d.W2, NB_H, 1), fseg(NB_EB_GW3, NB_H * NB_H, NB_H, d.W3, NB_H, 1),
                     fseg(NB_EB_GB2, NB_H, NB_H, d.b2, 0, 1), fseg(NB_EB_GB3, NB_H, NB_H, d.b3, 0, 1),
                     fseg(NB_EB_GW4, NB_H, NB_H, d.w4, 0, 1),
                     fseg(NB_EB_GWR, NB_H, 1, d.w1 + d.col_rad, d.ldw1, 0),           // column col_rad of W1
                     fseg(NB_EB_GWE, nef * NB_H, NB_H, d.w1 + d.col_ef, 1, d.ldw1),   // (f, c) -> W1[c][col_ef + f]
                     fseg(NB_EB_GB4, 1, 1, d.b4, 0, 0)},
                    st);
}

// run: when given, the finalisation is NOT queued here; the partial slices of consecutive launches are contiguous (the
// caller queues one reduction over all of them, edge_bwd_finalize): *run_base = first slice, *run_parts += this grid
static int launch_edge_bwd(NbEdgeBwdArgs& a, float* dst, const EdgeGradDst& d, int accumulate, void* st,
                           float** run_base = nullptr, int* run_parts = nullptr) {
  bool use_sel = false;
#ifndef NB_EMU
  if (g_edge_impl == 2) {
    if (!sel_geom(a.g)) { nb_set_error("selector edge kernels support at most 255 nodes per graph (N=%d)", a.g.N); return NB_ERR_INVALID; }
    use_sel = true;
  }
#endif
  int grid = imin(a.g.n_units, use_sel ? nb_num_sms() : edge_bwd_grid_cap());
  if (run_base && *run_parts > 0 && g_q.pused + ((int64_t)grid * NB_EB_PLEN + 63) / 64 * 64 > g_q.pcap) {
    // the scratch is full: reduce the run collected so far before q_alloc recycles it
    NB_TRY(edge_bwd_finalize(*run_base, *run_parts, a.g.nef, dst, d, accumulate, st));
    NB_TRY(q_flush(st));
    *run_parts = 0;
  }
  float* partial;
  NB_TRY(q_partial(&partial, (int64_t)grid * NB_EB_PLEN, st));
  a.partial = partial;
  if (run_base) {
    if (*run_parts == 0) *run_base = partial;
    else if (partial != *run_base + (int64_t)*run_parts * NB_EB_PLEN) { nb_set_error("edge backward partial slices are not contiguous"); return NB_ERR_INVALID; }
  }
  bool done = false;
#ifndef NB_EMU
  if (use_sel) {
    const size_t smem_sel = NB_EDGE_BWD_SEL_SMEM(a.g.blk ? 0 : a.g.G * a.g.EPG) +
                            (a.g.blk ? NB_EDGE_BWD_SEL_BLK_EXTRA(a.g.N) : NB_SB_ONES64_BYTES);
    int pi_sel = prof_begin(1, st);
    if (a.gef) {
      if (a.g.blk) {
        NB_SET_SMEM((k_edge_bwd_sel<true, true>), smem_sel);
        NB_LAUNCH_COUNTED((k_edge_bwd_sel<true, true>), (unsigned)grid, NB_SB_THREADS, smem_sel, st, a);
      } else {
        NB_SET_SMEM((k_edge_bwd_sel<false, true>), smem_sel);
        NB_LAUNCH_COUNTED((k_edge_bwd_sel<false, true>), (unsigned)grid, NB_SB_THREADS, smem_sel, st, a);
      }
    } else if (a.g.blk) {
      NB_SET_SMEM((k_edge_bwd_sel<true, false>), smem_sel);
      NB_LAUNCH_COUNTED((k_edge_bwd_sel<true, false>), (unsigned)grid, NB_SB_THREADS, smem_sel, st, a);
    } else {
      NB_SET_SMEM((k_edge_bwd_sel<false, false>), smem_sel);
      NB_LAUNCH_COUNTED((k_edge_bwd_sel<false, false>), (unsigned)grid, NB_SB_THREADS, smem_sel, st, a);
    }
    prof_end(1, pi_sel, st);
    NB_TRY(nb_check_launch("k_edge_bwd_sel"));
    done = true;
  }
#endif
  if (!done) {
    const size_t smem = NB_EDGE_BWD_SMEM_FLOATS(a.g.G * a.g.N) * sizeof(float);
    int pi = prof_begin(1, st);
    if (a.gef) {
      NB_SET_SMEM(k_edge_bwd<true>, smem);
      NB_LAUNCH_COUNTED(k_edge_bwd<true>, (unsigned)grid, NB_THREADS, smem, st, a);
    } else {
      NB_SET_SMEM(k_edge_bwd<false>, smem);
      NB_LAUNCH_COUNTED(k_edge_bwd<false>, (unsigned)grid, NB_THREADS, smem, st, a);
    }
    prof_end(1, pi, st);
    NB_TRY(nb_check_launch("k_edge_bwd"));
  }
  if (run_base) {
    *run_parts += grid;
    return NB_OK;
  }
  return edge_bwd_finalize(partial, grid, a.g.nef, dst, d, accumulate, st);
}

// ============================================================================= twiddles
static int make_twiddle(int T, int modes, NbTwiddle* tw) {
  if (T < 1 || T > NB_MAX_T || modes < 1 || modes > T / 2 + 1) {
    nb_set_error("unsupported temporal conv: T=%d (<= %d), modes=%d (<= T/2+1)", T, NB_MAX_T, modes);
    return NB_ERR_INVALID;
  }
  memset(tw, 0, sizeof(*tw));
  tw->T = T;
  tw->modes = modes;
  tw->nyq = (T % 2 == 0 && modes - 1 >= T / 2) ? T / 2 : -1;
  if (T == 1) tw->nyq = -1;
  tw->ncoef = 1 + 2 * (modes - 1);
  for (int m = 0; m < modes; ++m)
    for (int t = 0; t < T; ++t) {
      double th = 2.0 * M_PI * (double)((m * t) % T) / (double)T;
      tw->c[m][t] = (float)cos(th);
      tw->s[m][t] = (m == 0 || m == tw->nyq) ? 0.f : (float)sin(th);
    }
  return NB_OK;
}

// ============================================================================= EGNO
#define NB_MAX_LAYERS 32
struct EgnoLayerOff {
  int64_t e_w1, e_b1, e_w2, e_b2, c_w1, c_b1, c_w2, c_b2, v_w1, v_b1, v_w2, v_b2, n_w1, n_b1, n_w2, n_b2, tc, tcx;
};
struct EgnoLayout {
  int F, E;  // embedding inputs, first edge layer inputs
  int64_t emb_w, emb_b, total;
  EgnoLayerOff L[NB_MAX_LAYERS];
};

static int egno_validate(const NbEgnoConfig* c) {
  if (!c) { nb_set_error("null config"); return NB_ERR_INVALID; }
  if (c->B < 1 || c->N < 2 || c->N > NB_MAX_NODES) { nb_set_error("unsupported B=%d N=%d (2 <= N <= %d)", c->B, c->N, NB_MAX_NODES); return NB_ERR_INVALID; }
  if (c->n_layers < 1 || c->n_layers > NB_MAX_LAYERS) { nb_set_error("unsupported n_layers=%d", c->n_layers); return NB_ERR_INVALID; }
  if (c->T < 1 || c->T > NB_MAX_T) { nb_set_error("unsupported num_timesteps=%d (<= %d)", c->T, NB_MAX_T); return NB_ERR_INVALID; }
  if (c->use_time_conv && (c->num_modes < 1 || c->num_modes > c->T / 2 + 1)) { nb_set_error("num_modes=%d must be in [1, T/2+1] for T=%d", c->num_modes, c->T); return NB_ERR_INVALID; }
  if (c->in_edge_nf < 0 || c->in_edge_nf > NB_MAX_EDGE_FEA) { nb_set_error("unsupported in_edge_nf=%d", c->in_edge_nf); return NB_ERR_INVALID; }
  if (c->num_inputs < 0 || c->num_inputs > c->T) { nb_set_error("num_inputs=%d must be in [1, num_timesteps=%d]", c->num_inputs, c->T); return NB_ERR_INVALID; }
  if (c->in_node_nf < 1 || c->time_emb_dim < 0 || c->time_emb_dim > 64 || (c->time_emb_dim & 1) ||
      c->in_node_nf + c->time_emb_dim * (c->num_inputs > 1 ? 2 : 1) > 128 || (c->num_inputs > 1 && c->time_emb_dim == 0)) {
    nb_set_error("unsupported in_node_nf=%d time_emb_dim=%d num_inputs=%d", c->in_node_nf, c->time_emb_dim, c->num_inputs);
    return NB_ERR_INVALID;
  }
  if ((int64_t)c->T * c->B * c->N * (c->N - 1) > 2000000000LL) { nb_set_error("too many edges for 32-bit indexing"); return NB_ERR_INVALID; }
  return NB_OK;
}

static void egno_layout(const NbEgnoConfig* c, EgnoLayout* lo) {
  const int H = NB_H;
  lo->F = c->in_node_nf + c->time_emb_dim * (c->num_inputs > 1 ? 2 : 1);   // egno.py:13-16
  lo->E = 1 + 2 * H + c->in_edge_nf;
  int64_t o = 0;
  // named_parameters() order of the reference: `layers` is registered before `embedding` (basic.py:193-197)
  for (int l = 0; l < c->n_layers; ++l) {
    EgnoLayerOff& L = lo->L[l];
    L.e_w1 = o; o += (int64_t)H * lo->E;
    L.e_b1 = o; o += H;
    L.e_w2 = o; o += H * H;
    L.e_b2 = o; o += H;
    L.c_w1 = o; o += H * H;
    L.c_b1 = o; o += H;
    L.c_w2 = o; o += H;
    L.c_b2 = o; o += 1;
    L.v_w1 = o; o += H * H;
    L.v_b1 = o; o += H;
    L.v_w2 = o; o += H;
    L.v_b2 = o; o += 1;
    L.n_w1 = o; o += H * 2 * H;
    L.n_b1 = o; o += H;
    L.n_w2 = o; o += H * H;
    L.n_b2 = o; o += H;
  }
  lo->emb_w = o; o += (int64_t)H * lo->F;
  lo->emb_b = o; o += H;
  if (c->use_time_conv) {
    for (int l = 0; l < c->n_layers; ++l) { lo->L[l].tc = o; o += (int64_t)H * H * c->num_modes * 2; }
    for (int l = 0; l < c->n_layers; ++l) { lo->L[l].tcx = o; o += (int64_t)2 * 2 * c->num_modes * 2; }
  }
  lo->total = o;
}

struct EgnoLayerBufs {
  float *h0, *h1, *M, *U5, *UV, *P, *Q, *x0, *v0, *x1, *v1, *Fsum;
  uint32_t* tmask;   // [Nn0][16][2]: sign bits of the temporal convolution's pre-activation (bit 4 t + channel), see k_tconv_fwd
};
// P, Q (the per-node halves of the first edge layer) are kept for the backward edge tile: 26 MB per layer at B = 256
// instead of one more two-job GEMM launch per layer in the backward pass
static inline int64_t egno_layer_floats(int64_t Nn, int64_t Nn0) { return Nn * (7 * NB_H + 5 * 3) + Nn0 * 32; }
static EgnoLayerBufs egno_layer_bufs(float* base, int64_t Nn) {
  EgnoLayerBufs b;
  b.h0 = base; b.h1 = b.h0 + Nn * NB_H; b.M = b.h1 + Nn * NB_H; b.U5 = b.M + Nn * NB_H; b.UV = b.U5 + Nn * NB_H;
  b.P = b.UV + Nn * NB_H; b.Q = b.P + Nn * NB_H;
  b.x0 = b.Q + Nn * NB_H; b.v0 = b.x0 + Nn * 3; b.x1 = b.v0 + Nn * 3; b.v1 = b.x1 + Nn * 3; b.Fsum = b.v1 + Nn * 3;
  b.tmask = reinterpret_cast<uint32_t*>(b.Fsum + Nn * 3);
  return b;
}
static inline int64_t align64(int64_t v) { return (v + 63) / 64 * 64; }

extern "C" int64_t nb_egno_param_count(const NbEgnoConfig* cfg) {
  if (egno_validate(cfg) != NB_OK) return -1;
  EgnoLayout lo;
  egno_layout(cfg, &lo);
  return lo.total;
}

extern "C" int64_t nb_egno_saved_floats(const NbEgnoConfig* cfg) {
  if (egno_validate(cfg) != NB_OK) return -1;
  int64_t Nn = (int64_t)cfg->T * cfg->B * cfg->N;
  return align64(egno_layer_floats(Nn, (int64_t)cfg->B * cfg->N)) * cfg->n_layers;
}

// two tables (output times, input times) of T*B*D floats each: first region of the workspace
static inline int64_t egno_table_floats(const NbEgnoConfig* c) { return 2 * align64((int64_t)c->T * c->B * (c->time_emb_dim > 0 ? c->time_emb_dim : 1)); }
// frame -> input map of repeat_elements_to_exact_shape (EGNO/utils.py:115-131)
static NbFrameMap egno_frame_map(const NbEgnoConfig* c) {
  NbFrameMap fm;
  memset(&fm, 0, sizeof(fm));
  fm.L = c->num_inputs > 1 ? c->num_inputs : 1;
  const int reps = c->T / fm.L;
  for (int t = 0; t < c->T && t < NB_MAX_T; ++t) fm.m[t] = fm.L > 1 ? (t / reps < fm.L - 1 ? t / reps : fm.L - 1) : 0;
  return fm;
}
struct EgnoCtx {
  const NbEgnoConfig* c;
  EgnoLayout lo;
  NbTwiddle tw;
  NbFrameMap fm;
  int64_t Nn0, Nn;
  const float* params;
  void* st;
};

static int egno_ctx_init(EgnoCtx* X, const NbEgnoConfig* cfg, const float* params, void* st) {
  NB_TRY(egno_validate(cfg));
  X->c = cfg;
  egno_layout(cfg, &X->lo);
  if (cfg->use_time_conv) NB_TRY(make_twiddle(cfg->T, cfg->num_modes, &X->tw));
  X->fm = egno_frame_map(cfg);
  X->Nn0 = (int64_t)cfg->B * cfg->N;
  X->Nn = X->Nn0 * cfg->T;
  X->params = params;
  X->st = st;
  return NB_OK;
}

static NbEdgeGeom egno_edge_geom(const EgnoCtx& X) {
  NbEdgeGeom g = edge_geom(X.c->T * X.c->B, X.c->B, X.c->N, X.c->in_edge_nf, 0);
  g.multi = X.fm.L > 1;
  for (int t = 0; t < NB_MAX_T; ++t) g.tmap[t] = X.fm.m[t];
  return g;
}
// the time inputs of an EGNO call: int64 frame indices (nb_egno_forward, nb_egno_backward[_ex]) or fp32 times
// (nb_egno_forward_ft, nb_egno_backward_ft); exactly one of the two pairs is set
struct EgnoTimes {
  const int64_t *out, *in;
  const float *fout, *fin;
};
// embedding inputs (egno.py:50,59-76): fills the kernel arguments, builds the time table(s), materialises the input
// rows 64 wide into ein0 (features 0..63) and ein1 (features 64.., only when F > 64)
static int egno_embed_inputs(const EgnoCtx& X, NbEmbedArgs& e, const float* nodes, const EgnoTimes& ts, float* table,
                             float* ein0, float* ein1, void* stream) {
  const NbEgnoConfig* cfg = X.c;
  memset(&e, 0, sizeof(e));
  e.T = cfg->T; e.Nn0 = cfg->B * cfg->N; e.B = cfg->B; e.F0 = cfg->in_node_nf; e.D = cfg->time_emb_dim;
  e.nodes = nodes; e.tsteps = ts.out; e.tsteps_in = ts.in;
  e.L = X.fm.L;
  for (int t = 0; t < NB_MAX_T; ++t) e.tmap[t] = X.fm.m[t];
  if (X.fm.L > 1 && (ts.fout ? !ts.fin : !ts.in)) { nb_set_error("num_inputs > 1 needs timesteps_in"); return NB_ERR_INVALID; }
  const int half = e.D / 2;
  for (int k = 0; k < half; ++k) {
    float sc = (float)(log(10000.0) / (double)(half - 1));  // layer_no.py:10-11 (fp32 arange * python scalar)
    e.freq[k] = expf((float)k * -sc);
  }
  e.table = table;
  e.table_in = table + egno_table_floats(cfg) / 2;
  const int64_t Nn = (int64_t)e.T * e.Nn0;
  if (e.D > 0) {
    const unsigned tg = (unsigned)imin(cdiv((int64_t)e.T * e.B * e.D, 256), 4 * nb_num_sms());
    if (ts.fout) {
      NB_LAUNCH_COUNTED(k_time_table_f, tg, 256, 0, stream, e, ts.fout, ts.fin, 0);
      if (X.fm.L > 1) NB_LAUNCH_COUNTED(k_time_table_f, tg, 256, 0, stream, e, ts.fout, ts.fin, 1);
    } else {
      NB_LAUNCH_COUNTED(k_time_table, tg, 256, 0, stream, e, 0);
      if (X.fm.L > 1) NB_LAUNCH_COUNTED(k_time_table, tg, 256, 0, stream, e, 1);
    }
    NB_TRY(nb_check_launch("k_time_table"));
  }
  NB_LAUNCH_COUNTED(k_embed_inputs, (unsigned)ew_grid(Nn * 16), 256, 0, stream, e, ein0, 0);
  if (X.lo.F > NB_H) NB_LAUNCH_COUNTED(k_embed_inputs, (unsigned)ew_grid(Nn * 16), 256, 0, stream, e, ein1, NB_H);
  return nb_check_launch("k_embed_inputs");
}

static int64_t egno_coef_floats(const NbEgnoConfig* c) {
  int ncoef = c->use_time_conv ? 1 + 2 * (c->num_modes - 1) : 0;
  return align64((int64_t)ncoef * c->B * c->N * NB_H);
}

// ---- workspace layouts: each function carves the regions of one workspace, in order, from `base`.  With base ==
// nullptr it only counts: the nb_*_workspace_floats queries return its `total`, so sizes and offsets have one source.
struct Carve {
  float* base;
  int64_t used;
  float* take(int64_t n) { float* p = base ? base + used : nullptr; used += n; return p; }
};

// EGNO forward; inference (nothing saved) adds two ping-pong layer sets
struct EgnoFwdWs {
  float *wimg, *ttab, *P, *Q, *coef, *ycoef, *infer;
  int64_t total;
};
static EgnoFwdWs egno_fwd_ws(const NbEgnoConfig* c, bool infer, float* base) {
  const int64_t Nn = (int64_t)c->T * c->B * c->N, nh = align64(Nn * NB_H), cf = egno_coef_floats(c);
  Carve w = {base, 0};
  EgnoFwdWs s;
  s.wimg = w.take(wimg_floats(EGNO_WIMG_PER_LAYER * c->n_layers)); s.ttab = w.take(egno_table_floats(c));
  s.P = w.take(nh); s.Q = w.take(nh); s.coef = w.take(cf); s.ycoef = w.take(cf);
  s.infer = infer ? w.take(2 * align64(egno_layer_floats(Nn, (int64_t)c->B * c->N))) : nullptr;
  s.total = w.used;
  return s;
}

// EGNO backward.  A buffer set holds everything a queued weight-gradient job reads and the next layer rewrites; with
// deferred flushes layer l uses set l & 1 and partial-sum arena l & 1 (see defer_flush), otherwise set 0 and arena 0.
struct EgnoBwdSet {
  float *gh, *GU5, *GUV, *gP, *gQ, *coef, *gycoef;
};
struct EgnoBwdWs {
  float *wimg, *ttab, *P, *Q, *ycoef, *gcoef, *ghA, *gM, *gx[2], *gvA, *gvB, *gFsum, *arena[2];
  EgnoBwdSet set[2];
  int64_t total;
};
static EgnoBwdWs egno_bwd_ws(const NbEgnoConfig* c, float* base) {
  const int64_t Nn = (int64_t)c->T * c->B * c->N, nh = align64(Nn * NB_H), n3 = align64(Nn * 3), cf = egno_coef_floats(c);
  Carve w = {base, 0};
  EgnoBwdWs s;
  EgnoBwdSet &s0 = s.set[0], &s1 = s.set[1];
  s.wimg = w.take(wimg_floats(EGNO_WIMG_PER_LAYER * c->n_layers)); s.ttab = w.take(egno_table_floats(c));
  s.P = w.take(nh); s.Q = w.take(nh);
  s0.coef = w.take(cf); s.ycoef = w.take(cf); s0.gycoef = w.take(cf); s.gcoef = w.take(cf);
  s.ghA = w.take(nh); s0.gh = w.take(nh); s0.GU5 = w.take(nh); s0.GUV = w.take(nh); s.gM = w.take(nh); s0.gP = w.take(nh);
  s0.gQ = w.take(nh);
  s.gx[0] = w.take(n3); s.gx[1] = w.take(n3); s.gvA = w.take(n3); s.gvB = w.take(n3); s.gFsum = w.take(n3);
  s.arena[0] = w.take(NB_PARTIAL_FLOATS);
  s1.gh = w.take(nh); s1.GU5 = w.take(nh); s1.GUV = w.take(nh); s1.gP = w.take(nh); s1.gQ = w.take(nh);
  s1.coef = w.take(cf); s1.gycoef = w.take(cf);
  s.arena[1] = w.take(NB_PARTIAL_FLOATS);
  s.total = w.used;
  return s;
}

// input-gradient workspace of nb_egno_backward_ex: the per-row edge-feature gradients of every layer launch (each
// launch writes its own slice of T * B*N(N-1) * in_edge_nf floats, no read-modify-write across layers), then the
// embedding-output gradient summed over the T frames
static inline int64_t egno_edge_rows(const NbEgnoConfig* c) { return (int64_t)c->B * c->N * (c->N - 1); }
struct EgnoInputGradWs { float *gef_rows, *gh_sum; int64_t ef_slice, total; };
static EgnoInputGradWs egno_input_grad_ws(const NbEgnoConfig* c, float* base) {
  Carve w = {base, 0};
  EgnoInputGradWs s;
  s.ef_slice = (int64_t)c->T * egno_edge_rows(c) * c->in_edge_nf;
  s.gef_rows = w.take(align64(s.ef_slice * c->n_layers));
  s.gh_sum = w.take(align64((int64_t)c->B * c->N * NB_H));
  s.total = w.used;
  return s;
}

extern "C" int64_t nb_egno_workspace_floats(const NbEgnoConfig* cfg, int mode) {
  if (egno_validate(cfg) != NB_OK) return -1;
  if (mode < 0 || mode > 2) { nb_set_error("workspace mode must be 0 (inference), 1 (backward) or 2 (training forward)"); return -1; }
  if (mode == NB_WS_BACKWARD) return egno_bwd_ws(cfg, nullptr).total;
  return egno_fwd_ws(cfg, mode == NB_WS_FORWARD_INFER, nullptr).total;
}

extern "C" int64_t nb_egno_input_grad_workspace_floats(const NbEgnoConfig* cfg) {
  if (egno_validate(cfg) != NB_OK) return -1;
  return egno_input_grad_ws(cfg, nullptr).total;
}

// the 64 x 64 weight blocks the node GEMMs of a layer multiply with (forward: as stored; backward: transposed views of
// the same images): first edge layer's h_row / h_col columns, node_net layer 1 (h | M halves) and 2, node_v_net layer 1
static int egno_weight_images(const EgnoCtx& X, float* scratch) {
  const float* W[NB_MAX_LAYERS * EGNO_WIMG_PER_LAYER];
  int ld[NB_MAX_LAYERS * EGNO_WIMG_PER_LAYER];
  int n = 0;
  for (int l = 0; l < X.c->n_layers; ++l) {
    const EgnoLayerOff& L = X.lo.L[l];
    W[n] = X.params + L.e_w1 + 1; ld[n++] = X.lo.E;
    W[n] = X.params + L.e_w1 + 1 + NB_H; ld[n++] = X.lo.E;
    W[n] = X.params + L.n_w1; ld[n++] = 2 * NB_H;
    W[n] = X.params + L.n_w1 + NB_H; ld[n++] = 2 * NB_H;
    W[n] = X.params + L.n_w2; ld[n++] = NB_H;
    W[n] = X.params + L.v_w1; ld[n++] = NB_H;
  }
  return wimg_prepare(W, ld, n, scratch, X.st);
}

// ---- temporal conv on h: mixing GEMMs coef -> ycoef (shared by forward and the backward's recompute)
static int egno_tc_mix(const EgnoCtx& X, int l, const float* coef, float* ycoef) {
  const int modes = X.c->num_modes;
  const float* W = X.params + X.lo.L[l].tc;
  const int64_t plane = X.Nn0 * NB_H;
  const int64_t sk = (int64_t)NB_H * modes * 2, sn = (int64_t)modes * 2;  // B[k=i][n=o] = W[i][o][m][c]
  NbGemmArgs jobs[2 * NB_MAX_T];
  int nj = 0;
  for (int m = 0; m < modes; ++m) {
    int ci = nb_coef_index(X.tw, m);
    const float* Wr = W + m * 2;
    const float* Wi = W + m * 2 + 1;
    if (m == 0 || m == X.tw.nyq) {
      NbGemmArgs a = gemm_args((int)X.Nn0);
      a.nsrc = 1; a.src[0] = gsrc(coef + ci * plane, NB_H, 0, Wr, sk, sn);
      a.out = ycoef + ci * plane;
      jobs[nj++] = a;
    } else {
      NbGemmArgs a = gemm_args((int)X.Nn0);  // P = C Wr + S Wi
      a.nsrc = 2;
      a.src[0] = gsrc(coef + ci * plane, NB_H, 0, Wr, sk, sn);
      a.src[1] = gsrc(coef + (ci + 1) * plane, NB_H, 0, Wi, sk, sn);
      a.out = ycoef + ci * plane;
      jobs[nj++] = a;
      NbGemmArgs b = gemm_args((int)X.Nn0);  // Q = C Wi - S Wr
      b.nsrc = 2;
      b.src[0] = gsrc(coef + ci * plane, NB_H, 0, Wi, sk, sn);
      b.src[1] = gsrc(coef + (ci + 1) * plane, NB_H, 0, Wr, sk, sn, -1.f);
      b.out = ycoef + (ci + 1) * plane;
      jobs[nj++] = b;
    }
  }
  return launch_gemm_batch(jobs, nj, X.st, /*exact_fp32=*/true);
}

static NbDftArgs dft_args(const EgnoCtx& X) {
  NbDftArgs d;
  memset(&d, 0, sizeof(d));
  d.tw = X.tw;
  d.Nn0 = (int)X.Nn0;
  return d;
}

// fused temporal convolution kernels (k_tconv_fwd / k_tconv_bwd) serve num_modes <= 2, the configured case
static inline bool egno_tconv_fused(const EgnoCtx& X) { return X.c->num_modes <= 2; }
static NbTconvArgs tconv_args(const EgnoCtx& X, int l) {
  NbTconvArgs t;
  memset(&t, 0, sizeof(t));
  t.tw = X.tw;
  t.Nn0 = (int)X.Nn0;
  t.W = X.params + X.lo.L[l].tc;
  return t;
}
static inline int tconv_grid(const EgnoCtx& X, int per_sm) {
  return imin(cdiv(X.Nn0, NB_TCV_ROWS), (int64_t)per_sm * nb_num_sms());
}
// k_tconv_fwd / k_tconv_bwd are instantiated for T <= 10 (the configured case, smaller register arrays) and NB_MAX_T
static int launch_tconv(const EgnoCtx& X, const NbTconvArgs& tc, bool bwd) {
  const bool t10 = X.c->T <= 10;
  void (*k)(NbTconvArgs) = bwd ? (t10 ? k_tconv_bwd<10> : k_tconv_bwd<NB_MAX_T>) : (t10 ? k_tconv_fwd<10> : k_tconv_fwd<NB_MAX_T>);
  const size_t smem = bwd ? NB_TCONV_BWD_SMEM : NB_TCONV_FWD_SMEM;
  int pi = prof_begin(4, X.st);
  NB_SET_SMEM(k, smem);
  NB_LAUNCH_COUNTED(k, (unsigned)tconv_grid(X, bwd ? 2 : 3), 256, smem, X.st, tc);
  prof_end(4, pi, X.st);
  return nb_check_launch(bwd ? "k_tconv_bwd" : "k_tconv_fwd");
}

// the fused per-layer node kernels (nb_egno_node.cuh) need the tcgen05 variants and this call's weight images;
// nb_set_node_fused(0) keeps the generic GEMM launches
static bool egno_node_fused(const EgnoCtx& X) {
#ifndef NB_EMU
  return g_node_fused && g_node_impl == 1 && g_wimg.n == EGNO_WIMG_PER_LAYER * X.c->n_layers;
#else
  (void)X;
  return false;
#endif
}

static NbEdgeW egno_edge_w(const EgnoCtx& X, int l) {
  const EgnoLayerOff& L = X.lo.L[l];
  NbEdgeW w;
  w.W1 = X.params + L.e_w1; w.ldw1 = X.lo.E; w.col_rad = 0; w.col_ef = 1 + 2 * NB_H;
  w.W2 = X.params + L.e_w2; w.b2 = X.params + L.e_b2; w.W3 = X.params + L.c_w1; w.b3 = X.params + L.c_b1;
  w.w4 = X.params + L.c_w2; w.b4 = X.params + L.c_b2;
  return w;
}

// ---- EGNO stages: each makes its own choice between the fused kernel and the generic launches; egno_forward /
// egno_backward only order them around the stream fork / join and flush points.

// h = Linear([nodes | time embeddings]) (egno.py:72-76): inputs materialised 64 wide (scratch: P, Q), then one GEMM;
// and x, v replicated over T (egno.py:89-96)
static int egno_embed_fwd(const EgnoCtx& X, const float* nodes, const EgnoTimes& times, const EgnoFwdWs& ws,
                          const float* x, const float* v, const EgnoLayerBufs& b0) {
  NbEmbedArgs e;
  NB_TRY(egno_embed_inputs(X, e, nodes, times, ws.ttab, ws.P, ws.Q, X.st));
  NbGemmArgs ga = gemm_args((int)X.Nn);
  ga.nsrc = 1; ga.src[0] = gsrc(ws.P, NB_H, 0, X.params + X.lo.emb_w, 1, X.lo.F);
  ga.src[0].kmax = X.lo.F < NB_H ? X.lo.F : NB_H;
  if (X.lo.F > NB_H) {
    ga.nsrc = 2; ga.src[1] = gsrc(ws.Q, NB_H, 0, X.params + X.lo.emb_w + NB_H, 1, X.lo.F);
    ga.src[1].kmax = X.lo.F - NB_H;
  }
  ga.bias = X.params + X.lo.emb_b; ga.out = b0.h0;
  NB_TRY(launch_gemm(ga, X.st));
  const int n3 = (int)(X.Nn0 * 3);
  NB_LAUNCH_COUNTED(k_replicate3, (unsigned)ew_grid(X.Nn * 3), 256, 0, X.st, x, b0.x0, n3, X.c->T, X.fm);
  NB_LAUNCH_COUNTED(k_replicate3, (unsigned)ew_grid(X.Nn * 3), 256, 0, X.st, v, b0.v0, n3, X.c->T, X.fm);
  return nb_check_launch("k_replicate3");
}

// dW_emb = gh^T [nodes | time embeddings], db_emb = column sums of gh: the inputs re-materialised 64 wide in P, Q (unless
// `built` already) are reduced by the weight-gradient kernel; columns >= F are not written
static int egno_embed_bwd(const EgnoCtx& X, NbEmbedArgs& e, bool built, const float* nodes, const EgnoTimes& times,
                          const EgnoBwdWs& ws, const float* gh, float* grad) {
  if (!built) NB_TRY(egno_embed_inputs(X, e, nodes, times, ws.ttab, ws.P, ws.Q, X.st));
  const int F = X.lo.F;
  NB_TRY(wgrad_to((int)X.Nn, wpair(gh, ws.P), grad, X.lo.emb_w, F, 1, X.lo.emb_b, 0, X.st, F < NB_H ? F : NB_H));
  if (F > NB_H) NB_TRY(wgrad_to((int)X.Nn, wpair(gh, ws.Q), grad, X.lo.emb_w + NB_H, F, 1, -1, 0, X.st, F - NB_H));
  return NB_OK;
}

// (x - mean, v) <- (x - mean, v) + conv(.)     (egno.py:103-108, layer_no.py:151-178)
static NbTcxArgs tcx_args(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* v0, const float* loc_mean) {
  NbTcxArgs t;
  memset(&t, 0, sizeof(t));
  t.tw = X.tw; t.n3 = (int)(X.Nn0 * 3); t.x0 = b.x0; t.v0 = v0; t.mean = loc_mean; t.W = X.params + X.lo.L[l].tcx;
  for (int tt = 0; tt < NB_MAX_T; ++tt) t.tmap[tt] = X.fm.m[tt];
  return t;
}
static int egno_tcx_fwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* v0, const float* loc_mean, void* st) {
  NbTcxArgs t = tcx_args(X, l, b, v0, loc_mean);
  t.x1 = b.x1; t.v1 = b.v1;
  NB_LAUNCH_COUNTED(k_tcx_fwd, (unsigned)ew_grid(X.Nn0 * 3), 256, 0, st, t);
  return nb_check_launch("k_tcx_fwd");
}
// on `st`, its partials reduced by the next flush; dL/dloc_mean right behind it, where both planes are final
static int egno_tcx_bwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* v0, const float* loc_mean,
                        float* gx1, float* gv1, float* gx0, float* gv0, float* g_loc_mean, float* grad, void* st) {
  const int nw = 2 * 2 * X.c->num_modes * 2;
  NbTcxArgs t = tcx_args(X, l, b, v0, loc_mean);
  t.gx1 = gx1; t.gv1 = gv1; t.gx0 = gx0; t.gv0 = gv0;
  const int grid = imin(cdiv(X.Nn0 * 3, 256), 2 * nb_num_sms());
  NB_TRY(q_partial(&t.partial, (int64_t)grid * nw, X.st));
  NB_LAUNCH_COUNTED(k_tcx_bwd, (unsigned)grid, 256, 0, st, t);
  NB_TRY(nb_check_launch("k_tcx_bwd"));
  if (g_loc_mean) {
    NB_LAUNCH_COUNTED(k_loc_mean_grad, (unsigned)ew_grid(X.Nn0 * 3), 256, 0, st, (const float*)gx1, (const float*)gx0,
                      g_loc_mean, (int)(X.Nn0 * 3), X.c->T, l == X.c->n_layers - 1 ? 0 : 1);
    NB_TRY(nb_check_launch("k_loc_mean_grad"));
  }
  return q_finalize(t.partial, grid, nw, grad, 0, {fseg(0, nw, nw, X.lo.L[l].tcx, 0, 1)}, X.st);
}

// h1 = h0 + LeakyReLU(conv(h0))      (layer_no.py:96-126): the fused kernel (mask: the LeakyReLU's sign bits for the
// backward, training only), or DFT, mode-mixing GEMMs and inverse DFT through coef / ycoef
static int egno_tconv_fwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, uint32_t* mask, float* coef, float* ycoef) {
  if (egno_tconv_fused(X)) {
    NbTconvArgs tc = tconv_args(X, l);
    tc.x = b.h0; tc.out = b.h1; tc.mask = mask;
    return launch_tconv(X, tc, false);
  }
  NbDftArgs d = dft_args(X);
  d.x = b.h0; d.coef = coef;
  NB_LAUNCH_COUNTED(k_dft_fwd, (unsigned)ew_grid(X.Nn0 * 16), 256, 0, X.st, d);
  NB_TRY(nb_check_launch("k_dft_fwd"));
  NB_TRY(egno_tc_mix(X, l, coef, ycoef));
  d.ycoef = ycoef; d.out = b.h1;
  NB_LAUNCH_COUNTED(k_idft_fwd, (unsigned)ew_grid(X.Nn0 * 16), 256, 0, X.st, d);
  return nb_check_launch("k_idft_fwd");
}
// its backward dL/dh1 (gout) -> dL/dh0 (S.gh) and the mixing weight gradients: reduced by the next flush after the fused
// kernel, here in the generic path (before the inverse DFT overwrites S.gh, which queued jobs of the layer above read)
static int egno_tconv_bwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* gout, const EgnoBwdSet& S,
                          const EgnoBwdWs& ws, float* grad) {
  const int modes = X.c->num_modes;
  const bool fused = egno_tconv_fused(X);
  NbDftArgs d = dft_args(X);
  if (fused) {
    NbTconvArgs tc = tconv_args(X, l);
    tc.x = b.h0; tc.gout = gout; tc.gx = S.gh; tc.coef = S.coef; tc.gycoef = S.gycoef; tc.mask = b.tmask;
    NB_TRY(launch_tconv(X, tc, true));
  } else {
    d.x = b.h0; d.coef = S.coef;
    NB_LAUNCH_COUNTED(k_dft_fwd, (unsigned)ew_grid(X.Nn0 * 16), 256, 0, X.st, d);
    NB_TRY(nb_check_launch("k_dft_fwd"));
    NB_TRY(egno_tc_mix(X, l, S.coef, ws.ycoef));
    d.ycoef = ws.ycoef; d.gout = gout; d.gycoef = S.gycoef;
    NB_LAUNCH_COUNTED(k_idft_bwd, (unsigned)ew_grid(X.Nn0 * 16), 256, 0, X.st, d);
    NB_TRY(nb_check_launch("k_idft_bwd"));
  }
  const float* W = X.params + X.lo.L[l].tc;
  const int64_t plane = X.Nn0 * NB_H;
  const int64_t tk = (int64_t)modes * 2, tn = (int64_t)NB_H * modes * 2;  // B[k=o][n=i] = W[i][o][m][c]
  NbGemmArgs gj[2 * NB_MAX_T];
  int ngj = 0;
  for (int m = 0; m < modes; ++m) {
    int ci = nb_coef_index(X.tw, m);
    const float *Wr = W + m * 2, *Wi = W + m * 2 + 1;
    const float *C = S.coef + ci * plane, *Sn = S.coef + (ci + 1) * plane;
    const float *gPm = S.gycoef + ci * plane, *gQm = S.gycoef + (ci + 1) * plane;
    const int64_t wr_off = X.lo.L[l].tc + m * 2, wi_off = X.lo.L[l].tc + m * 2 + 1;
    if (m == 0 || m == X.tw.nyq) {
      if (!fused) {
        NbGemmArgs a = gemm_args((int)X.Nn0);  // gC = gP Wr^T
        a.nsrc = 1; a.src[0] = gsrc(gPm, NB_H, 0, Wr, tk, tn);
        a.out = ws.gcoef + ci * plane;
        gj[ngj++] = a;
      }
      NB_TRY(wgrad_to((int)X.Nn0, wpair(C, gPm), grad, wr_off, tn, tk, -1, 0, X.st));
    } else {
      if (!fused) {
        NbGemmArgs a = gemm_args((int)X.Nn0);  // gC = gP Wr^T + gQ Wi^T
        a.nsrc = 2;
        a.src[0] = gsrc(gPm, NB_H, 0, Wr, tk, tn);
        a.src[1] = gsrc(gQm, NB_H, 0, Wi, tk, tn);
        a.out = ws.gcoef + ci * plane;
        gj[ngj++] = a;
        NbGemmArgs s2 = gemm_args((int)X.Nn0);  // gS = gP Wi^T - gQ Wr^T
        s2.nsrc = 2;
        s2.src[0] = gsrc(gPm, NB_H, 0, Wi, tk, tn);
        s2.src[1] = gsrc(gQm, NB_H, 0, Wr, tk, tn, -1.f);
        s2.out = ws.gcoef + (ci + 1) * plane;
        gj[ngj++] = s2;
      }
      // dWr[i][o] = sum C_i gP_o - S_i gQ_o ; dWi[i][o] = sum S_i gP_o + C_i gQ_o
      NB_TRY(wgrad_to((int)X.Nn0, 2, wpair(C, gPm), wpair(Sn, gQm, 0, -1.f), grad, wr_off, tn, tk, -1, 0, X.st));
      NB_TRY(wgrad_to((int)X.Nn0, 2, wpair(Sn, gPm), wpair(C, gQm), grad, wi_off, tn, tk, -1, 0, X.st));
    }
  }
  if (fused) return NB_OK;
  NB_TRY(launch_gemm_batch(gj, ngj, X.st));
  NB_TRY(q_flush(X.st));
  d.gcoef = ws.gcoef; d.gx = S.gh;
  NB_LAUNCH_COUNTED(k_dft_bwd, (unsigned)ew_grid(X.Nn0 * 16), 256, 0, X.st, d);
  return nb_check_launch("k_dft_bwd");
}

#ifndef NB_EMU
template <bool FWD>
static int launch_egno_pair(const EgnoCtx& X, const NbEgnoPairArgs& pa) {
  NB_SET_SMEM(k_egno_pair<FWD>, NB_EPR_SMEM);
  int pi = prof_begin(2, X.st);
  NB_LAUNCH_COUNTED(k_egno_pair<FWD>, (unsigned)imin(cdiv(X.Nn, NB_TILE), 2 * nb_num_sms()), NB_THREADS, NB_EPR_SMEM, X.st, pa);
  prof_end(2, pi, X.st);
  return nb_check_launch("k_egno_pair");
}
#endif
// P = h W1[:, h_row]^T + b1, Q = h W1[:, h_col]^T: the per-node halves of the first edge layer (basic.py:98,170)
static int egno_pq(const EgnoCtx& X, int l, const float* h1, float* P, float* Q) {
  const EgnoLayerOff& L = X.lo.L[l];
  const int E = X.lo.E;
#ifndef NB_EMU
  if (egno_node_fused(X)) {
    NbEgnoPairArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.rows = (int)X.Nn; pa.img = g_wimg.img[EGNO_WIMG_PER_LAYER * l]; pa.A0 = h1; pa.bias = X.params + L.e_b1; pa.O0 = P; pa.O1 = Q;
    return launch_egno_pair<true>(X, pa);
  }
#endif
  NbGemmArgs a = gemm_args((int)X.Nn);  // P = h W1[:, h_row]^T + b1   (cols 1..64, basic.py:98,170)
  a.nsrc = 1; a.src[0] = gsrc(h1, NB_H, 0, X.params + L.e_w1 + 1, 1, E);
  a.bias = X.params + L.e_b1; a.out = P;
  NbGemmArgs b = gemm_args((int)X.Nn);  // Q = h W1[:, h_col]^T         (cols 65..128)
  b.nsrc = 1; b.src[0] = gsrc(h1, NB_H, 0, X.params + L.e_w1 + 1 + NB_H, 1, E);
  b.out = Q;
  NbGemmArgs ab[2] = {a, b};
  return launch_gemm_batch(ab, 2, X.st);
}
// its backward: gh1 += gP W1[:, h_row] + gQ W1[:, h_col], and the weight gradients
static int egno_pair_bwd(const EgnoCtx& X, int l, const float* h1, const float* gP, const float* gQ, float* gh1, float* grad) {
  const EgnoLayerOff& L = X.lo.L[l];
#ifndef NB_EMU
  if (egno_node_fused(X)) {
    NbEgnoPairArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.rows = (int)X.Nn; pa.img = g_wimg.img[EGNO_WIMG_PER_LAYER * l]; pa.A0 = gP; pa.A1 = gQ; pa.O0 = gh1;
    NB_TRY(launch_egno_pair<false>(X, pa));
  } else
#endif
  {
    NbGemmArgs a = gemm_args((int)X.Nn);
    a.nsrc = 2;
    a.src[0] = gsrc(gP, NB_H, 0, X.params + L.e_w1 + 1, X.lo.E, 1);
    a.src[1] = gsrc(gQ, NB_H, 0, X.params + L.e_w1 + 1 + NB_H, X.lo.E, 1);
    a.out = gh1; a.accumulate = 1;
    NB_TRY(launch_gemm(a, X.st));
  }
  NB_TRY(wgrad_to((int)X.Nn, wpair(gP, h1), grad, L.e_w1 + 1, X.lo.E, 1, L.e_b1, 0, X.st));
  return wgrad_to((int)X.Nn, wpair(gQ, h1), grad, L.e_w1 + 1 + NB_H, X.lo.E, 1, -1, 0, X.st);
}

// node_net, node_v_net and the coordinate update (basic.py:181-186): one pass over the rows (nb_egno_node.cuh), or the
// generic GEMMs and k_egno_xupd_fwd.  U5, UV are kept for the backward (fused inference: on chip only)
static int egno_node_fwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* h1, const float* x1,
                         const float* v1, bool train, float* h_next, float* x_next) {
  const EgnoLayerOff& L = X.lo.L[l];
  const float* params = X.params;
  const int64_t Nn = X.Nn;
#ifndef NB_EMU
  if (egno_node_fused(X)) {
    NbEgnoNodeFwdArgs na;
    memset(&na, 0, sizeof(na));
    na.rows = (int)Nn; na.N = X.c->N; na.img = g_wimg.img[EGNO_WIMG_PER_LAYER * l + 2];
    na.h = h1; na.M = b.M; na.b5 = params + L.n_b1; na.b6 = params + L.n_b2; na.bv1 = params + L.v_b1;
    na.wv2 = params + L.v_w2; na.bv2 = params + L.v_b2; na.x = x1; na.v = v1; na.Fsum = b.Fsum;
    na.U5 = train ? b.U5 : nullptr; na.UV = train ? b.UV : nullptr;
    na.h_out = h_next; na.x_out = x_next;
    NB_SET_SMEM(k_egno_node_fwd, NB_ENF_SMEM);
    int pi = prof_begin(6, X.st);
    NB_LAUNCH_COUNTED(k_egno_node_fwd, (unsigned)imin(cdiv(Nn, NB_TILE), 2 * nb_num_sms()), NB_THREADS, NB_ENF_SMEM, X.st, na);
    prof_end(6, pi, X.st);
    return nb_check_launch("k_egno_node_fwd");
  }
#endif
  NbGemmArgs a = gemm_args((int)Nn);  // U5 = [h, M] W5^T + b5      (basic.py:183-185)
  a.nsrc = 2;
  a.src[0] = gsrc(h1, NB_H, 0, params + L.n_w1, 1, 2 * NB_H);
  a.src[1] = gsrc(b.M, NB_H, 0, params + L.n_w1 + NB_H, 1, 2 * NB_H);
  a.bias = params + L.n_b1; a.out_pre = b.U5;
  NbGemmArgs u = gemm_args((int)Nn);  // UV = h Wv1^T + bv1         (node_v_net, pre-update h)
  u.nsrc = 1; u.src[0] = gsrc(h1, NB_H, 0, params + L.v_w1, 1, NB_H);
  u.bias = params + L.v_b1; u.out_pre = b.UV;
  NbGemmArgs au[2] = {a, u};
  NB_TRY(launch_gemm_batch(au, 2, X.st));
  NbGemmArgs c2 = gemm_args((int)Nn);  // h' = SiLU(U5) W6^T + b6  (no residual)
  c2.nsrc = 1; c2.src[0] = gsrc(b.U5, NB_H, 1, params + L.n_w2, 1, NB_H);
  c2.bias = params + L.n_b2; c2.out = h_next;
  NB_TRY(launch_gemm(c2, X.st));
  NbXupdArgs xa;
  memset(&xa, 0, sizeof(xa));
  xa.rows = Nn; xa.N = X.c->N; xa.x = x1; xa.v = v1; xa.UV = b.UV; xa.w2 = params + L.v_w2; xa.b2 = params + L.v_b2;
  xa.Fsum = b.Fsum; xa.x_out = x_next;
  NB_LAUNCH_COUNTED(k_egno_xupd_fwd, (unsigned)imin(cdiv(Nn, 8), 8 * nb_num_sms()), 256, 0, X.st, xa);
  return nb_check_launch("k_egno_xupd_fwd");
}
// its backward: x' = x + s v + clamp(mean f) gives dL/dv1 (gv_out), dL/dFsum, dL/dUV and the 64->1 head of node_v_net;
// node_net backwards gives GU5, dL/dh1 (gh1) and dL/dM.  One pass over the rows, or k_egno_xupd_bwd and the generic GEMMs
static int egno_node_bwd(const EgnoCtx& X, int l, const EgnoLayerBufs& b, const float* h1, const float* gh_in, float* gx,
                         const float* gv_in, float* gv_out, const EgnoBwdSet& S, const EgnoBwdWs& ws, float* gh1, float* grad) {
  const EgnoLayerOff& L = X.lo.L[l];
  const float* params = X.params;
  const int64_t Nn = X.Nn;
  const bool fused = egno_node_fused(X);
  const int grid = fused ? imin(cdiv(Nn, NB_TILE), 2 * nb_num_sms()) : imin(cdiv(Nn, 8), 4 * nb_num_sms());
  float* partial;
  NB_TRY(q_partial(&partial, (int64_t)grid * 65, X.st));
#ifndef NB_EMU
  if (fused) {
    NbEgnoNodeBwdArgs na;
    memset(&na, 0, sizeof(na));
    na.rows = (int)Nn; na.N = X.c->N; na.img = g_wimg.img[EGNO_WIMG_PER_LAYER * l + 2];
    na.gh = gh_in; na.U5 = b.U5; na.UV = b.UV; na.wv2 = params + L.v_w2; na.bv2 = params + L.v_b2;
    na.gx = gx; na.gv = gv_in; na.v = b.v1; na.Fsum = b.Fsum; na.gv_out = gv_out; na.gFsum = ws.gFsum;
    na.GU5 = S.GU5; na.GUV = S.GUV; na.gh1 = gh1; na.gM = ws.gM; na.partial = partial;
    NB_SET_SMEM(k_egno_node_bwd, NB_ENB_SMEM);
    int pi = prof_begin(7, X.st);
    NB_LAUNCH_COUNTED(k_egno_node_bwd, (unsigned)grid, NB_THREADS, NB_ENB_SMEM, X.st, na);
    prof_end(7, pi, X.st);
    NB_TRY(nb_check_launch("k_egno_node_bwd"));
  } else
#endif
  {
    NbXupdArgs xa;
    memset(&xa, 0, sizeof(xa));
    xa.rows = Nn; xa.N = X.c->N; xa.v = b.v1; xa.UV = b.UV; xa.w2 = params + L.v_w2; xa.b2 = params + L.v_b2;
    xa.Fsum = b.Fsum; xa.gx = gx; xa.gv = gv_in; xa.gv_out = gv_out; xa.gFsum = ws.gFsum; xa.GUV = S.GUV;
    xa.partial = partial;
    NB_LAUNCH_COUNTED(k_egno_xupd_bwd, (unsigned)grid, 256, 0, X.st, xa);
    NB_TRY(nb_check_launch("k_egno_xupd_bwd"));
    NbGemmArgs a = gemm_args((int)Nn);  // GU5 = (gh W6) * SiLU'(U5)
    a.nsrc = 1; a.src[0] = gsrc(gh_in, NB_H, 0, params + L.n_w2, NB_H, 1);
    a.epi = NB_EPI_MUL_DSILU; a.U = b.U5; a.out = S.GU5;
    NB_TRY(launch_gemm(a, X.st));
    NbGemmArgs g1 = gemm_args((int)Nn);  // gh1 = GU5 W5[:, :64] + GUV Wv1
    g1.nsrc = 2;
    g1.src[0] = gsrc(S.GU5, NB_H, 0, params + L.n_w1, 2 * NB_H, 1);
    g1.src[1] = gsrc(S.GUV, NB_H, 0, params + L.v_w1, NB_H, 1);
    g1.out = gh1;
    NbGemmArgs g2 = gemm_args((int)Nn);  // gM = GU5 W5[:, 64:]
    g2.nsrc = 1; g2.src[0] = gsrc(S.GU5, NB_H, 0, params + L.n_w1 + NB_H, 2 * NB_H, 1);
    g2.out = ws.gM;
    NbGemmArgs g12[2] = {g1, g2};
    NB_TRY(launch_gemm_batch(g12, 2, X.st));
  }
  NB_TRY(q_finalize(partial, grid, 65, grad, 0, {fseg(0, NB_H, NB_H, L.v_w2, 0, 1), fseg(NB_H, 1, 1, L.v_b2, 0, 0)}, X.st));
  NB_TRY(wgrad_to((int)Nn, wpair(gh_in, b.U5, 1), grad, L.n_w2, NB_H, 1, L.n_b2, 0, X.st));
  NB_TRY(wgrad_to((int)Nn, wpair(S.GU5, h1), grad, L.n_w1, 2 * NB_H, 1, L.n_b1, 0, X.st));
  NB_TRY(wgrad_to((int)Nn, wpair(S.GU5, b.M), grad, L.n_w1 + NB_H, 2 * NB_H, 1, -1, 0, X.st));
  return wgrad_to((int)Nn, wpair(S.GUV, h1), grad, L.v_w1, NB_H, 1, L.v_b1, 0, X.st);
}

static int egno_forward(const NbEgnoConfig* cfg, const float* params, const float* x, const float* nodes,
                        const float* edge_fea, const float* v, const float* loc_mean, const EgnoTimes& times,
                        float* x_out, float* v_out, float* h_out, float* saved, float* workspace, void* stream) {
  NB_RANGE("nb_egno_forward");
  EgnoCtx X;
  NB_TRY(egno_ctx_init(&X, cfg, params, stream));
  const int Ln = cfg->n_layers;
  const int64_t lf = align64(egno_layer_floats(X.Nn, X.Nn0));
  const EgnoFwdWs ws = egno_fwd_ws(cfg, !saved, workspace);
  WimgGuard wimg_guard;
  NB_TRY(egno_weight_images(X, ws.wimg));
  // training keeps every layer's buffers in `saved`; inference alternates two sets in the workspace
  auto bufs = [&](int l) { return egno_layer_bufs(saved ? saved + (int64_t)l * lf : ws.infer + (int64_t)(l & 1) * lf, X.Nn); };

  NB_TRY(egno_embed_fwd(X, nodes, times, ws, x, v, bufs(0)));
  const float* v_prev = bufs(0).v0;
  for (int l = 0; l < Ln; ++l) {
    EgnoLayerBufs b = bufs(l);
    const float *h1 = b.h0, *x1 = b.x0;
    void* side = stream;
    if (cfg->use_time_conv) {
      // the (x - mean, v) convolution is independent of the h path until the edge kernel: it runs on the side stream
      // underneath the 64-channel convolution and the P | Q product
      side = side_fork(stream);
      NB_TRY(egno_tcx_fwd(X, l, b, v_prev, loc_mean, side));
      NB_TRY(egno_tconv_fwd(X, l, b, saved ? b.tmask : nullptr, ws.coef, ws.ycoef));
      h1 = b.h1; x1 = b.x1;
    } else {
      cudaMemcpyAsync(b.v1, v_prev, X.Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    }
    // ---- EGNN layer (basic.py:167-186)
    float* P = saved ? b.P : ws.P;  // training: kept for the backward edge tile
    float* Q = saved ? b.Q : ws.Q;
    NB_TRY(egno_pq(X, l, h1, P, Q));
    side_join(side, stream);
    NbEdgeFwdArgs ea;
    ea.g = egno_edge_geom(X);
    ea.w = egno_edge_w(X, l);
    ea.x = x1; ea.P = P; ea.Q = Q; ea.ef = edge_fea; ea.M = b.M; ea.Fsum = b.Fsum;
    NB_TRY(launch_edge_fwd(ea, stream));
    const bool last = l + 1 == Ln;
    NB_TRY(egno_node_fwd(X, l, b, h1, x1, b.v1, saved != nullptr, last ? h_out : bufs(l + 1).h0, last ? x_out : bufs(l + 1).x0));
    v_prev = b.v1;
  }
  cudaMemcpyAsync(v_out, v_prev, X.Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
  return nb_check_launch("nb_egno_forward");
}

extern "C" int nb_egno_forward(const NbEgnoConfig* cfg, const float* params, const float* x, const float* nodes,
                               const float* edge_fea, const float* v, const float* loc_mean,
                               const int64_t* timesteps_out, const int64_t* timesteps_in, float* x_out, float* v_out,
                               float* h_out, float* saved, float* workspace, void* stream) {
  const EgnoTimes times = {timesteps_out, timesteps_in, nullptr, nullptr};
  return egno_forward(cfg, params, x, nodes, edge_fea, v, loc_mean, times, x_out, v_out, h_out, saved, workspace, stream);
}

extern "C" int nb_egno_forward_ft(const NbEgnoConfig* cfg, const float* params, const float* x, const float* nodes,
                                  const float* edge_fea, const float* v, const float* loc_mean, const float* timesteps_out,
                                  const float* timesteps_in, float* x_out, float* v_out, float* h_out, float* saved,
                                  float* workspace, void* stream) {
  const EgnoTimes times = {nullptr, nullptr, timesteps_out, timesteps_in};
  return egno_forward(cfg, params, x, nodes, edge_fea, v, loc_mean, times, x_out, v_out, h_out, saved, workspace, stream);
}

static int egno_backward(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                         const float* loc_mean, const EgnoTimes& times, const float* saved, const float* g_x_out,
                         const float* g_v_out, const float* g_h_out, float* grad_params, float* g_x_in, float* g_v_in,
                         float* g_nodes, float* g_edge_fea, float* g_loc_mean, float* g_t_out, float* g_t_in,
                         float* workspace, float* input_grad_workspace, void* stream) {
  NB_RANGE("nb_egno_backward");
  EgnoCtx X;
  NB_TRY(egno_ctx_init(&X, cfg, params, stream));
  if (!saved) { nb_set_error("nb_egno_backward needs the saved buffer of a forward call"); return NB_ERR_INVALID; }
  const int T = cfg->T, Ln = cfg->n_layers;
  const int64_t Nn = X.Nn, Nn0 = X.Nn0;
  // input gradients (single input frame only): per-row edge-feature gradients of every layer, summed at the end
  const bool want_ef = g_edge_fea && cfg->in_edge_nf > 0;
  if ((g_nodes || g_edge_fea || g_loc_mean) && X.fm.L > 1) {
    nb_set_error("gradients w.r.t. nodes / edge_fea / loc_mean are implemented for num_inputs = 1 only");
    return NB_ERR_INVALID;
  }
  if ((g_t_out || g_t_in) && !times.fout) {
    nb_set_error("time gradients need floating-point times (nb_egno_backward_ft)");
    return NB_ERR_INVALID;
  }
  if (g_t_in && X.fm.L == 1) {
    nb_set_error("g_t_in needs num_inputs > 1 (a single input frame has no input times)");
    return NB_ERR_INVALID;
  }
  if ((g_nodes || want_ef) && !input_grad_workspace) {
    nb_set_error("nb_egno_backward_ex needs the input-gradient workspace (nb_egno_input_grad_workspace_floats)");
    return NB_ERR_INVALID;
  }
  const EgnoInputGradWs iws = egno_input_grad_ws(cfg, input_grad_workspace);
  const int64_t lf = align64(egno_layer_floats(Nn, Nn0));
  EgnoBwdWs ws = egno_bwd_ws(cfg, workspace);
  WimgGuard wimg_guard;
  NB_TRY(egno_weight_images(X, ws.wimg));
  DeferState D = {cfg->use_time_conv && egno_tconv_fused(X) && defer_available(), 0, ws.arena};
  q_begin(ws.arena[0], NB_PARTIAL_FLOATS);
  // deferred flushes: layer l writes set l & 1, its queued jobs read that set and the gh / spectral planes of the other
  auto set_of = [&](int l) -> EgnoBwdSet& { return ws.set[D.on ? l & 1 : 0]; };
  auto layer = [&](int l) { return egno_layer_bufs(const_cast<float*>(saved) + (int64_t)l * lf, Nn); };
  cudaStream_t cst = (cudaStream_t)stream;

  cudaMemsetAsync(grad_params, 0, X.lo.total * sizeof(float), cst);
  // incoming gradients: gx must be writable (the edge backward accumulates into it)
  int gxi = 0;
  if (g_x_out) cudaMemcpyAsync(ws.gx[0], g_x_out, Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  else cudaMemsetAsync(ws.gx[0], 0, Nn * 3 * sizeof(float), cst);
  const float* gv_in = g_v_out;
  if (!gv_in) { cudaMemsetAsync(ws.gvA, 0, Nn * 3 * sizeof(float), cst); gv_in = ws.gvA; }
  // the embedding layer's inputs (re-materialised for its weight gradient at the very end) depend on nothing but the
  // call's inputs: with the second stream they are built there now, off the dependent chain
  NbEmbedArgs emb_args;
  if (D.on) NB_TRY(egno_embed_inputs(X, emb_args, nodes, times, ws.ttab, ws.P, ws.Q, side2_fork(stream)));
  const float* gh_in = g_h_out;
  if (!gh_in) {   // in the set "layer Ln" would have written
    gh_in = set_of(Ln).gh;
    cudaMemsetAsync(set_of(Ln).gh, 0, Nn * NB_H * sizeof(float), cst);
  }

  for (int l = Ln - 1; l >= 0; --l) {
    EgnoBwdSet& S = set_of(l);
    const EgnoLayerBufs b = layer(l);
    const float* h1 = cfg->use_time_conv ? b.h1 : b.h0;
    const float* x1 = cfg->use_time_conv ? b.x1 : b.x0;
    float* gx = ws.gx[gxi];
    // 1 + 2. coordinate update, node_v_net and node_net backwards
    NB_TRY(egno_node_bwd(X, l, b, h1, gh_in, gx, gv_in, ws.gvB, S, ws, ws.ghA, grad_params));
    // 3. edge tile backward (recompute from the saved P, Q)
    {
      NbEdgeBwdArgs ea;
      memset(&ea, 0, sizeof(ea));
      ea.g = egno_edge_geom(X);
      ea.w = egno_edge_w(X, l);
      ea.x = x1; ea.P = b.P; ea.Q = b.Q; ea.ef = edge_fea; ea.gM = ws.gM; ea.gFsum = ws.gFsum; ea.gP = S.gP; ea.gQ = S.gQ; ea.gx = gx;
      if (want_ef) ea.gef = iws.gef_rows + (int64_t)l * iws.ef_slice;
      const EgnoLayerOff& L = X.lo.L[l];
      EdgeGradDst d;
      d.w1 = L.e_w1; d.W2 = L.e_w2; d.b2 = L.e_b2; d.W3 = L.c_w1; d.b3 = L.c_b1; d.w4 = L.c_w2; d.b4 = L.c_b2;
      d.ldw1 = X.lo.E; d.col_rad = 0; d.col_ef = 1 + 2 * NB_H; d.b_unused = 0;
      NB_TRY(launch_edge_bwd(ea, grad_params, d, 0, stream));
    }
    // 4. pre-projection backward
    NB_TRY(egno_pair_bwd(X, l, h1, S.gP, S.gQ, ws.ghA, grad_params));
    // 5. temporal convolutions
    if (cfg->use_time_conv) {
      void* side = stream;
      if (egno_tconv_fused(X)) {
        // queued weight-gradient jobs read gh_in (= S.gh of the layer above), GU5, gP, ...: run them before S.gh is
        // overwritten.  The spectral weight gradients of THIS layer are queued after the kernel that produces their
        // operands (coef, gycoef) and run with the next flush, before those planes are overwritten again.
        NB_TRY(defer_flush(D, stream));
        // the 2-channel convolution's backward is independent of the 64-channel one: side stream, joined after it;
        // its partial slice is reduced by the next flush (on the caller's stream, after the join)
        side = side_fork(stream);
      }
      const float* v0 = l == 0 ? b.v0 : layer(l - 1).v1;
      NB_TRY(egno_tcx_bwd(X, l, b, v0, loc_mean, gx, ws.gvB, ws.gx[gxi ^ 1], ws.gvA, g_loc_mean, grad_params, side));
      gxi ^= 1;
      gv_in = ws.gvA;
      NB_TRY(egno_tconv_bwd(X, l, b, ws.ghA, S, ws, grad_params));
      side_join(side, stream);
      gh_in = S.gh;
    } else {
      NB_TRY(q_flush(stream));
      // without the temporal conv gv1 must survive in gvB while the next layer writes its own gv1: swap roles (gh too)
      gv_in = ws.gvB;
      std::swap(ws.gvA, ws.gvB);
      gh_in = ws.ghA;
      std::swap(ws.ghA, S.gh);
    }
  }
  // ---- embedding backward and the reduction of the T replicas of x, v
  NB_TRY(egno_embed_bwd(X, emb_args, D.on, nodes, times, ws, gh_in, grad_params));
  NB_TRY(defer_flush(D, stream));
  const NbFrameMap& fm = X.fm;
  if (g_x_in) NB_LAUNCH_COUNTED(k_sum_over_t, (unsigned)ew_grid(Nn0 * 3 * fm.L), 256, 0, stream, (const float*)ws.gx[gxi], g_x_in, (int)(Nn0 * 3), T, fm);
  if (g_v_in) NB_LAUNCH_COUNTED(k_sum_over_t, (unsigned)ew_grid(Nn0 * 3 * fm.L), 256, 0, stream, gv_in, g_v_in, (int)(Nn0 * 3), T, fm);
  if (g_nodes) {   // dL/dnodes = (sum_t dL/dh_emb[t]) W_emb[:, :in_node_nf]
    NB_LAUNCH_COUNTED(k_sum_over_t, (unsigned)ew_grid(Nn0 * NB_H), 256, 0, stream, gh_in, iws.gh_sum, (int)(Nn0 * NB_H), T, fm);
    NB_LAUNCH_COUNTED(k_embed_input_grad, (unsigned)ew_grid(Nn0 * cfg->in_node_nf), 256, 0, stream, (const float*)iws.gh_sum,
                      params + X.lo.emb_w, X.lo.F, cfg->in_node_nf, Nn0, g_nodes);
  }
  if (want_ef)     // fixed-order sum over the n_layers * T slices of B*N(N-1) rows
    NB_LAUNCH_COUNTED(k_sum_slices, (unsigned)ew_grid(egno_edge_rows(cfg) * cfg->in_edge_nf), 256, 0, stream,
                      (const float*)iws.gef_rows, g_edge_fea, egno_edge_rows(cfg) * cfg->in_edge_nf, Ln * T);
  if (g_loc_mean && !cfg->use_time_conv) cudaMemsetAsync(g_loc_mean, 0, Nn0 * 3 * sizeof(float), cst);
  if (g_t_out || g_t_in) {   // dL/dtimes from the same gh_in as the embedding's weight gradient
    if (cfg->time_emb_dim == 0) {   // the times are unused
      if (g_t_out) cudaMemsetAsync(g_t_out, 0, (int64_t)cfg->B * T * sizeof(float), cst);
    } else {
      NB_LAUNCH_COUNTED(k_time_grad, (unsigned)cfg->B, NB_TGRAD_THREADS, 0, stream, emb_args, times.fout, times.fin, gh_in,
                        params + X.lo.emb_w, X.lo.F, g_t_out, g_t_in);
      NB_TRY(nb_check_launch("k_time_grad"));
    }
  }
  defer_join(D, stream);
  return nb_check_launch("nb_egno_backward");
}

extern "C" int nb_egno_backward(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                                const float* loc_mean, const int64_t* timesteps_out, const int64_t* timesteps_in,
                                const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                                float* grad_params, float* g_x_in, float* g_v_in, float* workspace, void* stream) {
  return nb_egno_backward_ex(cfg, params, nodes, edge_fea, loc_mean, timesteps_out, timesteps_in, saved, g_x_out, g_v_out,
                             g_h_out, grad_params, g_x_in, g_v_in, nullptr, nullptr, nullptr, workspace, nullptr, stream);
}

extern "C" int nb_egno_backward_ex(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                                   const float* loc_mean, const int64_t* timesteps_out, const int64_t* timesteps_in,
                                   const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                                   float* grad_params, float* g_x_in, float* g_v_in, float* g_nodes, float* g_edge_fea,
                                   float* g_loc_mean, float* workspace, float* input_grad_workspace, void* stream) {
  const EgnoTimes times = {timesteps_out, timesteps_in, nullptr, nullptr};
  return egno_backward(cfg, params, nodes, edge_fea, loc_mean, times, saved, g_x_out, g_v_out, g_h_out, grad_params,
                       g_x_in, g_v_in, g_nodes, g_edge_fea, g_loc_mean, nullptr, nullptr, workspace, input_grad_workspace,
                       stream);
}

extern "C" int nb_egno_backward_ft(const NbEgnoConfig* cfg, const float* params, const float* nodes, const float* edge_fea,
                                   const float* loc_mean, const float* timesteps_out, const float* timesteps_in,
                                   const float* saved, const float* g_x_out, const float* g_v_out, const float* g_h_out,
                                   float* grad_params, float* g_x_in, float* g_v_in, float* g_nodes, float* g_edge_fea,
                                   float* g_loc_mean, float* g_t_out, float* g_t_in, float* workspace,
                                   float* input_grad_workspace, void* stream) {
  const EgnoTimes times = {nullptr, nullptr, timesteps_out, timesteps_in};
  return egno_backward(cfg, params, nodes, edge_fea, loc_mean, times, saved, g_x_out, g_v_out, g_h_out, grad_params,
                       g_x_in, g_v_in, g_nodes, g_edge_fea, g_loc_mean, g_t_out, g_t_in, workspace, input_grad_workspace,
                       stream);
}

// ============================================================================= SEGNO
struct SegnoLayout {
  int E;
  int64_t emb_w, emb_b, e_w1, e_b1, e_w2, e_b2, n_w1, n_b1, n_w2, n_b2, c_w1, c_b1, c_w2, c_b2, cv_w1, cv_b1, cv_w2,
      cv_b2, total;
};

static int segno_validate(const NbSegnoConfig* c) {
  if (!c) { nb_set_error("null config"); return NB_ERR_INVALID; }
  if (c->B < 1 || c->N < 2 || c->N > NB_MAX_NODES) { nb_set_error("unsupported B=%d N=%d (2 <= N <= %d)", c->B, c->N, NB_MAX_NODES); return NB_ERR_INVALID; }
  if (c->T < 1 || c->T > 4096) { nb_set_error("unsupported T=%d", c->T); return NB_ERR_INVALID; }
  if (c->in_edge_nf < 0 || c->in_edge_nf > NB_MAX_EDGE_FEA) { nb_set_error("unsupported in_edge_nf=%d", c->in_edge_nf); return NB_ERR_INVALID; }
  if (c->in_node_nf < 1 || c->in_node_nf > 64) { nb_set_error("unsupported in_node_nf=%d", c->in_node_nf); return NB_ERR_INVALID; }
  if ((int64_t)c->B * c->N * (c->N - 1) > 2000000000LL) { nb_set_error("too many edges for 32-bit indexing"); return NB_ERR_INVALID; }
  return NB_OK;
}

static void segno_layout(const NbSegnoConfig* c, SegnoLayout* lo) {
  const int H = NB_H;
  lo->E = 2 * H + 1 + c->in_edge_nf;
  int64_t o = 0;
  lo->emb_w = o; o += (int64_t)H * c->in_node_nf;
  lo->emb_b = o; o += H;
  lo->e_w1 = o; o += (int64_t)H * lo->E;
  lo->e_b1 = o; o += H;
  lo->e_w2 = o; o += H * H;
  lo->e_b2 = o; o += H;
  lo->n_w1 = o; o += H * 2 * H;
  lo->n_b1 = o; o += H;
  lo->n_w2 = o; o += H * H;
  lo->n_b2 = o; o += H;
  lo->c_w1 = o; o += H * H;
  lo->c_b1 = o; o += H;
  lo->c_w2 = o; o += H;
  lo->c_b2 = o; o += 1;
  lo->cv_w1 = o; o += H * H;
  lo->cv_b1 = o; o += H;
  lo->cv_w2 = o; o += H;
  lo->cv_b2 = o; o += 1;
  lo->total = o;
}

#define SEGNO_PARTIAL_FLOATS ((int64_t)32 * 1024 * 1024)
#define SEGNO_WIMG 5  /* edge layer 1 (h_row | h_col), node_mlp layer 1 (h | M), layer 2 */
struct SegnoIterBufs {
  float *h, *M, *U5, *x;
};
static inline int64_t segno_iter_floats(int64_t Nn) { return align64(Nn * (3 * NB_H + 3)); }
static SegnoIterBufs segno_iter_bufs(float* base, int64_t Nn) {
  SegnoIterBufs b;
  b.h = base; b.M = b.h + Nn * NB_H; b.U5 = b.M + Nn * NB_H; b.x = b.U5 + Nn * NB_H;
  return b;
}

extern "C" int64_t nb_segno_param_count(const NbSegnoConfig* cfg) {
  if (segno_validate(cfg) != NB_OK) return -1;
  SegnoLayout lo;
  segno_layout(cfg, &lo);
  return lo.total;
}
extern "C" int64_t nb_segno_saved_floats(const NbSegnoConfig* cfg) {
  if (segno_validate(cfg) != NB_OK) return -1;
  return segno_iter_floats((int64_t)cfg->B * cfg->N) * cfg->T;
}
struct SegnoCtx {
  const NbSegnoConfig* c;
  SegnoLayout lo;
  int64_t Nn;
  float inv_T, cw;   // the integrator's step 1 / T and coords_weight
  const float* params;
  void* st;
};

static int segno_ctx_init(SegnoCtx* X, const NbSegnoConfig* cfg, const float* params, void* st) {
  NB_TRY(segno_validate(cfg));
  X->c = cfg; segno_layout(cfg, &X->lo); X->Nn = (int64_t)cfg->B * cfg->N; X->params = params; X->st = st;
  X->inv_T = (float)(1.0 / (double)cfg->T); X->cw = cfg->coords_weight;
  return NB_OK;
}
// the buffers sub-step k saved in the forward
static SegnoIterBufs segno_saved(const SegnoCtx& X, const float* saved, int k) {
  return segno_iter_bufs(const_cast<float*>(saved) + (int64_t)k * segno_iter_floats(X.Nn), X.Nn);
}

// SEGNO forward; inference (nothing saved) adds two ping-pong sub-step sets
struct SegnoFwdWs {
  float *wimg, *P, *Q, *Fsum, *v[2], *infer;
  int64_t total;
};
static SegnoFwdWs segno_fwd_ws(const NbSegnoConfig* c, bool infer, float* base) {
  const int64_t Nn = (int64_t)c->B * c->N, nh = align64(Nn * NB_H), n3 = align64(Nn * 3);
  Carve w = {base, 0};
  SegnoFwdWs s;
  s.wimg = w.take(wimg_floats(SEGNO_WIMG));
  s.P = w.take(nh); s.Q = w.take(nh); s.Fsum = w.take(n3); s.v[0] = w.take(n3); s.v[1] = w.take(n3);
  s.infer = infer ? w.take(2 * segno_iter_floats(Nn)) : nullptr;
  s.total = w.used;
  return s;
}

// SEGNO backward: P, Q, gh, GU5, gP, gQ are kept PER sub-step (nh floats apart), so that the weight-gradient
// reductions of all sub-steps run as a few large batches instead of one small batch (+ finalize) per sub-step.  gh has
// T + 1 slots: the gradient entering sub-step k sits at slot k + 1, slot k receives its output
struct SegnoBwdWs {
  float *wimg, *P, *Q, *gM, *gh, *GU5, *gP, *gQ, *gx, *gv[2], *gFsum, *partial;
  int64_t nh, total;
};
static SegnoBwdWs segno_bwd_ws(const NbSegnoConfig* c, float* base) {
  const int64_t Nn = (int64_t)c->B * c->N, T = c->T, nh = align64(Nn * NB_H), n3 = align64(Nn * 3);
  Carve w = {base, 0};
  SegnoBwdWs s;
  s.nh = nh;
  s.wimg = w.take(wimg_floats(SEGNO_WIMG));
  s.P = w.take(T * nh); s.Q = w.take(T * nh); s.gM = w.take(nh); s.gh = w.take((T + 1) * nh);
  s.GU5 = w.take(T * nh); s.gP = w.take(T * nh); s.gQ = w.take(T * nh);
  s.gx = w.take(n3); s.gv[0] = w.take(n3); s.gv[1] = w.take(n3); s.gFsum = w.take(n3);
  s.partial = w.take(SEGNO_PARTIAL_FLOATS);
  s.total = w.used;
  return s;
}

// input-gradient workspace of nb_segno_backward_ex: the per-row edge-attribute gradients of every sub-step launch (a
// slice of B*N(N-1) * in_edge_nf floats each), summed in a fixed order at the end
struct SegnoInputGradWs { float* gef_rows; int64_t ef_slice, total; };
static SegnoInputGradWs segno_input_grad_ws(const NbSegnoConfig* c, float* base) {
  Carve w = {base, 0};
  SegnoInputGradWs s;
  s.ef_slice = (int64_t)c->B * c->N * (c->N - 1) * c->in_edge_nf;
  s.gef_rows = w.take(align64(c->T * s.ef_slice));
  s.total = w.used;
  return s;
}

extern "C" int64_t nb_segno_workspace_floats(const NbSegnoConfig* cfg, int mode) {
  if (segno_validate(cfg) != NB_OK) return -1;
  if (mode < 0 || mode > 2) { nb_set_error("workspace mode must be 0 (inference), 1 (backward) or 2 (training forward)"); return -1; }
  if (mode == NB_WS_BACKWARD) return segno_bwd_ws(cfg, nullptr).total;
  return segno_fwd_ws(cfg, mode == NB_WS_FORWARD_INFER, nullptr).total;
}

extern "C" int64_t nb_segno_input_grad_workspace_floats(const NbSegnoConfig* cfg) {
  if (segno_validate(cfg) != NB_OK) return -1;
  return segno_input_grad_ws(cfg, nullptr).total;
}

static int segno_weight_images(const SegnoCtx& X, float* scratch) {
  const float* W[SEGNO_WIMG] = {X.params + X.lo.e_w1, X.params + X.lo.e_w1 + NB_H, X.params + X.lo.n_w1, X.params + X.lo.n_w1 + NB_H,
                                X.params + X.lo.n_w2};
  const int ld[SEGNO_WIMG] = {X.lo.E, X.lo.E, 2 * NB_H, 2 * NB_H, NB_H};
  return wimg_prepare(W, ld, SEGNO_WIMG, scratch, X.st);
}

// nblocks > 1: h is the first of `nblocks` row blocks of Nn rows, `hstride` floats apart (the saved hidden states of all
// sub-steps); P, Q are then [nblocks * Nn][64]
static int segno_pq(const SegnoCtx& X, const float* h, float* P, float* Q, int nblocks = 1, int64_t hstride = 0) {
  NbGemmArgs a = gemm_args((int)(X.Nn * nblocks));  // cols: h_row | h_col | radial | edge_attr  (gcl.py:78)
  a.nsrc = 1; a.src[0] = gsrc(h, NB_H, 0, X.params + X.lo.e_w1, 1, X.lo.E);
  a.bias = X.params + X.lo.e_b1; a.out = P;
  NbGemmArgs b = gemm_args((int)(X.Nn * nblocks));
  b.nsrc = 1; b.src[0] = gsrc(h, NB_H, 0, X.params + X.lo.e_w1 + NB_H, 1, X.lo.E);
  b.out = Q;
  if (nblocks > 1) {
    a.src[0].seg_rows = b.src[0].seg_rows = (int)X.Nn;
    a.src[0].seg_a = b.src[0].seg_a = hstride;
  }
  NbGemmArgs ab[2] = {a, b};
  return launch_gemm_batch(ab, 2, X.st);
}

static NbEdgeW segno_edge_w(const SegnoCtx& X) {
  NbEdgeW w;
  w.W1 = X.params + X.lo.e_w1; w.ldw1 = X.lo.E; w.col_rad = 2 * NB_H; w.col_ef = 2 * NB_H + 1;
  w.W2 = X.params + X.lo.e_w2; w.b2 = X.params + X.lo.e_b2; w.W3 = X.params + X.lo.c_w1; w.b3 = X.params + X.lo.c_b1;
  w.w4 = X.params + X.lo.c_w2; w.b4 = X.params + X.lo.c_b2;
  return w;
}

static void segno_embed_args(const SegnoCtx& X, const float* his, NbEmbedArgs* e) {
  memset(e, 0, sizeof(*e));
  e->T = 1; e->Nn0 = (int)X.Nn; e->B = X.c->B; e->F0 = X.c->in_node_nf; e->D = 0;
  e->nodes = his; e->tsteps = nullptr; e->W = X.params + X.lo.emb_w; e->bias = X.params + X.lo.emb_b;
}

// ---- SEGNO stages (see the EGNO stages)

// h = his W_emb^T + b_emb (model.py:73)
static int segno_embed_fwd(const SegnoCtx& X, const float* his, float* h) {
  NbEmbedArgs e;
  segno_embed_args(X, his, &e);
  e.out = h;
  const size_t smem = ((size_t)e.F0 * NB_H + 4 * e.F0) * sizeof(float);
  NB_LAUNCH_COUNTED(k_embed_fwd, (unsigned)imin(cdiv(X.Nn, 4), 8 * nb_num_sms()), 256, smem, X.st, e);
  return nb_check_launch("k_embed_fwd");
}

static int embed_bwd_grid(int64_t rows) { return imin(cdiv(rows, 32), 2 * nb_num_sms()); }
// grad[embedding.weight | embedding.bias] = dL/dW, dL/db of h = his W^T + b over eb.e.Nn0 rows (overwritten)
static int segno_embed_bwd(NbEmbedBwdArgs& eb, const SegnoLayout& lo, float* grad, void* st) {
  const int F = eb.e.F0, grid = embed_bwd_grid(eb.e.Nn0), plen = NB_H * F + NB_H;
  NB_TRY(q_partial(&eb.partial, (int64_t)grid * plen, st));
  const size_t smem = (32 * (size_t)F + 32 * NB_H) * sizeof(float);
  NB_LAUNCH_COUNTED(k_embed_bwd, (unsigned)grid, 256, smem, st, eb);
  NB_TRY(nb_check_launch("k_embed_bwd"));
  NB_TRY(q_finalize(eb.partial, grid, plen, grad, 0,
                    {fseg(0, NB_H * F, NB_H * F, lo.emb_w, 0, 1), fseg(NB_H * F, NB_H, NB_H, lo.emb_b, 0, 1)}, st));
  return q_flush(st);
}

// the whole forward as one kernel, node state in shared memory (nb_segno_fused.cuh), for the tcgen05 variants and
// whole-graph selector units (N <= 27); otherwise *done = false and the call runs one sub-step at a time
static int segno_fused_fwd(const SegnoCtx& X, const SegnoFwdWs& ws, const float* his, const float* x, const float* v,
                           const float* edge_attr, float* x_out, float* h_out, float* v_out, float* saved, bool* done) {
  *done = false;
#ifndef NB_EMU
  const NbSegnoConfig* cfg = X.c;
  NbEdgeGeom fg = edge_geom(cfg->B, cfg->B, cfg->N, cfg->in_edge_nf, 1);
  if (!(g_segno_fused && g_edge_impl == 2 && g_node_impl == 1 && sel_geom(fg) && !fg.blk)) return NB_OK;
  *done = true;
  // embedding into scratch (the fused kernel writes h_k of every sub-step into `saved` itself)
  if (!cfg->h_given) NB_TRY(segno_embed_fwd(X, his, ws.P));
  const float* params = X.params;
  NbSegnoFusedArgs fa;
  memset(&fa, 0, sizeof(fa));
  fa.g = fg; fa.T = cfg->T; fa.recurrent = cfg->recurrent; fa.inv_T = X.inv_T; fa.cw = X.cw;
  fa.W1 = params + X.lo.e_w1; fa.b1 = params + X.lo.e_b1; fa.ldw1 = X.lo.E; fa.col_rad = 2 * NB_H; fa.col_ef = 2 * NB_H + 1;
  fa.W2 = params + X.lo.e_w2; fa.b2 = params + X.lo.e_b2; fa.W3 = params + X.lo.c_w1; fa.b3 = params + X.lo.c_b1;
  fa.w4 = params + X.lo.c_w2; fa.b4 = params + X.lo.c_b2;
  fa.W5 = params + X.lo.n_w1; fa.b5 = params + X.lo.n_b1; fa.W6 = params + X.lo.n_w2; fa.b6 = params + X.lo.n_b2;
  fa.h_in = cfg->h_given ? his : ws.P; fa.x_in = x; fa.v_in = v; fa.ef = edge_attr;
  fa.h_out = h_out; fa.x_out = x_out; fa.v_out = v_out; fa.saved = saved; fa.iter_stride = segno_iter_floats(X.Nn);
  const size_t fsm = NB_SEGNO_FUSED_SMEM(fg.G * fg.EPG);
  NB_SET_SMEM(k_segno_fused_fwd, fsm);
  int pi = prof_begin(5, X.st);
  NB_LAUNCH_COUNTED(k_segno_fused_fwd, (unsigned)imin(fg.n_units, nb_num_sms()), NB_SB_THREADS, fsm, X.st, fa);
  prof_end(5, pi, X.st);
  return nb_check_launch("k_segno_fused_fwd");
#else
  return NB_OK;
#endif
}

// one sub-step (gcl.py:76-94, model.py:95-102): edge layer, integrator, node_mlp
static int segno_step_fwd(const SegnoCtx& X, const SegnoFwdWs& ws, const SegnoIterBufs& b, const float* v,
                          const float* edge_attr, float* h_next, float* x_next, float* v_next) {
  const NbSegnoConfig* cfg = X.c;
  const float* params = X.params;
  NB_TRY(segno_pq(X, b.h, ws.P, ws.Q));
  NbEdgeFwdArgs ea;
  ea.g = edge_geom(cfg->B, cfg->B, cfg->N, cfg->in_edge_nf, 1);
  ea.w = segno_edge_w(X);
  ea.x = b.x; ea.P = ws.P; ea.Q = ws.Q; ea.ef = edge_attr; ea.M = b.M; ea.Fsum = ws.Fsum;
  NB_TRY(launch_edge_fwd(ea, X.st));
  NbIntegArgs ia;
  memset(&ia, 0, sizeof(ia));
  ia.n3 = X.Nn * 3; ia.N = cfg->N; ia.inv_T = X.inv_T; ia.cw = X.cw;
  ia.x = b.x; ia.v = v; ia.Fsum = ws.Fsum; ia.x_out = x_next; ia.v_out = v_next;
  NB_LAUNCH_COUNTED(k_segno_integ_fwd, (unsigned)ew_grid(X.Nn * 3), 256, 0, X.st, ia);
  NB_TRY(nb_check_launch("k_segno_integ_fwd"));
  NbGemmArgs a = gemm_args((int)X.Nn);  // U5 = [h, M] W5^T + b5      (gcl.py:89-92)
  a.nsrc = 2;
  a.src[0] = gsrc(b.h, NB_H, 0, params + X.lo.n_w1, 1, 2 * NB_H);
  a.src[1] = gsrc(b.M, NB_H, 0, params + X.lo.n_w1 + NB_H, 1, 2 * NB_H);
  a.bias = params + X.lo.n_b1; a.out_pre = b.U5;
  NB_TRY(launch_gemm(a, X.st));
  NbGemmArgs c2 = gemm_args((int)X.Nn);  // h' = h + SiLU(U5) W6^T + b6   (recurrent, gcl.py:93-94)
  c2.nsrc = 1; c2.src[0] = gsrc(b.U5, NB_H, 1, params + X.lo.n_w2, 1, NB_H);
  c2.bias = params + X.lo.n_b2; c2.out = h_next;
  if (cfg->recurrent) c2.R = b.h;
  return launch_gemm(c2, X.st);
}

extern "C" int nb_segno_forward(const NbSegnoConfig* cfg, const float* params, const float* his, const float* x,
                                const float* v, const float* edge_attr, float* x_out, float* h_out, float* v_out,
                                float* saved, float* workspace, void* stream) {
  NB_RANGE("nb_segno_forward");
  SegnoCtx X;
  NB_TRY(segno_ctx_init(&X, cfg, params, stream));
  const int64_t Nn = X.Nn, itf = segno_iter_floats(Nn);
  const int T = cfg->T;
  const SegnoFwdWs ws = segno_fwd_ws(cfg, !saved, workspace);
  WimgGuard wimg_guard;
  bool fused = false;
  NB_TRY(segno_fused_fwd(X, ws, his, x, v, edge_attr, x_out, h_out, v_out, saved, &fused));
  if (fused) return NB_OK;
  NB_TRY(segno_weight_images(X, ws.wimg));
  // training keeps every sub-step's buffers in `saved`; inference alternates two sets in the workspace
  auto bufs = [&](int k) { return segno_iter_bufs(saved ? saved + (int64_t)k * itf : ws.infer + (int64_t)(k & 1) * itf, Nn); };
  cudaStream_t cst = (cudaStream_t)stream;
  const SegnoIterBufs b0 = bufs(0);
  if (cfg->h_given) cudaMemcpyAsync(b0.h, his, Nn * NB_H * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  else NB_TRY(segno_embed_fwd(X, his, b0.h));
  cudaMemcpyAsync(b0.x, x, Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  const float* vcur = v;
  for (int k = 0; k < T; ++k) {
    const bool last = k + 1 == T;
    float* v_next = last ? v_out : ws.v[k & 1];
    NB_TRY(segno_step_fwd(X, ws, bufs(k), vcur, edge_attr, last ? h_out : bufs(k + 1).h, last ? x_out : bufs(k + 1).x, v_next));
    vcur = v_next;
  }
  return nb_check_launch("nb_segno_forward");
}

// The node-level chain between the edge sweeps of two sub-steps is ONE launch (k_segno_node_bwd) when the tcgen05 node
// kernels and their weight images are in use; nb_set_segno_fused(0) runs it stepwise
static bool segno_chain() {
#ifndef NB_EMU
  return g_segno_fused && g_node_impl == 1 && g_wimg.n == SEGNO_WIMG;
#else
  return false;
#endif
}
// the chain launch: node_mlp and integrator backward of sub-step j after edge layer 1's h halves backwards of j + 1, or
// (FIRST, j = T - 1) from the incoming g_h_out (null: zero)
template <bool FIRST>
static int segno_node_bwd(const SegnoCtx& X, const SegnoBwdWs& ws, const float* saved, int j, const float* g_h_out,
                          const float* gv_in, float* gv_out) {
#ifndef NB_EMU
  const int64_t nh = ws.nh;
  NbSegnoNodeBwdArgs na;
  memset(&na, 0, sizeof(na));
  na.rows = (int)X.Nn; na.recurrent = X.c->recurrent; na.img = g_wimg.img[0];
  if (FIRST) {
    na.gh_in = g_h_out;
  } else {
    na.gP = ws.gP + (int64_t)(j + 1) * nh; na.gQ = ws.gQ + (int64_t)(j + 1) * nh; na.gh_k = ws.gh + (int64_t)(j + 1) * nh;
  }
  na.U5 = segno_saved(X, saved, j).U5;
  na.GU5 = ws.GU5 + (int64_t)j * nh; na.gh_km1 = ws.gh + (int64_t)j * nh; na.gM = ws.gM;
  na.n3 = X.Nn * 3; na.N = X.c->N; na.inv_T = X.inv_T; na.cw = X.cw;
  na.gx = ws.gx; na.gv = gv_in; na.gv_out = gv_out; na.gFsum = ws.gFsum;
  NB_SET_SMEM(k_segno_node_bwd<FIRST>, NB_SNB_SMEM);
  int pi = prof_begin(2, X.st);
  NB_LAUNCH_COUNTED(k_segno_node_bwd<FIRST>, (unsigned)imin(cdiv(X.Nn, NB_TILE), nb_num_sms()), NB_THREADS, NB_SNB_SMEM, X.st, na);
  prof_end(2, pi, X.st);
  return nb_check_launch("k_segno_node_bwd");
#else
  nb_set_error("the host emulator runs SEGNO one sub-step at a time");
  return NB_ERR_INVALID;
#endif
}
// the stepwise node_mlp and integrator backward of sub-step k (gh_in: dL/dh entering it)
static int segno_step_bwd(const SegnoCtx& X, const SegnoBwdWs& ws, const float* saved, int k, const float* gh_in,
                          const float* gv_in, float* gv_out) {
  const SegnoLayout& lo = X.lo;
  const float* params = X.params;
  float* GU5 = ws.GU5 + (int64_t)k * ws.nh;
  NbGemmArgs a = gemm_args((int)X.Nn);  // GU5 = (gh W6) * SiLU'(U5)
  a.nsrc = 1; a.src[0] = gsrc(gh_in, NB_H, 0, params + lo.n_w2, NB_H, 1);
  a.epi = NB_EPI_MUL_DSILU; a.U = segno_saved(X, saved, k).U5; a.out = GU5;
  NB_TRY(launch_gemm(a, X.st));
  NbGemmArgs g1 = gemm_args((int)X.Nn);  // gh = GU5 W5[:, :64] (+ gh: residual)
  g1.nsrc = 1; g1.src[0] = gsrc(GU5, NB_H, 0, params + lo.n_w1, 2 * NB_H, 1);
  if (X.c->recurrent) g1.R = gh_in;
  g1.out = ws.gh + (int64_t)k * ws.nh;
  NbGemmArgs g2 = gemm_args((int)X.Nn);  // gM = GU5 W5[:, 64:]
  g2.nsrc = 1; g2.src[0] = gsrc(GU5, NB_H, 0, params + lo.n_w1 + NB_H, 2 * NB_H, 1);
  g2.out = ws.gM;
  NbGemmArgs g12[2] = {g1, g2};
  NB_TRY(launch_gemm_batch(g12, 2, X.st));
  NbIntegArgs ia;   // integrator backward
  memset(&ia, 0, sizeof(ia));
  ia.n3 = X.Nn * 3; ia.N = X.c->N; ia.inv_T = X.inv_T; ia.cw = X.cw;
  ia.gx = ws.gx; ia.gv = gv_in; ia.gx_out = ws.gx; ia.gv_out = gv_out; ia.gFsum = ws.gFsum;
  NB_LAUNCH_COUNTED(k_segno_integ_bwd, (unsigned)ew_grid(X.Nn * 3), 256, 0, X.st, ia);
  return nb_check_launch("k_segno_integ_bwd");
}
// weight gradients of the shared layers: ONE reduction per weight block over the rows of sub-steps [k0, k1) (the
// operands of sub-step k sit k blocks apart: saved state at stride itf, the sweep's gradients at stride nh); queued on
// `st`, every job accumulates onto grad
static int segno_queue_wgrads(const SegnoCtx& X, const SegnoBwdWs& ws, const float* saved, const float* g_h_out, int k0,
                              int k1, float* grad, void* st) {
  const SegnoLayout& lo = X.lo;
  const int64_t nh = ws.nh, itf = segno_iter_floats(X.Nn), Nn = X.Nn;
  const int T = X.c->T;
  const SegnoIterBufs b0 = segno_saved(X, saved, k0);
  const int rows = (int)(Nn * (k1 - k0)), sr = (int)Nn;
  const float* ghin0 = ws.gh + (int64_t)(k0 + 1) * nh;   // gh entering sub-step k = slot k + 1 ...
  // ... except for the last sub-step when the caller supplied dL/dh_out: that one lives in the caller's buffer
  if (g_h_out && k1 == T) {
    if (k1 - 1 > k0) {
      NB_TRY(wgrad_to((int)(Nn * (k1 - 1 - k0)), wpair_seg(ghin0, b0.U5, 1, sr, nh, itf), grad, lo.n_w2, NB_H, 1, lo.n_b2, 1, st));
      NB_TRY(q_flush_wgrad(st));   // same destination as the job below: separate reduction batches
      NB_TRY(q_flush_fin(st, false));
    }
    NB_TRY(wgrad_to((int)Nn, wpair(g_h_out, segno_saved(X, saved, T - 1).U5, 1), grad, lo.n_w2, NB_H, 1, lo.n_b2, 1, st));
  } else {
    NB_TRY(wgrad_to(rows, wpair_seg(ghin0, b0.U5, 1, sr, nh, itf), grad, lo.n_w2, NB_H, 1, lo.n_b2, 1, st));
  }
  NB_TRY(wgrad_to(rows, wpair_seg(ws.GU5 + (int64_t)k0 * nh, b0.h, 0, sr, nh, itf), grad, lo.n_w1, 2 * NB_H, 1, lo.n_b1, 1, st));
  NB_TRY(wgrad_to(rows, wpair_seg(ws.GU5 + (int64_t)k0 * nh, b0.M, 0, sr, nh, itf), grad, lo.n_w1 + NB_H, 2 * NB_H, 1, -1, 1, st));
  NB_TRY(wgrad_to(rows, wpair_seg(ws.gP + (int64_t)k0 * nh, b0.h, 0, sr, nh, itf), grad, lo.e_w1, lo.E, 1, lo.e_b1, 1, st));
  return wgrad_to(rows, wpair_seg(ws.gQ + (int64_t)k0 * nh, b0.h, 0, sr, nh, itf), grad, lo.e_w1 + NB_H, lo.E, 1, -1, 1, st);
}

extern "C" int nb_segno_backward(const NbSegnoConfig* cfg, const float* params, const float* his,
                                 const float* edge_attr, const float* saved, const float* g_x_out,
                                 const float* g_h_out, const float* g_v_out, float* grad_params, float* g_x_in,
                                 float* g_v_in, float* g_h_in, float* workspace, void* stream) {
  return nb_segno_backward_ex(cfg, params, his, edge_attr, saved, g_x_out, g_h_out, g_v_out, grad_params, g_x_in, g_v_in,
                              g_h_in, nullptr, nullptr, workspace, nullptr, stream);
}

extern "C" int nb_segno_backward_ex(const NbSegnoConfig* cfg, const float* params, const float* his,
                                    const float* edge_attr, const float* saved, const float* g_x_out,
                                    const float* g_h_out, const float* g_v_out, float* grad_params, float* g_x_in,
                                    float* g_v_in, float* g_h_in, float* g_his, float* g_edge_attr, float* workspace,
                                    float* input_grad_workspace, void* stream) {
  NB_RANGE("nb_segno_backward");
  SegnoCtx X;
  NB_TRY(segno_ctx_init(&X, cfg, params, stream));
  if (!saved) { nb_set_error("nb_segno_backward needs the saved buffer of a forward call"); return NB_ERR_INVALID; }
  if (g_his && cfg->h_given) {
    nb_set_error("g_his is the gradient of the raw node features: with h_given = 1 the hidden state's gradient is g_h_in");
    return NB_ERR_INVALID;
  }
  const bool want_ef = g_edge_attr && cfg->in_edge_nf > 0;
  if (want_ef && !input_grad_workspace) {
    nb_set_error("nb_segno_backward_ex needs the input-gradient workspace (nb_segno_input_grad_workspace_floats)");
    return NB_ERR_INVALID;
  }
  const SegnoLayout& lo = X.lo;
  const int64_t Nn = X.Nn;
  const int T = cfg->T;
  const SegnoBwdWs ws = segno_bwd_ws(cfg, workspace);
  const SegnoInputGradWs iws = segno_input_grad_ws(cfg, input_grad_workspace);
  const int64_t nh = ws.nh;
  WimgGuard wimg_guard;
  NB_TRY(segno_weight_images(X, ws.wimg));
  // the last quarter of the partial-sum scratch belongs to the deferred reductions (below); it is only ever touched on
  // the second stream, which is in order, so one arena serves every deferred flush
  const int64_t def_cap = SEGNO_PARTIAL_FLOATS / 4;
  float* def_arena = ws.partial + (SEGNO_PARTIAL_FLOATS - def_cap);
  q_begin(ws.partial, SEGNO_PARTIAL_FLOATS - def_cap);
  cudaStream_t cst = (cudaStream_t)stream;

  cudaMemsetAsync(grad_params, 0, lo.total * sizeof(float), cst);
  if (g_x_out) cudaMemcpyAsync(ws.gx, g_x_out, Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  else cudaMemsetAsync(ws.gx, 0, Nn * 3 * sizeof(float), cst);
  if (!g_h_out) cudaMemsetAsync(ws.gh + (int64_t)T * nh, 0, Nn * NB_H * sizeof(float), cst);
  // dL/dh and dL/dv entering sub-step k's node_mlp / integrator backward, and the dL/dv leaving it (a ping-pong pair)
  auto gh_in = [&](int k) { return k == T - 1 && g_h_out ? g_h_out : ws.gh + (int64_t)(k + 1) * nh; };
  auto gv_out = [&](int k) { return ws.gv[(T - 1 - k) & 1]; };
  auto gv_in = [&](int k) -> const float* { return k == T - 1 ? g_v_out : gv_out(k + 1); };

  // edge layer 1's per-node halves of EVERY sub-step: one GEMM launch over the saved hidden states before the sweep
  // instead of one small launch per sub-step
  if (nh == Nn * NB_H) {
    NB_TRY(segno_pq(X, segno_saved(X, saved, 0).h, ws.P, ws.Q, T, segno_iter_floats(Nn)));
  } else {   // row blocks of P / Q are padded: one launch per sub-step
    for (int k = 0; k < T; ++k) NB_TRY(segno_pq(X, segno_saved(X, saved, k).h, ws.P + (int64_t)k * nh, ws.Q + (int64_t)k * nh));
  }
  EdgeGradDst ed;
  ed.w1 = lo.e_w1; ed.W2 = lo.e_w2; ed.b2 = lo.e_b2; ed.W3 = lo.c_w1; ed.b3 = lo.c_b1; ed.w4 = lo.c_w2; ed.b4 = lo.c_b2;
  ed.ldw1 = lo.E; ed.col_rad = 2 * NB_H; ed.col_ef = 2 * NB_H + 1; ed.b_unused = 0;
  float* run_base = nullptr;   // the edge kernels' per-CTA partial slices of consecutive sub-steps are contiguous:
  int run_parts = 0;           // one reduction over all of them after the sweep
  // Deferred reductions.  A sweep leaves most of the GPU idle (the node chain runs 40 CTAs; the second half of every edge
  // launch 108 of 148), and the reductions above used to run after it, alone.  With the second stream (defer_available)
  // the sub-steps the sweep has finished are reduced every DEFER_CHUNK sub-steps underneath the rest of the sweep:
  // their operands are per-sub-step buffers nobody rewrites, the partial slices live in their own arena, every
  // reduction still has a fixed order.  The caller's stream joins before its own last reduction touches grad_params.
  const bool chain = segno_chain();
  const int DEFER_CHUNK = 3;
  const bool defer = chain && defer_available();
  int k_hi = T;             // sub-steps [0, k_hi) still have to be reduced
  bool deferred_any = false;
  // the sweep: the last sub-step's node-level backward, then per sub-step k the edge backward and the node-level chain
  // into sub-step k - 1 (one launch, or the stepwise GEMMs)
  if (chain) NB_TRY(segno_node_bwd<true>(X, ws, saved, T - 1, g_h_out, gv_in(T - 1), gv_out(T - 1)));
  else NB_TRY(segno_step_bwd(X, ws, saved, T - 1, gh_in(T - 1), gv_in(T - 1), gv_out(T - 1)));
  for (int k = T - 1; k >= 0; --k) {
    NbEdgeBwdArgs ea;
    memset(&ea, 0, sizeof(ea));
    ea.g = edge_geom(cfg->B, cfg->B, cfg->N, cfg->in_edge_nf, 1);
    ea.w = segno_edge_w(X);
    ea.x = segno_saved(X, saved, k).x; ea.P = ws.P + (int64_t)k * nh; ea.Q = ws.Q + (int64_t)k * nh; ea.ef = edge_attr;
    ea.gM = ws.gM; ea.gFsum = ws.gFsum; ea.gP = ws.gP + (int64_t)k * nh; ea.gQ = ws.gQ + (int64_t)k * nh; ea.gx = ws.gx;
    if (want_ef) ea.gef = iws.gef_rows + (int64_t)k * iws.ef_slice;
    NB_TRY(launch_edge_bwd(ea, grad_params, ed, 1, stream, &run_base, &run_parts));
    if (defer && k > 0 && k_hi - k >= DEFER_CHUNK) {   // sub-steps [k, k_hi): every operand is final once this launch is done
      void* s2 = side2_fork(stream);
      float* const sv_base = g_q.pbase;
      const int64_t sv_cap = g_q.pcap, sv_used = g_q.pused;
      g_q.pbase = def_arena; g_q.pcap = def_cap; g_q.pused = 0;
      int rc = edge_bwd_finalize(run_base, run_parts, cfg->in_edge_nf, grad_params, ed, 1, s2);
      run_parts = 0;   // the next launch starts a new run right behind this one
      if (rc == NB_OK) rc = segno_queue_wgrads(X, ws, saved, g_h_out, k, k_hi, grad_params, s2);
      if (rc == NB_OK) rc = q_flush(s2);
      g_q.pbase = sv_base; g_q.pcap = sv_cap; g_q.pused = sv_used;
      NB_TRY(rc);
      side2_done(0);
      k_hi = k;
      deferred_any = true;
    }
    if (chain && k > 0) {
      NB_TRY(segno_node_bwd<false>(X, ws, saved, k - 1, nullptr, gv_in(k - 1), gv_out(k - 1)));
    } else {
      NbGemmArgs pa = gemm_args((int)Nn);  // gh_k += gP W1[:, h_row] + gQ W1[:, h_col]
      pa.nsrc = 2;
      pa.src[0] = gsrc(ws.gP + (int64_t)k * nh, NB_H, 0, params + lo.e_w1, lo.E, 1);
      pa.src[1] = gsrc(ws.gQ + (int64_t)k * nh, NB_H, 0, params + lo.e_w1 + NB_H, lo.E, 1);
      pa.out = ws.gh + (int64_t)k * nh; pa.accumulate = 1;
      NB_TRY(launch_gemm(pa, stream));
      if (k > 0) NB_TRY(segno_step_bwd(X, ws, saved, k - 1, gh_in(k - 1), gv_in(k - 1), gv_out(k - 1)));
    }
  }
  // ---- what the deferred flushes have not taken: the remaining sub-steps' reductions on the caller's stream, after the
  // second stream's last finalisation (both accumulate onto grad_params)
  if (deferred_any) side2_wait(stream, 0);
  if (run_parts > 0) NB_TRY(edge_bwd_finalize(run_base, run_parts, cfg->in_edge_nf, grad_params, ed, 1, stream));
  NB_TRY(segno_queue_wgrads(X, ws, saved, g_h_out, 0, k_hi, grad_params, stream));
  NB_TRY(q_flush(stream));
  if (cfg->h_given) {
    if (g_h_in) cudaMemcpyAsync(g_h_in, ws.gh, Nn * NB_H * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  } else {
    NbEmbedBwdArgs eb;
    memset(&eb, 0, sizeof(eb));
    segno_embed_args(X, his, &eb.e);
    eb.g = ws.gh;   // dL/dh entering the first sub-step
    NB_TRY(segno_embed_bwd(eb, lo, grad_params, stream));
    if (g_his)   // dL/dhis = dL/dh_emb W_emb
      NB_LAUNCH_COUNTED(k_embed_input_grad, (unsigned)ew_grid(Nn * cfg->in_node_nf), 256, 0, stream, ws.gh, params + lo.emb_w,
                        cfg->in_node_nf, cfg->in_node_nf, Nn, g_his);
  }
  if (want_ef)     // fixed-order sum over the T sub-step slices
    NB_LAUNCH_COUNTED(k_sum_slices, (unsigned)ew_grid(iws.ef_slice), 256, 0, stream, (const float*)iws.gef_rows,
                      g_edge_attr, iws.ef_slice, T);
  if (g_x_in) cudaMemcpyAsync(g_x_in, ws.gx, Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  if (g_v_in) cudaMemcpyAsync(g_v_in, gv_out(0), Nn * 3 * sizeof(float), cudaMemcpyDeviceToDevice, cst);
  return nb_check_launch("nb_segno_backward");
}

// ============================================================================= multi-input SEGNO (model.py:65-90, 105-139)
// The integration segments are nb_segno_forward / nb_segno_backward with h_given = 1; these entry points cover what the
// reference does around them: the embedding of every observed frame, the 'sum' / attention merge of an integrated state
// with the next observed frame, and the sum of the per-segment gradients of the shared parameters.
extern "C" int nb_segno_embed_forward(const NbSegnoConfig* cfg, const float* params, int64_t rows, const float* his, float* h,
                                      void* stream) {
  NB_RANGE("nb_segno_embed_forward");
  SegnoCtx X;
  NB_TRY(segno_ctx_init(&X, cfg, params, stream));
  if (rows < 1 || rows > 2000000000LL || !params || !his || !h) { nb_set_error("nb_segno_embed_forward: bad rows / null pointer"); return NB_ERR_INVALID; }
  X.Nn = rows;
  return segno_embed_fwd(X, his, h);
}
extern "C" int64_t nb_segno_embed_backward_workspace_floats(const NbSegnoConfig* cfg, int64_t rows) {
  if (!cfg || rows < 1) return -1;
  return (int64_t)embed_bwd_grid(rows) * (NB_H * cfg->in_node_nf + NB_H) + 64;
}
// grad_params[embedding.weight | embedding.bias] = dL/dW, dL/db of h = his W^T + b over `rows` rows (overwritten)
extern "C" int nb_segno_embed_backward(const NbSegnoConfig* cfg, int64_t rows, const float* his, const float* g_h,
                                       float* grad_params, float* workspace, void* stream) {
  NB_RANGE("nb_segno_embed_backward");
  NB_TRY(segno_validate(cfg));
  if (rows < 1 || rows > 2000000000LL || !his || !g_h || !grad_params || !workspace) { nb_set_error("nb_segno_embed_backward: bad rows / null pointer"); return NB_ERR_INVALID; }
  SegnoLayout lo;
  segno_layout(cfg, &lo);
  NbEmbedBwdArgs eb;
  memset(&eb, 0, sizeof(eb));
  eb.e.T = 1; eb.e.Nn0 = (int)rows; eb.e.B = 1; eb.e.F0 = cfg->in_node_nf; eb.e.D = 0; eb.e.nodes = his;
  eb.g = g_h;
  q_begin(workspace, nb_segno_embed_backward_workspace_floats(cfg, rows));
  return segno_embed_bwd(eb, lo, grad_params, stream);
}

static int merge_check(int32_t mode, int64_t n, int32_t L, int32_t frame) {
  if (mode < NB_MERGE_COPY || mode > NB_MERGE_ATTN || n < 1 || n > 2000000000LL / 64 || L < 1 || frame < 0 || frame >= L) {
    nb_set_error("nb_segno_merge: unsupported arguments (mode=%d, n=%lld, L=%d, frame=%d)", mode, (long long)n, L, frame);
    return NB_ERR_INVALID;
  }
  return NB_OK;
}
// mode 0: (h, x, v)_out = observed frame `frame` of the [n][L][.] tensors; 1: observed + integrated ('sum', model.py:82-85);
// 2: attention-weighted sum of the pair (model.py:86-90, 105-139; attn_params = attn_mlp.0.weight[64][65] | .0.bias[64] |
// .2.weight[64] | .2.bias, alpha[n][2] keeps the weights for the backward)
extern "C" int nb_segno_merge_forward(int32_t mode, int64_t n, int32_t L, int32_t frame, const float* h_all, const float* x_all,
                                      const float* v_all, const float* h_int, const float* x_int, const float* v_int,
                                      const float* attn_params, float* h_out, float* x_out, float* v_out, float* alpha,
                                      void* stream) {
  NB_RANGE("nb_segno_merge_forward");
  NB_TRY(merge_check(mode, n, L, frame));
  if (!h_all || !x_all || !v_all || !h_out || !x_out || !v_out || (mode != NB_MERGE_COPY && (!h_int || !x_int || !v_int)) ||
      (mode == NB_MERGE_ATTN && (!attn_params || !alpha))) {
    nb_set_error("nb_segno_merge_forward: null pointer");
    return NB_ERR_INVALID;
  }
  NbMergeArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = mode; a.n = (int)n; a.L = L; a.frame = frame; a.h_all = h_all; a.x_all = x_all; a.v_all = v_all;
  a.h_int = h_int; a.x_int = x_int; a.v_int = v_int; a.ap = attn_params; a.h_out = h_out; a.x_out = x_out; a.v_out = v_out;
  a.alpha = alpha;
  NB_LAUNCH_COUNTED(k_segno_merge_fwd, (unsigned)imin(cdiv(n, 8), 8 * nb_num_sms()), 256, NB_MERGE_SMEM, stream, a);
  return nb_check_launch("k_segno_merge_fwd");
}
static int merge_bwd_grid(int64_t n) { return imin(cdiv(n, 8), 2 * nb_num_sms()); }
extern "C" int64_t nb_segno_merge_backward_workspace_floats(int64_t n) {
  return n < 1 ? -1 : (int64_t)merge_bwd_grid(n) * NB_AT_PLEN + 64;
}
// gradients of the merged state -> slice [:, frame, :] of g_*_all (observed frame) and g_*_int (integrated state);
// mode 2 also (accumulate ? adds : writes) the NB_AT_PLEN attention-parameter gradients into g_attn
extern "C" int nb_segno_merge_backward(int32_t mode, int64_t n, int32_t L, int32_t frame, const float* h_all, const float* x_all,
                                       const float* v_all, const float* h_int, const float* x_int, const float* v_int,
                                       const float* attn_params, const float* alpha, const float* g_h, const float* g_x,
                                       const float* g_v, float* g_h_all, float* g_x_all, float* g_v_all, float* g_h_int,
                                       float* g_x_int, float* g_v_int, float* g_attn, int32_t accumulate, float* workspace,
                                       void* stream) {
  NB_RANGE("nb_segno_merge_backward");
  NB_TRY(merge_check(mode, n, L, frame));
  if (!g_h_all || !g_x_all || !g_v_all || (mode != NB_MERGE_COPY && (!g_h_int || !g_x_int || !g_v_int)) ||
      (mode == NB_MERGE_ATTN && (!h_all || !x_all || !v_all || !h_int || !x_int || !v_int || !attn_params || !alpha || !g_attn || !workspace))) {
    nb_set_error("nb_segno_merge_backward: null pointer");
    return NB_ERR_INVALID;
  }
  NbMergeArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = mode; a.n = (int)n; a.L = L; a.frame = frame; a.h_all = h_all; a.x_all = x_all; a.v_all = v_all;
  a.h_int = h_int; a.x_int = x_int; a.v_int = v_int; a.ap = attn_params; a.alpha = const_cast<float*>(alpha);
  a.g_h = g_h; a.g_x = g_x; a.g_v = g_v; a.g_h_all = g_h_all; a.g_x_all = g_x_all; a.g_v_all = g_v_all;
  a.g_h_int = g_h_int; a.g_x_int = g_x_int; a.g_v_int = g_v_int;
  const int grid = mode == NB_MERGE_ATTN ? merge_bwd_grid(n) : imin(cdiv(n, 8), 8 * nb_num_sms());
  if (mode == NB_MERGE_ATTN) {
    q_begin(workspace, nb_segno_merge_backward_workspace_floats(n));
    NB_TRY(q_partial(&a.partial, (int64_t)grid * NB_AT_PLEN, stream));
  }
  NB_LAUNCH_COUNTED(k_segno_merge_bwd, (unsigned)grid, 256, NB_MERGE_SMEM, stream, a);
  NB_TRY(nb_check_launch("k_segno_merge_bwd"));
  if (mode != NB_MERGE_ATTN) return NB_OK;
  NB_TRY(q_finalize(a.partial, grid, NB_AT_PLEN, g_attn, accumulate ? 1 : 0, {fseg(0, NB_AT_PLEN, NB_AT_PLEN, 0, 0, 1)}, stream));
  return q_flush(stream);
}
// dst[0:n] += src[0:n]: the shared parameters' gradients of the integration segments
extern "C" int nb_accumulate(int64_t n, float* dst, const float* src, void* stream) {
  NB_RANGE("nb_accumulate");
  if (n < 0 || !dst || !src) { nb_set_error("nb_accumulate: null pointer or negative size"); return NB_ERR_INVALID; }
  if (n == 0) return NB_OK;
  NB_LAUNCH_COUNTED(k_accumulate, (unsigned)ew_grid(n), 256, 0, stream, dst, src, n);
  return nb_check_launch("k_accumulate");
}

// ============================================================================= exported building blocks
extern "C" int nb_check_canonical_edges(const int64_t* row, const int64_t* col, int64_t n_edges, int32_t B, int32_t N,
                                        int32_t* flag_dev, void* stream) {
  NB_RANGE("nb_check_canonical_edges");
  if (N < 2 || B < 1 || n_edges != (int64_t)B * N * (N - 1)) {
    nb_set_error("edge_index has %lld edges, expected B*N*(N-1) = %lld", (long long)n_edges, (long long)B * N * (N - 1));
    return NB_ERR_INVALID;
  }
  cudaMemsetAsync(flag_dev, 0, sizeof(int32_t), (cudaStream_t)stream);
  NB_LAUNCH_COUNTED(k_check_edges, (unsigned)ew_grid(n_edges), 256, 0, stream, row, col, n_edges, (int)B, (int)N, (int*)flag_dev);
  return nb_check_launch("k_check_edges");
}

extern "C" int nb_egcl_edge_forward(int32_t n_gt, int32_t B, int32_t N, int32_t n_edge_fea, int32_t clamp_per_edge,
                                    const float* x, const float* P, const float* Q, const float* edge_fea,
                                    const float* w1, int32_t ldw1, int32_t col_rad, int32_t col_ef, const float* W2,
                                    const float* b2, const float* W3, const float* b3, const float* w4, const float* b4,
                                    float* M, float* Fsum, void* stream) {
  NB_RANGE("nb_egcl_edge_forward");
  if (N < 2 || N > NB_MAX_NODES || n_edge_fea < 0 || n_edge_fea > NB_MAX_EDGE_FEA || n_gt < 1 || B < 1) {
    nb_set_error("nb_egcl_edge_forward: unsupported shape");
    return NB_ERR_INVALID;
  }
  NbEdgeFwdArgs a;
  a.g = edge_geom(n_gt, B, N, n_edge_fea, clamp_per_edge);
  a.w.W1 = w1; a.w.ldw1 = ldw1; a.w.col_rad = col_rad; a.w.col_ef = col_ef;
  a.w.W2 = W2; a.w.b2 = b2; a.w.W3 = W3; a.w.b3 = b3; a.w.w4 = w4; a.w.b4 = b4;
  a.x = x; a.P = P; a.Q = Q; a.ef = edge_fea; a.M = M; a.Fsum = Fsum;
  return launch_edge_fwd(a, stream);
}

extern "C" int64_t nb_egcl_edge_backward_workspace_floats(int32_t n_gt, int32_t N) {
  (void)n_gt; (void)N;
  return NB_PARTIAL_FLOATS;
}

extern "C" int nb_egcl_edge_backward(int32_t n_gt, int32_t B, int32_t N, int32_t n_edge_fea, int32_t clamp_per_edge,
                                     const float* x, const float* P, const float* Q, const float* edge_fea,
                                     const float* w1, int32_t ldw1, int32_t col_rad, int32_t col_ef, const float* W2,
                                     const float* b2, const float* W3, const float* b3, const float* w4, const float* b4,
                                     const float* gM, const float* gFsum, float* gP, float* gQ, float* gx,
                                     float* gw, float* workspace, void* stream) {
  NB_RANGE("nb_egcl_edge_backward");
  if (N < 2 || N > NB_MAX_NODES || n_edge_fea < 0 || n_edge_fea > NB_MAX_EDGE_FEA || n_gt < 1 || B < 1) {
    nb_set_error("nb_egcl_edge_backward: unsupported shape");
    return NB_ERR_INVALID;
  }
  NbEdgeBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.g = edge_geom(n_gt, B, N, n_edge_fea, clamp_per_edge);
  a.w.W1 = w1; a.w.ldw1 = ldw1; a.w.col_rad = col_rad; a.w.col_ef = col_ef;
  a.w.W2 = W2; a.w.b2 = b2; a.w.W3 = W3; a.w.b3 = b3; a.w.w4 = w4; a.w.b4 = b4;
  a.x = x; a.P = P; a.Q = Q; a.ef = edge_fea; a.gM = gM; a.gFsum = gFsum; a.gP = gP; a.gQ = gQ; a.gx = gx;
  // gw layout: [gW2 64x64 | gW3 64x64 | gb2 | gb3 | gw4 | gw_rad | gw_ef[n_edge_fea][64] | gb4]
  EdgeGradDst d;
  d.w1 = 2 * NB_H * NB_H + 3 * NB_H;  // gw_rad at w1 + col_rad (0), gw_ef at w1 + col_ef + f + c*ldw1
  d.W2 = 0; d.W3 = NB_H * NB_H; d.b2 = 2 * NB_H * NB_H; d.b3 = d.b2 + NB_H; d.w4 = d.b3 + NB_H;
  d.ldw1 = 1 + n_edge_fea; d.col_rad = 0; d.col_ef = 1; d.b_unused = 0;
  d.b4 = d.w1 + (int64_t)NB_H * d.ldw1;
  q_begin(workspace, NB_PARTIAL_FLOATS);
  NB_TRY(launch_edge_bwd(a, gw, d, 0, stream));
  return q_flush(stream);
}

// ============================================================================= caller-side device helpers
extern "C" int nb_nbody_features(int32_t B, int32_t N, int32_t with_charge, const float* loc, const float* vel,
                                 const float* charges, const float* edge_attr_o, float* nodes, float* loc_mean,
                                 float* edge_attr, void* stream) {
  NB_RANGE("nb_nbody_features");
  if (B < 1 || N < 2 || N > 1024 || !loc || !vel || !charges || !nodes || !edge_attr) {
    nb_set_error("nb_nbody_features: unsupported shape or null pointer (B=%d, N=%d)", B, N);
    return NB_ERR_INVALID;
  }
  NbFeatArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = N; a.with_charge = with_charge ? 1 : 0; a.loc = loc; a.vel = vel; a.charges = charges;
  a.edge_attr_o = edge_attr_o; a.nodes = nodes; a.loc_mean = loc_mean; a.edge_attr = edge_attr;
  NB_LAUNCH_COUNTED(k_nbody_features, (unsigned)imin(B, 8 * nb_num_sms()), 128, (size_t)N * 4 * sizeof(float), stream, a);
  return nb_check_launch("k_nbody_features");
}

extern "C" int nb_nbody_energy(int32_t kind, int32_t F, int32_t B, int32_t N, float G, const float* loc, const float* vel,
                               const float* charges, float* energy, void* stream) {
  NB_RANGE("nb_nbody_energy");
  if ((kind != 0 && kind != 1) || F < 1 || B < 1 || N < 1 || N > 1024 || !loc || !vel || !charges || !energy) {
    nb_set_error("nb_nbody_energy: unsupported arguments (kind=%d, F=%d, B=%d, N=%d)", kind, F, B, N);
    return NB_ERR_INVALID;
  }
  NbEnergyArgs a;
  memset(&a, 0, sizeof(a));
  a.F = F; a.B = B; a.N = N; a.kind = kind; a.G = G; a.loc = loc; a.vel = vel; a.charges = charges; a.out = energy;
  NB_LAUNCH_COUNTED(k_nbody_energy, (unsigned)imin((int64_t)F * B, 16 * nb_num_sms()), 128,
                    ((size_t)N * 4 + 128) * sizeof(float), stream, a);
  return nb_check_launch("k_nbody_energy");
}

#define NB_MSE_CHUNKS 64
extern "C" int64_t nb_traj_mse_workspace_floats(int32_t T) { return (int64_t)(T > 0 ? T : 0) * NB_MSE_CHUNKS; }
extern "C" int nb_traj_mse(int32_t T, int64_t rows, int32_t target_layout, int32_t only_first, const float* pred,
                           const float* target, float* losses, float* loss, float* grad, float* workspace, void* stream) {
  NB_RANGE("nb_traj_mse");
  if (T < 1 || T > NB_MAX_T || rows < 1 || (target_layout != 0 && target_layout != 1) || !pred || !target || !losses ||
      !loss || !workspace) {
    nb_set_error("nb_traj_mse: unsupported arguments (T=%d (<= %d), rows=%lld, layout=%d) or null pointer", T, NB_MAX_T,
                 (long long)rows, target_layout);
    return NB_ERR_INVALID;
  }
  NbMseArgs a;
  memset(&a, 0, sizeof(a));
  a.T = T; a.layout = target_layout; a.only_first = only_first ? 1 : 0; a.R = rows; a.pred = pred; a.target = target;
  a.grad = grad; a.partial = workspace; a.losses = losses; a.loss = loss;
  a.nchunk = (int)imin(cdiv(rows * 3, 256), NB_MSE_CHUNKS);
  NB_LAUNCH_COUNTED(k_traj_mse, dim3((unsigned)a.nchunk, (unsigned)T), 256, 0, stream, a);
  NB_LAUNCH_COUNTED(k_traj_mse_fin, 1, 32, 0, stream, a);
  return nb_check_launch("k_traj_mse");
}

// trajectory simulators (float64; see nb_sim.cuh)
extern "C" int nb_sim_charged(int32_t B, int32_t N, int32_t T, int32_t sample_freq, double dt, double strength, double max_force,
                              double box_size, const double* loc0, const double* vel0, const double* charges, double* loc,
                              double* vel, void* stream) {
  NB_RANGE("nb_sim_charged");
  if (B < 1 || N < 1 || N > NB_SIM_MAX_N || T < 2 || sample_freq < 1 || T % sample_freq || !loc0 || !vel0 || !charges ||
      (T / sample_freq > 1 && (!loc || !vel))) {
    nb_set_error("nb_sim_charged: unsupported arguments (B=%d, N=%d (<= %d), T=%d, sample_freq=%d) or null pointer", B, N,
                 NB_SIM_MAX_N, T, sample_freq);
    return NB_ERR_INVALID;
  }
  NbSimChargedArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = N; a.T = T; a.sample_freq = sample_freq; a.dt = dt; a.strength = strength; a.max_f = max_force;
  a.box = box_size; a.loc0 = loc0; a.vel0 = vel0; a.charges = charges; a.loc = loc; a.vel = vel;
  NB_LAUNCH_COUNTED(k_sim_charged, (unsigned)B, NB_SIM_MAX_N, 0, stream, a);
  return nb_check_launch("k_sim_charged");
}
extern "C" int nb_sim_gravity(int32_t B, int32_t N, int32_t T, int32_t sample_freq, double dt, double G, double softening,
                              const double* pos0, const double* vel0, const double* mass, double* pos, double* vel,
                              double* force, void* stream) {
  NB_RANGE("nb_sim_gravity");
  if (B < 1 || N < 1 || N > NB_SIM_MAX_N || T < 1 || sample_freq < 1 || T % sample_freq || !pos0 || !vel0 || !mass || !pos ||
      !vel || !force) {
    nb_set_error("nb_sim_gravity: unsupported arguments (B=%d, N=%d (<= %d), T=%d, sample_freq=%d) or null pointer", B, N,
                 NB_SIM_MAX_N, T, sample_freq);
    return NB_ERR_INVALID;
  }
  NbSimGravityArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = N; a.T = T; a.sample_freq = sample_freq; a.dt = dt; a.G = G; a.soft2 = softening * softening;
  a.pos0 = pos0; a.vel0 = vel0; a.mass = mass; a.pos = pos; a.vel = vel; a.force = force;
  NB_LAUNCH_COUNTED(k_sim_gravity, (unsigned)B, NB_SIM_MAX_N, 0, stream, a);
  return nb_check_launch("k_sim_gravity");
}

// fused Adam: `step` is a device float holding the number of steps taken so far (incremented here when tick != 0);
// [params, grads, exp_avg, exp_avg_sq] are flat fp32 buffers of n elements
static int adam_launch(int64_t n, float* params, const float* grads, const void* const* peer_grads, int npeer, float* exp_avg,
                       float* exp_avg_sq, float* step, int32_t tick, double lr, double beta1, double beta2, double eps,
                       double weight_decay, double grad_scale, void* stream) {
  if (n < 0 || !params || (!grads && npeer <= 0) || !exp_avg || !exp_avg_sq || !step) {
    nb_set_error("nb_adam_step: null pointer or negative size");
    return NB_ERR_INVALID;
  }
  if (npeer < 0 || npeer > NB_MAX_PEERS) { nb_set_error("nb_adam_step_peers: 1 <= npeer <= %d", NB_MAX_PEERS); return NB_ERR_INVALID; }
  if (tick) NB_LAUNCH_COUNTED(k_adam_tick, 1, 1, 0, stream, step);
  if (n > 0) {
    NbAdamArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n; a.p = params; a.g = grads; a.m = exp_avg; a.v = exp_avg_sq; a.step = step;
    a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay; a.grad_scale = (float)grad_scale;
    a.npeer = npeer;
    for (int r = 0; r < npeer; ++r) {
      if (!peer_grads || !peer_grads[r]) { nb_set_error("nb_adam_step_peers: null peer buffer %d", r); return NB_ERR_INVALID; }
      a.peer[r] = (const float*)peer_grads[r];
    }
    NB_LAUNCH_COUNTED(k_adam, (unsigned)imin(cdiv(n, 256), 4 * nb_num_sms()), 256, 0, stream, a);
  }
  return nb_check_launch("k_adam");
}
extern "C" int nb_adam_step(int64_t n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* step,
                            int32_t tick, double lr, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                            void* stream) {
  NB_RANGE("nb_adam_step");
  return adam_launch(n, params, grads, nullptr, 0, exp_avg, exp_avg_sq, step, tick, lr, beta1, beta2, eps, weight_decay, grad_scale, stream);
}
extern "C" int nb_adam_step_peers(int64_t n, float* params, const void* const* peer_grads, int32_t npeer, float* exp_avg,
                                  float* exp_avg_sq, float* step, int32_t tick, double lr, double beta1, double beta2, double eps,
                                  double weight_decay, double grad_scale, void* stream) {
  NB_RANGE("nb_adam_step_peers");
  if (npeer < 1) { nb_set_error("nb_adam_step_peers: npeer must be >= 1"); return NB_ERR_INVALID; }
  return adam_launch(n, params, nullptr, peer_grads, npeer, exp_avg, exp_avg_sq, step, tick, lr, beta1, beta2, eps, weight_decay, grad_scale, stream);
}

// tcgen05 self test (see nb_tc.cuh): validates descriptors / layouts of the three MMA forms on the device.
__global__ void k_silu_selftest(int64_t n, const float* x, float* a, float* b) {
  NB_PDL_ENTER();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    a[i] = nb_silu(x[i]);
    b[i] = nb_silu_fma(x[i]);
  }
}
extern "C" int nb_silu_selftest(int64_t n, const float* x, float* out_mufu, float* out_fma, void* stream) {
  if (n < 0 || !x || !out_mufu || !out_fma) { nb_set_error("nb_silu_selftest: null pointer or negative size"); return NB_ERR_INVALID; }
  if (n > 0) NB_LAUNCH_COUNTED(k_silu_selftest, (unsigned)imin(cdiv(n, 256), 4 * nb_num_sms()), 256, 0, stream, n, x, out_mufu, out_fma);
  return nb_check_launch("k_silu_selftest");
}

extern "C" int nb_tc_selftest(int32_t mode, const float* A, const float* W, float* out, void* stream) {
#ifdef NB_EMU
  (void)mode; (void)A; (void)W; (void)out; (void)stream;
  nb_set_error("tcgen05 is not available in the host emulator");
  return NB_ERR_INVALID;
#else
  if (mode < 0 || mode > 10) { nb_set_error("mode must be 0..10"); return NB_ERR_INVALID; }
  const size_t smem = 5 * NB_TC_TILE_BYTES(128) + 1024;
  NB_SET_SMEM(k_tc_selftest, smem);
  NB_LAUNCH_COUNTED(k_tc_selftest, 1, 128, smem, stream, (int)mode, A, W, out);
  return nb_check_launch("k_tc_selftest");
#endif
}
