// kernels.cu -- hand-written CUDA kernels (sm_100a) of the MPGP / SMALXE hot path.
//
// Kernel families (DESIGN.md gives the byte counts and the roofline of each):
//   K_A   fused SpMV            Ap = A p  with epilogue  p.Ap, g.p, B p, alpha_f = max feasible step
//   K_B   fused update          x -= a p, g -= a Ap, QPCGrads split, reduced gradient / expansion half step,
//                               |gP|^2 |gc|^2 |gf|^2 Ap.gf B u
//   K_A'  fused SpMV            g = A x - b with epilogue split, p = gf and the three norms (expansion, init)
//   K_C   direction update      p = gf - beta p  |  p = gc
//   ctrl  one-thread kernels    step selection and stopping tests on device scalars (mpgp_ctl.h)
// plus the un-fused vector / QPC kernels used by set-up, post-solve, the option variants that are not on
// the headline path, and the public QPC*/Vec*/Mat* entry points.
//
// All reductions are deterministic: fixed per-thread order, fixed shuffle tree, one record per CTA, and the
// last CTA to finish adds the CTA records in index order (threadfence reduction).  Grids are persistent and
// sized from the SM count once per matrix, so results are reproducible run to run.
//
// Reference semantics restated by the fused epilogues (file:line into permon/permon):
//   QPCGrads_Box        src/qpc/impls/box/qpcbox.c:41-55      QPCGradReduced_Box  :86-92
//   QPCFeas_Box         src/qpc/impls/box/qpcbox.c:125-137    QPCProject_Box      :298-303
//   MPGP step formulas  src/qps/impls/mpgp/mpgp.c:299-323 (expansion), :553-560 (CG), :623-638 (proportioning)
#include <climits>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "device.h"

namespace pb {

// =====================================================================================================
// context, errors, profiling
// =====================================================================================================
static DevCtx      g_ctx;
int                g_p2p_size = 1;   // ranks of the peer-memory window (set by the communicator)
static std::string g_err;
DevCtx            &ctx() { return g_ctx; }
const char        *last_error() { return g_err.c_str(); }

void set_error(const char *fmt, ...)
{
  char    buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  if (getenv("PERMON_B200_VERBOSE")) fprintf(stderr, "[permon_b200] %s\n", buf);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
  set_error("CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
  return 97; /* PETSC_ERR_GPU */
}

int dev_init()
{
  DevCtx &c = g_ctx;
  if (c.ready) return 0;
  int         count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    set_error("no usable CUDA device (%s): permon_b200 has no CPU execution path", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return 97;
  }
  if (c.device < 0) {
    const char *lr = getenv("LOCAL_RANK");
    c.device = lr ? atoi(lr) % count : 0;
  }
  PB_CUDA(cudaSetDevice(c.device));
  cudaDeviceProp prop;
  PB_CUDA(cudaGetDeviceProperties(&prop, c.device));
  c.sm_count = prop.multiProcessorCount;
  if (prop.major < 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", c.device, prop.major, prop.minor);
    return 97;
  }
  PB_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
  PB_CUDA(cudaStreamCreateWithFlags(&c.comm_stream, cudaStreamNonBlocking));
  PB_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
  if (!c.stream) c.stream = c.own_stream;
  c.ready = true;
  return 0;
}

// ---- memory -----------------------------------------------------------------------------------------------------------
static bool g_pool_ready = false;
static bool pool_enabled()
{
  static int on = -1;
  if (on < 0) {
    const char *e = getenv("PERMON_B200_POOL");
    on = (e && !strcmp(e, "0")) ? 0 : 1;
  }
  return on != 0;
}
int dmalloc_bytes(void **p, size_t bytes)
{
  PB_CHK(dev_init());
  if (bytes == 0) bytes = 16;
  if (pool_enabled()) {
    if (!g_pool_ready) {
      cudaMemPool_t pool;
      PB_CUDA(cudaDeviceGetDefaultMemPool(&pool, g_ctx.device));
      uint64_t keep = UINT64_MAX;
      PB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
      g_pool_ready = true;
    }
    PB_CUDA(cudaMallocAsync(p, bytes, g_ctx.stream));
    return 0;
  }
  PB_CUDA(cudaMalloc(p, bytes));
  return 0;
}
void dfree(const void *p)
{
  if (!p) return;
  if (pool_enabled()) cudaFreeAsync((void *)p, g_ctx.stream);
  else cudaFree((void *)p);
}
static std::vector<std::pair<size_t, void *>> g_pinned_cache;
void *pinned_get(size_t bytes)
{
  for (size_t i = 0; i < g_pinned_cache.size(); i++)
    if (g_pinned_cache[i].first == bytes) {
      void *p = g_pinned_cache[i].second;
      g_pinned_cache.erase(g_pinned_cache.begin() + i);
      return p;
    }
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p;
}
void pinned_put(void *p, size_t bytes)
{
  if (!p) return;
  if (bytes <= (1u << 20) && g_pinned_cache.size() < 64) g_pinned_cache.push_back({bytes, p});
  else cudaFreeHost(p);
}

static double phase_now()
{
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}
PhaseTimer::PhaseTimer(const char *nm) : name(nm), t0(0.0), on(false)
{
  nvtxRangePushA(nm);   // NVTX range of every phase (header-only NVTX3: a no-op unless a profiler injects itself)
  static const bool enabled = getenv("PERMON_B200_TIMING") != nullptr;
  on = enabled;
  if (on) {
    if (g_ctx.ready) cudaDeviceSynchronize();
    t0 = phase_now();
  }
}
PhaseTimer::~PhaseTimer()
{
  nvtxRangePop();
  if (!on) return;
  if (g_ctx.ready) cudaDeviceSynchronize();
  fprintf(stderr, "[permon_b200 timing] %-44s %9.2f ms\n", name, 1e3 * (phase_now() - t0));
}

static const char *g_family_names[KF_COUNT] = {"K_A spmv+dots+feas", "K_B update+split", "K_A' spmv+grad+split", "K_C direction", "ctrl", "spmv plain", "vec", "qpc", "halo"};
const char        *family_name(int f) { return (f >= 0 && f < KF_COUNT) ? g_family_names[f] : "?"; }

struct ProfRec {
  int         fam;
  double      bytes;
  cudaEvent_t a, b;
};
static bool                 g_prof_on = false;
static std::vector<ProfRec> g_prof;
static size_t               g_prof_used = 0;
static double               g_prof_ms[KF_COUNT], g_prof_bytes[KF_COUNT], g_prof_work_ms[KF_COUNT];
static int64_t              g_prof_n[KF_COUNT], g_prof_work_n[KF_COUNT];

void prof_begin()
{
  g_prof_on   = true;
  g_prof_used = 0;
}
void prof_pre(int family, double bytes)
{
  g_ctx.launches++;
  if (!g_prof_on) return;
  if (g_prof_used == g_prof.size()) {
    if (g_prof.size() >= 200000) return;
    ProfRec r;
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    g_prof.push_back(r);
  }
  ProfRec &r = g_prof[g_prof_used];
  r.fam   = family;
  r.bytes = bytes;
  cudaEventRecord(r.a, g_ctx.stream);
}
void prof_post(int family)
{
  (void)family;
  if (!g_prof_on) return;
  if (g_prof_used >= g_prof.size()) return;
  cudaEventRecord(g_prof[g_prof_used].b, g_ctx.stream);
  g_prof_used++;
}
int prof_end()
{
  g_prof_on = false;
  cudaStreamSynchronize(g_ctx.stream);
  for (int f = 0; f < KF_COUNT; f++) g_prof_ms[f] = g_prof_bytes[f] = g_prof_work_ms[f] = 0.0, g_prof_n[f] = g_prof_work_n[f] = 0;
  std::vector<float> ms(g_prof_used, 0.f);
  float              mx[KF_COUNT];
  for (int f = 0; f < KF_COUNT; f++) mx[f] = 0.f;
  for (size_t i = 0; i < g_prof_used; i++) {
    cudaEventElapsedTime(&ms[i], g_prof[i].a, g_prof[i].b);
    const int f = g_prof[i].fam;
    g_prof_ms[f] += ms[i];
    g_prof_bytes[f] += g_prof[i].bytes;
    g_prof_n[f]++;
    if (ms[i] > mx[f]) mx[f] = ms[i];
  }
  // "working" launches: a device-driven kernel that has nothing to do (K_A' outside expansion steps, anything enqueued behind the
  // stopping iteration) exits within a few microseconds.  Per family: when the 95th percentile of the durations is more than 8x the
  // shortest launch the family has early exits, and everything above the geometric mean of the two did the work; otherwise every launch
  // did.  A rare launch that takes several times the median of the working ones (host hiccup between the two events) is left out of
  // the working time but still counted in the total.
  for (int f = 0; f < KF_COUNT; f++) {
    std::vector<float> d;
    for (size_t i = 0; i < g_prof_used; i++)
      if (g_prof[i].fam == f) d.push_back(ms[i]);
    if (d.empty()) continue;
    std::sort(d.begin(), d.end());
    const float lo = d.front(), p95 = d[(size_t)(0.95 * (d.size() - 1))];
    const float thr = (p95 > 8.f * lo) ? sqrtf(fmaxf(lo, 1e-4f) * p95) : 0.f;
    std::vector<float> w;
    for (float v : d)
      if (v > thr) w.push_back(v);
    if (w.empty()) continue;
    const float med = w[w.size() / 2];
    for (float v : w) {
      if (v > 4.f * med) continue;
      g_prof_work_ms[f] += v;
      g_prof_work_n[f]++;
    }
  }
  return KF_COUNT;
}
int prof_dump(const char *path)
{   // per-launch timeline (ms since the first recorded launch) -- a poor man's nsys for gap analysis
  FILE *f = fopen(path, "w");
  if (!f) return 65;
  fprintf(f, "family,start_ms,stop_ms\n");
  for (size_t i = 0; i < g_prof_used; i++) {
    float a = 0.f, b = 0.f;
    cudaEventElapsedTime(&a, g_prof[0].a, g_prof[i].a);
    cudaEventElapsedTime(&b, g_prof[0].a, g_prof[i].b);
    fprintf(f, "%s,%.4f,%.4f\n", family_name(g_prof[i].fam), a, b);
  }
  fclose(f);
  return 0;
}
int prof_get_working(int f, int64_t *launches, double *ms)
{
  if (f < 0 || f >= KF_COUNT) return 63;
  *launches = g_prof_work_n[f];
  *ms       = g_prof_work_ms[f];
  return 0;
}
int prof_get(int f, int64_t *launches, double *ms, double *bytes_per_launch)
{
  if (f < 0 || f >= KF_COUNT) return 63;
  *launches         = g_prof_n[f];
  *ms               = g_prof_ms[f];
  *bytes_per_launch = g_prof_n[f] ? g_prof_bytes[f] / (double)g_prof_n[f] : 0.0;
  return 0;
}

#define LAUNCH_CHECK()                                                           \
  do {                                                                           \
    cudaError_t e_ = cudaGetLastError();                                         \
    if (e_ != cudaSuccess) return cuda_fail(e_, "kernel launch", __FILE__, __LINE__); \
  } while (0)

static bool aligned16(const void *p) { return (((uintptr_t)p) & 15) == 0; }

// Programmatic dependent launch: every kernel of the fused iteration starts with pdl_enter() -- wait until the previous kernel of
// the stream has completed and its writes are visible, then let the NEXT kernel's CTAs be scheduled as soon as SM resources free
// up (they block in their own pdl_enter()).  Launch latency and the ramp-up of kernel N+1 overlap the tail of kernel N.  Nothing
// that an earlier kernel produced may be read before pdl_enter().  Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_enter()
{
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// The producer warp of the TMA rings stages partial tiles / unaligned vectors with plain (generic-proxy) shared stores into slots that
// bulk copies (async proxy) write in other rounds: order the two proxies explicitly before the slot is handed over.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
static bool pdl_enabled()
{
  static int on = -1;
  if (on < 0) {
    const char *e = getenv("PERMON_B200_PDL");
    on = (e && !strcmp(e, "0")) ? 0 : 1;
  }
  return on != 0;
}
template <class... KArgs, class... Args>
static void launch_k(void (*kernel)(KArgs...), int grid, int block, size_t smem, Args &&...args)
{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim          = dim3((unsigned)grid);
  cfg.blockDim         = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream           = g_ctx.stream;
  cudaLaunchAttribute at[1];
  at[0].id                                         = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs    = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

static constexpr int NT = 256;   // threads per CTA everywhere

int elementwise_grid() { return g_ctx.sm_count * 8; }
int max_red_blocks() { return g_ctx.sm_count * 16; }

// =====================================================================================================
// deterministic grid reduction of an 8-double record (slots in MINMASK are min-reduced, others summed)
// =====================================================================================================
template <int MINMASK>
__device__ __forceinline__ double red_op(int k, double a, double b)
{
  if ((MINMASK >> k) & 1) return (b < a) ? b : a;
  return a + b;
}
template <int MINMASK>
__device__ __forceinline__ double red_identity(int k)
{
  return ((MINMASK >> k) & 1) ? HUGE_VAL : 0.0;
}

template <int MINMASK>
__device__ __forceinline__ void block_reduce8(double (&v)[PB_NRED], double (*sm)[32])
{
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < PB_NRED; k++) {
    double t = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = red_op<MINMASK>(k, t, __shfl_xor_sync(0xffffffffu, t, o));
    if (lane == 0) sm[k][warp] = t;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) {
      double t = (lane < nw) ? sm[k][lane] : red_identity<MINMASK>(k);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t = red_op<MINMASK>(k, t, __shfl_xor_sync(0xffffffffu, t, o));
      v[k] = t;   // valid in lane 0 of warp 0 (== thread 0)
    }
  }
  __syncthreads();
}

// every thread of every CTA of the grid must call this exactly once
template <int MINMASK>
__device__ void grid_reduce8(double (&v)[PB_NRED], RedBuf rb, const double *prev)
{
  __shared__ double sm[PB_NRED][32];
  __shared__ int    s_last;
  block_reduce8<MINMASK>(v, sm);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) rb.partials[(size_t)blockIdx.x * PB_NRED + k] = v[k];
    __threadfence();
    unsigned t = atomicAdd(rb.counter, 1u);
    s_last     = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    double w[PB_NRED];
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) {
      double t = red_identity<MINMASK>(k);
      for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) t = red_op<MINMASK>(k, t, __ldcg(&rb.partials[(size_t)b * PB_NRED + k]));
      if (rb.add_part && k == rb.add_slot)   // per-CTA partial sums left by an earlier kernel (K_C's g.p)
        for (int b = threadIdx.x; b < rb.add_n; b += blockDim.x) t += __ldcg(&rb.add_part[(size_t)b * PB_NRED]);
      w[k] = t;
    }
    block_reduce8<MINMASK>(w, sm);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < PB_NRED; k++) {
        const double f = prev ? red_op<MINMASK>(k, prev[k], w[k]) : w[k];
        rb.out[k] = f;
        sm[k][0]  = f;
      }
      *rb.counter = 0u;
    }
    if (rb.win) {   // peer-memory all-gather: push the record + sequence flag into every rank's window (NVLink stores)
      __syncthreads();
      const P2PWin *W = rb.win;
      if ((int)threadIdx.x < W->size) {
        const int        q = threadIdx.x;
        volatile double *dst = W->slot[q] + p2p_slot_index(rb.kind, rb.seq, W->rank);
#pragma unroll
        for (int k = 0; k < PB_NRED; k++) dst[k] = sm[k][0];
        __threadfence_system();
        *(volatile unsigned long long *)(W->flag[q] + p2p_flag_index(rb.kind, W->rank)) = rb.seq;
      }
    }
  }
}

// one value per CTA, no ticket: partials[blockIdx.x * PB_NRED] = sum over the CTA; a later kernel's final reduction adds them
__device__ void block_partial1(double v, double *partials)
{
  __shared__ double sm1[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) sm1[warp] = v;
  __syncthreads();
  if (warp == 0) {
    double t = (lane < nw) ? sm1[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) partials[(size_t)blockIdx.x * PB_NRED] = t;
  }
}

// spin until a flag in LOCAL memory (written by a peer over NVLink) reaches seq; a dead peer traps instead of hanging
__device__ __forceinline__ void wait_flag(const unsigned long long *f, unsigned long long seq)
{
  const volatile unsigned long long *vf = f;
  const long long                    t0 = clock64();
  while (*vf < seq) {
    if (clock64() - t0 > 20000000000LL) __trap();   // ~10 s
    __nanosleep(64);
  }
  __threadfence_system();
}

// =====================================================================================================
// box helpers (QPC box semantics)
// =====================================================================================================
struct BoxVal {
  double lb, ub;
  bool   has_lb, has_ub;
};
__device__ __forceinline__ BoxVal load_box(const BoxDev &bx, int r)
{
  BoxVal b;
  b.has_lb = bx.lb != nullptr;
  b.has_ub = bx.ub != nullptr;
  b.lb     = b.has_lb ? bx.lb[r] : 0.0;
  b.ub     = b.has_ub ? bx.ub[r] : 0.0;
  return b;
}
// QPCGrads (qpc.c:552-553 prefill + qpcbox.c:41-55)
__device__ __forceinline__ void box_split(double x, double g, const BoxVal &b, double astol, double &gf, double &gc)
{
  gf = g;
  gc = 0.0;
  if (b.has_lb && fabs(x - b.lb) <= astol) {
    gf = 0.0;
    gc = (g < 0.0) ? g : 0.0;
  } else if (b.has_ub && fabs(x - b.ub) <= astol) {
    gf = 0.0;
    gc = (g < 0.0) ? 0.0 : g;   // PetscMax(g,0)
  }
}
// QPCGradReduced (qpc.c:601 prefill + qpcbox.c:86-92)
// 1 when the split replaced g by +0.0 (bit comparison: a NaN gradient stays "not replaced", -0.0 counts as replaced)
__device__ __forceinline__ unsigned char gf_differs(double gf, double g) { return __double_as_longlong(gf) != __double_as_longlong(g); }

__device__ __forceinline__ double box_reduced(double x, double gf, const BoxVal &b, double alpha)
{
  double gr = gf;
  if (b.has_lb && gf > 0.0) {
    double t = (x - b.lb) / alpha;
    gr       = (gf < t) ? gf : t;
  } else if (b.has_ub && gf < 0.0) {
    double t = (x - b.ub) / alpha;
    gr       = (gf < t) ? t : gf;
  }
  return gr;
}
// QPCFeas_Box (qpcbox.c:125-137)
// Same minimum as box_feas, but the fp64 division (~25 instructions) only runs for candidates that can still lower the
// running minimum: (x - lb)/d >= cur is certain when x - lb > cur*d (+ rounding margin), and then `a < cur` is false.
__device__ __forceinline__ double box_feas_lazy(double x, double d, const BoxVal &b, double cur)
{
  const double PINF = 1.7976931348623157e+308 / 4.0;
  if (d > 0. && b.has_lb && b.lb > -PINF) {
    const double num = x - b.lb, thr = cur * d, mar = fabs(thr) * 4.5e-16;
    if (!(num > thr + mar) || !(fabs(thr) > 1e-290)) {
      double a = num / d;
      if (a < cur) cur = a;
    }
  }
  if (d < 0. && b.has_ub && b.ub < PINF) {
    const double num = x - b.ub, thr = cur * d, mar = fabs(thr) * 4.5e-16;
    if (!(num < thr - mar) || !(fabs(thr) > 1e-290)) {
      double a = num / d;
      if (a < cur) cur = a;
    }
  }
  return cur;
}

__device__ __forceinline__ double box_feas(double x, double d, const BoxVal &b, double cur)
{
  const double PINF = 1.7976931348623157e+308 / 4.0;
  if (d > 0. && b.has_lb && b.lb > -PINF) {
    double a = (x - b.lb) / d;
    if (a < cur) cur = a;
  }
  if (d < 0. && b.has_ub && b.ub < PINF) {
    double a = (x - b.ub) / d;
    if (a < cur) cur = a;
  }
  return cur;
}
// QPCProject_Box (qpcbox.c:298-303)
__device__ __forceinline__ double box_project(double x, const BoxVal &b)
{
  if (b.has_lb) {
    x = (x < b.lb) ? b.lb : x;
    if (b.has_ub) x = (x < b.ub) ? x : b.ub;
  } else if (b.has_ub) {
    x = (x < b.ub) ? x : b.ub;
  }
  return x;
}

// =====================================================================================================
// SpMV skeletons.  Epi supplies: active(), row(r, ax, acc), finalize(acc).
// =====================================================================================================

// tile-streamed CSR ("CSR-stream"): the CTA reads the nnz range of a 256-row tile with unit-stride loads,
// multiplies with the gathered x on the fly and parks the products in shared memory; then one thread per
// row adds its segment in storage order (== the reference's running sum) and runs the fused epilogue.
template <class Epi>
__global__ void __launch_bounds__(NT) k_spmv_stream(CsrDev A, const double *__restrict__ x, Epi epi)
{
  pdl_enter();
  if (!epi.active()) return;
  extern __shared__ double s_prod[];
  typename Epi::Acc acc;
  epi.init(acc);
  const int ntiles = (A.n + TR - 1) / TR;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * TR;
    const int r1 = min(r0 + TR, A.n);
    const int k0 = __ldg(A.ia + r0), k1 = __ldg(A.ia + r1);
    for (int k = k0 + threadIdx.x; k < k1; k += NT) s_prod[k - k0] = __ldg(A.a + k) * __ldg(x + __ldg(A.ja + k));
    __syncthreads();
    const int r = r0 + threadIdx.x;
    if (r < r1) {
      const int ks = __ldg(A.ia + r) - k0, ke = __ldg(A.ia + r + 1) - k0;
      double    s  = 0.0;
      for (int k = ks; k < ke; k++) s += s_prod[k];
      epi.row(A.rows ? __ldg(A.rows + r) : r, s, acc);
    }
    __syncthreads();
  }
  epi.finalize(acc);
}

// vector CSR: W lanes per row, unit-stride loads along the row, shuffle tree, lane 0 runs the epilogue
template <class Epi, int W>
__global__ void __launch_bounds__(NT) k_spmv_vector(CsrDev A, const double *__restrict__ x, Epi epi)
{
  pdl_enter();
  if (!epi.active()) return;
  typename Epi::Acc acc;
  epi.init(acc);
  const int lane    = threadIdx.x & (W - 1);
  const int gid     = (blockIdx.x * NT + threadIdx.x) / W;
  const int ngroups = gridDim.x * (NT / W);
  const int gpw     = 32 / W;                                    // groups per warp
  const int wfirst  = (gid / gpw) * gpw;                         // first group of my warp
  for (int base = wfirst; base < A.n; base += ngroups) {         // uniform trip count inside a warp
    const int r = base + (gid - wfirst);
    double    s = 0.0;
    if (r < A.n) {
      const int ks = __ldg(A.ia + r), ke = __ldg(A.ia + r + 1);
      int k = ks + lane;
      for (; k + 3 * W < ke; k += 4 * W) {   // four independent index -> gather chains in flight, products added in the same order
        const int    j0 = __ldg(A.ja + k), j1 = __ldg(A.ja + k + W), j2 = __ldg(A.ja + k + 2 * W), j3 = __ldg(A.ja + k + 3 * W);
        const double a0 = __ldg(A.a + k), a1 = __ldg(A.a + k + W), a2 = __ldg(A.a + k + 2 * W), a3 = __ldg(A.a + k + 3 * W);
        const double x0 = __ldg(x + j0), x1 = __ldg(x + j1), x2 = __ldg(x + j2), x3 = __ldg(x + j3);
        s += a0 * x0;
        s += a1 * x1;
        s += a2 * x2;
        s += a3 * x3;
      }
      for (; k < ke; k += W) s += __ldg(A.a + k) * __ldg(x + __ldg(A.ja + k));
    }
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0 && r < A.n) epi.row(A.rows ? __ldg(A.rows + r) : r, s, acc);
  }
  epi.finalize(acc);
}


// ---- Blackwell/Hopper async-copy primitives (PTX): mbarrier + 1-D bulk copy global -> shared (TMA engine) -------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
  uint32_t       ok = 0;
  const uint32_t addr = smem_u32(bar);
  for (unsigned spin = 0;; spin++) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    if (ok) break;
    if (spin > (1u << 24)) __trap();   // a lost transaction must abort the launch, never hang the GPU
  }
}

// TMA-staged CSR ("CSR-stream" with the DRAM streams on the copy engine): a producer warp feeds a ring of
// shared-memory stages with 1-D bulk copies (cp.async.bulk -> UBLKCP) of the tile's values, column indices, row
// pointers and the row slices of the epilogue vectors; 256 consumer threads (one per row) wait on the stage's
// mbarrier, gather x through L1/L2, add their segment in storage order and run the fused epilogue.  No LSU address
// generation for the streamed operands, loads of tile t+1.. overlap the compute of tile t.
struct TmaStage {   // byte offsets inside one stage
  int a_off, v_off, ja_off, ia_off, bytes;
};
__host__ __device__ inline TmaStage tma_stage_layout(int cap, int nv)
{
  TmaStage L;
  L.a_off  = 0;
  L.v_off  = cap * 8;
  L.ja_off = L.v_off + nv * TR * 8;
  L.ia_off = L.ja_off + cap * 4;
  L.bytes  = L.ia_off + (TR + 4) * 4;
  L.bytes  = (L.bytes + 127) & ~127;
  return L;
}
static constexpr int TMA_MAX_STAGES = 4;

template <class Epi>
__global__ void __launch_bounds__(NT + 32) k_spmv_tma(CsrDev A, const double *__restrict__ x, Epi epi, int cap, int nstages)
{
  pdl_enter();
  if (!epi.active()) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[TMA_MAX_STAGES], empty_bar[TMA_MAX_STAGES];
  __shared__ int      meta_k0a[TMA_MAX_STAGES];
  const int      nv = epi.nvec();
  const TmaStage L = tma_stage_layout(cap, nv);
  const int      ntiles = (A.n + TR - 1) / TR;
  const int      warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  typename Epi::Acc acc;
  epi.init(acc);
  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], NT / 32);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == NT / 32) {
    // ------------------------------ producer warp ------------------------------
    int k0n = 0, k1n = 0;
    if (blockIdx.x < ntiles) {
      const int r0 = blockIdx.x * TR, r1 = min(r0 + TR, A.n);
      k0n = __ldg(A.ia + r0);
      k1n = __ldg(A.ia + r1);
    }
    int      s = 0, filled = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int k0 = k0n, k1 = k1n;
      const int nt = tile + gridDim.x;
      if (nt < ntiles) {   // metadata of the next tile: in flight while this one is issued
        const int q0 = nt * TR, q1 = min(q0 + TR, A.n);
        k0n = __ldg(A.ia + q0);
        k1n = __ldg(A.ia + q1);
      }
      if (filled >= nstages) mbar_wait(&empty_bar[s], ph ^ 1u);
      else filled++;
      unsigned char *st = smem_raw + (size_t)s * L.bytes;
      const int      r0 = tile * TR, r1 = min(r0 + TR, A.n);
      const int      k0a = k0 & ~3;
      const int      na = (k1 - k0a + 3) & ~3;
      const bool     tma = (r1 - r0 == TR) && ((int64_t)k0a + na <= A.nnz_alloc) && (r0 + TR + 4 <= A.ia_alloc) && (na <= cap);
      if (tma) {
        if (lane == 0) {
          meta_k0a[s] = k0a;
          const uint32_t bytes = (uint32_t)na * 12u + (uint32_t)(TR + 4) * 4u + (uint32_t)nv * TR * 8u;
          mbar_arrive_expect_tx(&full_bar[s], bytes);
          if (na > 0) {
            bulk_g2s(st + L.a_off, A.a + k0a, (uint32_t)na * 8u, &full_bar[s]);
            bulk_g2s(st + L.ja_off, A.ja + k0a, (uint32_t)na * 4u, &full_bar[s]);
          }
          bulk_g2s(st + L.ia_off, A.ia + r0, (uint32_t)(TR + 4) * 4u, &full_bar[s]);
          for (int v = 0; v < nv; v++) bulk_g2s(st + L.v_off + (size_t)v * TR * 8, epi.vsrc(v) + r0, (uint32_t)TR * 8u, &full_bar[s]);
        }
      } else {
        // boundary tile (partial rows / end of the arrays): the warp loads it with plain loads
        double *a_s = (double *)(st + L.a_off);
        int    *ja_s = (int *)(st + L.ja_off), *ia_s = (int *)(st + L.ia_off);
        for (int k = k0 + lane; k < k1; k += 32) {
          a_s[k - k0a]  = __ldg(A.a + k);
          ja_s[k - k0a] = __ldg(A.ja + k);
        }
        for (int t = lane; t <= r1 - r0; t += 32) ia_s[t] = __ldg(A.ia + r0 + t);
        for (int v = 0; v < nv; v++) {
          double       *vs = (double *)(st + L.v_off) + (size_t)v * TR;
          const double *src = epi.vsrc(v) + r0;
          for (int t = lane; t < r1 - r0; t += 32) vs[t] = src[t];
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          meta_k0a[s] = k0a;
          mbar_arrive(&full_bar[s]);
        }
      }
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  } else {
    // ------------------------------ consumer warps: one thread per row ------------------------------
    const uint32_t smem_a = smem_u32(smem_raw);
    int            s = 0;
    uint32_t       ph = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      mbar_wait(&full_bar[s], ph);
      unsigned char *st = smem_raw + (size_t)s * L.bytes;
      const double  *a_s = (const double *)(st + L.a_off);
      const int     *ja_s = (const int *)(st + L.ja_off), *ia_s = (const int *)(st + L.ia_off);
      const uint32_t vs_a = smem_a + (uint32_t)s * (uint32_t)L.bytes + (uint32_t)L.v_off + 8u * threadIdx.x;
      const int      k0a = meta_k0a[s];
      const int      r = tile * TR + threadIdx.x;
      if (r < A.n) {
        const int ks = ia_s[threadIdx.x] - k0a, ke = ia_s[threadIdx.x + 1] - k0a;
        double    sum = 0.0;
        for (int k = ks; k < ke; k += 8) {   // 8 gathers in flight, products added in storage order
          double xv[8];
#pragma unroll
          for (int j = 0; j < 8; j++) xv[j] = (k + j < ke) ? __ldg(x + ja_s[k + j]) : 0.0;
#pragma unroll
          for (int j = 0; j < 8; j++)
            if (k + j < ke) sum += a_s[k + j] * xv[j];
        }
        epi.row_s(r, vs_a, sum, acc);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  }
  epi.finalize(acc);
}


// TMA-staged PACKED tiles (kind 3, format in pack.cpp): same producer/consumer ring as k_spmv_tma, but the matrix part of a
// tile is ONE bulk copy of its blob -- a per-tile dictionary of (col - row, value) pairs plus one byte per non-zero (or, for
// tiles with more than 256 distinct pairs, raw values + columns).  Consumers rebuild col = row + delta and add the products in
// storage order, so the result is bit-identical to the CSR kernels.  The matrix stream of a stencil Hessian shrinks from 12
// to ~1 byte per non-zero; what remains of K_A / K_A' is the traffic of the fused epilogue vectors.
static constexpr int PK_UNROLL = 8;
static constexpr int PK_CT = 128;   // consumer threads of the packed kernel: two rows of a 256-row tile each
// shared-memory loads by 32-bit address, in program order (volatile): the consumer code below issues every load of a row
// (code bytes -> dictionary deltas -> x gathers -> dictionary values) before the first multiply-add, so that a warp has
// 5-8 gathers in flight instead of one
__device__ __forceinline__ uint32_t lds_u8(uint32_t a)
{
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t a)
{
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ int lds_s32(uint32_t a)
{
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ double lds_f64(uint32_t a)
{
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a)
{
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}

// how the SpMV input is read: plain, or scaled on the fly (power method: the normalised iterate v = s * w is never stored)
struct GatherPlain {
  const double *x;
  __device__ __forceinline__ double ld(const double *p) const { return __ldg(p); }
  __device__ __forceinline__ double sc(double v) const { return v; }
};
struct GatherScaled {
  const double *x;
  double        s;
  __device__ __forceinline__ double ld(const double *p) const { return __ldg(p) * s; }
  __device__ __forceinline__ double sc(double v) const { return v * s; }
};

// two coded rows of compile-time length at once (each consumer thread owns rows t and t + PK_CT of a tile): 2 L gathers in flight
template <int L, bool PAD, class G>
__device__ __forceinline__ void pk_row2_fixed(uint32_t code_a0, uint32_t code_a1, uint32_t dv_a, uint32_t dd_a, const G &gx, int r0, int r1,
                                              uint32_t pad, double &s0, double &s1)
{
  uint32_t c0[L], c1[L];
  int      d0[L], d1[L];
  double   x0[L], x1[L];
#pragma unroll
  for (int j = 0; j < L; j++) c0[j] = lds_u8(code_a0 + j);
#pragma unroll
  for (int j = 0; j < L; j++) c1[j] = lds_u8(code_a1 + j);
#pragma unroll
  for (int j = 0; j < L; j++) d0[j] = lds_s32(dd_a + 4u * c0[j]);
#pragma unroll
  for (int j = 0; j < L; j++) d1[j] = lds_s32(dd_a + 4u * c1[j]);
#pragma unroll
  for (int j = 0; j < L; j++) x0[j] = gx.ld(gx.x + (r0 + d0[j]));   // a skip code gathers x[r] (delta 0) and drops it
#pragma unroll
  for (int j = 0; j < L; j++) x1[j] = gx.ld(gx.x + (r1 + d1[j]));
  // scheduling fence (the consumer warps are converged here): every gather above is issued before the first multiply-add below
  __syncwarp();
  s0 = 0.0;
#pragma unroll
  for (int j = 0; j < L; j++) {
    const double v = lds_f64(dv_a + 8u * c0[j]);
    if (!PAD || c0[j] != pad) s0 += v * x0[j];
  }
  s1 = 0.0;
#pragma unroll
  for (int j = 0; j < L; j++) {
    const double v = lds_f64(dv_a + 8u * c1[j]);
    if (!PAD || c1[j] != pad) s1 += v * x1[j];
  }
}

template <bool PAD, class G>
__device__ __forceinline__ bool pk_row2_dispatch(uint32_t ulen, uint32_t ca0, uint32_t ca1, uint32_t dv_a, uint32_t dd_a, const G &gx, int r0,
                                                 int r1, uint32_t pad, double &s0, double &s1)
{
  switch (ulen) {
  case 1: pk_row2_fixed<1, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 2: pk_row2_fixed<2, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 3: pk_row2_fixed<3, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 4: pk_row2_fixed<4, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 5: pk_row2_fixed<5, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 6: pk_row2_fixed<6, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 7: pk_row2_fixed<7, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  case 8: pk_row2_fixed<8, PAD, G>(ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1); return true;
  default: return false;
  }
}

// coded row of run-time length: chunks of PK_UNROLL with the same load-first order
template <class G>
__device__ __forceinline__ double pk_row_var(uint32_t code_a, int len, uint32_t dv_a, uint32_t dd_a, const G &gx, int r, uint32_t pad)
{
  double sum = 0.0;
  for (int k = 0; k < len; k += PK_UNROLL) {
    uint32_t c[PK_UNROLL];
    int      d[PK_UNROLL];
    double   xv[PK_UNROLL], vv[PK_UNROLL];
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) c[j] = (k + j < len) ? lds_u8(code_a + k + j) : 0u;
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) d[j] = lds_s32(dd_a + 4u * c[j]);
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) xv[j] = (k + j < len) ? gx.ld(gx.x + (r + d[j])) : 0.0;
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) vv[j] = lds_f64(dv_a + 8u * c[j]);
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++)
      if (k + j < len && c[j] != pad) sum += vv[j] * xv[j];
  }
  return sum;
}

template <class G>
__device__ __forceinline__ double pk_row_raw(uint32_t a_a, uint32_t ja_a, int len, const G &gx)
{
  double sum = 0.0;
  for (int k = 0; k < len; k += PK_UNROLL) {
    int    col[PK_UNROLL];
    double xv[PK_UNROLL], vv[PK_UNROLL];
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) col[j] = (k + j < len) ? lds_s32(ja_a + 4u * (k + j)) : 0;
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) xv[j] = (k + j < len) ? gx.ld(gx.x + col[j]) : 0.0;
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++) vv[j] = (k + j < len) ? lds_f64(a_a + 8u * (k + j)) : 0.0;
#pragma unroll
    for (int j = 0; j < PK_UNROLL; j++)
      if (k + j < len) sum += vv[j] * xv[j];
  }
  return sum;
}

// stencil tile (kind 2): every row of the tile is the tile's pattern -- L <= 8 (col - row, value) pairs in storage order -- with some
// entries missing (rows next to a grid boundary); one presence byte per row instead of one code byte per non-zero.  Deltas and values
// are warp-uniform (broadcast shared-memory loads), a row costs its gathers and multiply-adds only.  A missing entry is skipped
// (predicated load and multiply-add), so the sum runs over the row's stored entries in storage order: bit-identical to the CSR kernels.
template <int L, class G>
__device__ __forceinline__ void st_row2_fixed(uint32_t m0, uint32_t m1, uint32_t dv_a, uint32_t dd_a, const G &gx, int r0, int r1, double &s0, double &s1)
{
  constexpr uint32_t FULL = (1u << L) - 1u;
  int                d[L];
  double             x0[L], x1[L];
#pragma unroll
  for (int j = 0; j < L; j++) d[j] = lds_s32(dd_a + 4u * j);
  const double *xr0 = gx.x + r0, *xr1 = gx.x + r1;
  const bool    f0 = __all_sync(0xffffffffu, m0 == FULL), f1 = __all_sync(0xffffffffu, m1 == FULL);
  if (f0) {
#pragma unroll
    for (int j = 0; j < L; j++) x0[j] = gx.ld(xr0 + d[j]);
  } else {
#pragma unroll
    for (int j = 0; j < L; j++) x0[j] = ((m0 >> j) & 1u) ? gx.ld(xr0 + d[j]) : 0.0;
  }
  if (f1) {
#pragma unroll
    for (int j = 0; j < L; j++) x1[j] = gx.ld(xr1 + d[j]);
  } else {
#pragma unroll
    for (int j = 0; j < L; j++) x1[j] = ((m1 >> j) & 1u) ? gx.ld(xr1 + d[j]) : 0.0;
  }
  __syncwarp();   // scheduling fence: every gather above is issued before the first multiply-add below
  double v[L];
#pragma unroll
  for (int j = 0; j < L; j++) v[j] = lds_f64(dv_a + 8u * j);
  s0 = 0.0;
  s1 = 0.0;
  if (f0) {
#pragma unroll
    for (int j = 0; j < L; j++) s0 += v[j] * x0[j];
  } else {
#pragma unroll
    for (int j = 0; j < L; j++)
      if ((m0 >> j) & 1u) s0 += v[j] * x0[j];
  }
  if (f1) {
#pragma unroll
    for (int j = 0; j < L; j++) s1 += v[j] * x1[j];
  } else {
#pragma unroll
    for (int j = 0; j < L; j++)
      if ((m1 >> j) & 1u) s1 += v[j] * x1[j];
  }
}
template <class G>
__device__ __forceinline__ void st_row2_dispatch(uint32_t L, uint32_t m0, uint32_t m1, uint32_t dv_a, uint32_t dd_a, const G &gx, int r0, int r1, double &s0,
                                                 double &s1)
{
  switch (L) {
  case 1: st_row2_fixed<1>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 2: st_row2_fixed<2>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 3: st_row2_fixed<3>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 4: st_row2_fixed<4>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 5: st_row2_fixed<5>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 6: st_row2_fixed<6>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  case 7: st_row2_fixed<7>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  default: st_row2_fixed<8>(m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1); break;
  }
}

// i-th tile of the walk: tiles [ta, tb) first -- ascending, or descending when `rev` -- then the tiles outside that range
__device__ __forceinline__ int tile_at(int i, int ta, int tb, bool rev)
{
  const int ni = tb - ta;
  if (i < ni) return rev ? tb - 1 - i : ta + i;
  const int j = i - ni;
  return j < ta ? j : tb + (j - ta);
}

template <class Epi, int MINB>
__global__ void __launch_bounds__(PK_CT + 32, MINB) k_spmv_pk(CsrDev A, const double *__restrict__ x, Epi epi, int blob_cap, int nstages, int vec_tma, TileOrder ord)
{
  pdl_enter();
  if (!epi.active()) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[TMA_MAX_STAGES], empty_bar[TMA_MAX_STAGES];
  const int nv = epi.nvec();
  const int stage_bytes = blob_cap + nv * TR * 8;
  const int ntiles = (A.n + TR - 1) / TR;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool rev = epi.reverse();
  const typename Epi::Gather gx = epi.gather(x);
  typename Epi::Acc acc;
  epi.init(acc);
  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], PK_CT / 32);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == PK_CT / 32) {
    // ------------------------------ producer warp ------------------------------
    unsigned o0n = 0, o1n = 0;
    if (blockIdx.x < ntiles) {
      const int t0 = tile_at(blockIdx.x, ord.ta, ord.tb, rev);
      o0n = __ldg(A.pk_off + t0);
      o1n = __ldg(A.pk_off + t0 + 1);
    }
    int      s = 0, filled = 0;
    uint32_t ph = 0;
    for (int i = blockIdx.x; i < ntiles; i += gridDim.x) {
      const int      tile = tile_at(i, ord.ta, ord.tb, rev);
      const unsigned o0 = o0n, o1 = o1n;
      const int      ni = i + gridDim.x;
      if (ni < ntiles) {   // directory entry of the next tile: in flight while this one is issued
        const int nt = tile_at(ni, ord.ta, ord.tb, rev);
        o0n = __ldg(A.pk_off + nt);
        o1n = __ldg(A.pk_off + nt + 1);
      }
      if (filled >= nstages) mbar_wait(&empty_bar[s], ph ^ 1u);
      else filled++;
      unsigned char *st = smem_raw + (size_t)s * stage_bytes;
      const int      r0 = tile * TR, r1 = min(r0 + TR, A.n);
      const uint32_t blob_bytes = (o1 - o0) * 16u;
      if (r1 - r0 == TR && vec_tma) {
        if (lane == 0) {
          mbar_arrive_expect_tx(&full_bar[s], blob_bytes + (uint32_t)nv * TR * 8u);
          bulk_g2s(st, A.pk + (size_t)o0 * 16, blob_bytes, &full_bar[s]);
          for (int v = 0; v < nv; v++) bulk_g2s(st + blob_cap + (size_t)v * TR * 8, epi.vsrc(v) + r0, (uint32_t)TR * 8u, &full_bar[s]);
        }
      } else {
        // last (partial) tile, or caller vectors that are not 16-byte aligned: the warp stages the vector slices itself
        for (int v = 0; v < nv; v++) {
          double       *vs = (double *)(st + blob_cap) + (size_t)v * TR;
          const double *src = epi.vsrc(v) + r0;
          for (int t = lane; t < r1 - r0; t += 32) vs[t] = src[t];
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_expect_tx(&full_bar[s], blob_bytes);
          bulk_g2s(st, A.pk + (size_t)o0 * 16, blob_bytes, &full_bar[s]);
        }
      }
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  } else {
    // ------------------------------ consumer warps: two rows (t, t + PK_CT) per thread ------------------------------
    const uint32_t smem_a = smem_u32(smem_raw);
    int            s = 0;
    uint32_t       ph = 0;
    for (int i = blockIdx.x; i < ntiles; i += gridDim.x) {
      const int tile = tile_at(i, ord.ta, ord.tb, rev);
      mbar_wait(&full_bar[s], ph);
      const uint32_t st_a = smem_a + (uint32_t)s * (uint32_t)stage_bytes;
      const uint32_t vs_a = st_a + (uint32_t)blob_cap + 8u * threadIdx.x;
      const uint4    hw = lds_v4(st_a);   // PkHeader
      const uint32_t kind = hw.x & 0xFFFFu, nd = hw.x >> 16, nnz = hw.y, ulen = hw.z & 0xFFFFu, nrows = hw.z >> 16;
      const uint32_t pad = hw.w - 1u;   // skip code of padded tiles, 0xFFFFFFFF when the tile has none
      const int      r0 = tile * TR + threadIdx.x, r1 = r0 + PK_CT;
      const uint32_t dv_a = st_a + (uint32_t)sizeof(PkHeader);
      const uint32_t dd_a = dv_a + ((nd + 1u) & ~1u) * 8u;
      const uint32_t q_a = dd_a + ((nd + 3u) & ~3u) * 4u;
      bool           done = false;
      if (kind == 2) {
        // stencil tile: pattern of nd entries + one presence byte per row (rows beyond the matrix end carry an empty mask)
        const uint32_t m0 = (threadIdx.x < nrows) ? lds_u8(q_a + threadIdx.x) : 0u;
        const uint32_t m1 = (threadIdx.x + PK_CT < nrows) ? lds_u8(q_a + threadIdx.x + PK_CT) : 0u;
        double         s0, s1;
        st_row2_dispatch(nd, m0, m1, dv_a, dd_a, gx, r0, r1, s0, s1);
        if (r0 < A.n) epi.row_s(r0, vs_a, s0, acc);
        if (r1 < A.n) epi.row_s(r1, vs_a + PK_CT * 8u, s1, acc);
        done = true;
      } else if (kind == 1 && ulen != 0xFFFFu && nrows == TR) {
        // full tile of equal-length coded rows: both rows together, loads up front
        const uint32_t ca0 = q_a + threadIdx.x * ulen, ca1 = ca0 + PK_CT * ulen;
        double         s0 = 0.0, s1 = 0.0;
        done = pad != 0xFFFFFFFFu ? pk_row2_dispatch<true>(ulen, ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1)
                                  : pk_row2_dispatch<false>(ulen, ca0, ca1, dv_a, dd_a, gx, r0, r1, pad, s0, s1);
        if (done) {
          epi.row_s(r0, vs_a, s0, acc);
          epi.row_s(r1, vs_a + PK_CT * 8u, s1, acc);
        }
      }
      if (!done) {
#pragma unroll 1
        for (int h = 0; h < 2; h++) {
          const uint32_t t = threadIdx.x + h * PK_CT;
          const int      r = tile * TR + (int)t;
          if (r >= A.n) break;
          double sum;
          if (kind == 1) {
            if (ulen != 0xFFFFu) {
              sum = pk_row_var(q_a + t * ulen, (int)ulen, dv_a, dd_a, gx, r, pad);
            } else {
              const uint32_t ks = lds_u16(q_a + 2u * t), ke = lds_u16(q_a + 2u * t + 2u);
              sum = pk_row_var(q_a + ((nrows + 1u + 7u) & ~7u) * 2u + ks, (int)(ke - ks), dv_a, dd_a, gx, r, pad);
            }
          } else {
            const uint32_t a_a = st_a + (uint32_t)sizeof(PkHeader);
            const uint32_t ja_a = a_a + ((nnz + 1u) & ~1u) * 8u;
            const uint32_t ro_a = ja_a + ((nnz + 3u) & ~3u) * 4u;
            const uint32_t ks = lds_u16(ro_a + 2u * t), ke = lds_u16(ro_a + 2u * t + 2u);
            sum = pk_row_raw(a_a + 8u * ks, ja_a + 4u * ks, (int)(ke - ks), gx);
          }
          epi.row_s(r, st_a + (uint32_t)blob_cap + 8u * t, sum, acc);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  }
  epi.finalize(acc);
}


// ---- all-stencil matrices (kind 4): x windows staged by bulk copies, gathers are shared-memory loads ----------------------------
// Stage layout: [16 B descriptor: pattern id, windowed flag][256 B presence bytes][st_nwin windows of PB_ST_WCAP bytes][nv row slices of
// the epilogue vectors].  The pattern table sits in front of the stages.  A tile whose windows would reach outside x (the first / last
// rows of the local block) or that is partial takes the gather path (LDG) with the same pattern; everything else never issues a
// long-latency load from a consumer warp: the copy engine streams, the consumer warps only do shared-memory loads and DFMAs.
static constexpr uint32_t ST_MASK_OFF = 16, ST_WIN_OFF = 16 + TR;
template <int L, class G>
__device__ __forceinline__ void st_win2_fixed(uint32_t m0, uint32_t m1, uint32_t P_a, uint32_t win_a, const G &gx, double &s0, double &s1)
{
  constexpr uint32_t FULL = (1u << L) - 1u;
  uint32_t           e[L];
  double             v[L];
#pragma unroll
  for (int j = 0; j < L; j++) e[j] = win_a + (uint32_t)lds_s32(P_a + (uint32_t)offsetof(StPattern, erel) + 4u * j);
#pragma unroll
  for (int j = 0; j < L; j++) v[j] = lds_f64(P_a + (uint32_t)offsetof(StPattern, v) + 8u * j);
  s0 = 0.0;
  s1 = 0.0;
  if (__all_sync(0xffffffffu, m0 == FULL)) {
#pragma unroll
    for (int j = 0; j < L; j++) s0 += v[j] * gx.sc(lds_f64(e[j]));
  } else {
#pragma unroll
    for (int j = 0; j < L; j++)
      if ((m0 >> j) & 1u) s0 += v[j] * gx.sc(lds_f64(e[j]));
  }
  if (__all_sync(0xffffffffu, m1 == FULL)) {
#pragma unroll
    for (int j = 0; j < L; j++) s1 += v[j] * gx.sc(lds_f64(e[j] + PK_CT * 8u));
  } else {
#pragma unroll
    for (int j = 0; j < L; j++)
      if ((m1 >> j) & 1u) s1 += v[j] * gx.sc(lds_f64(e[j] + PK_CT * 8u));
  }
}
template <class G>
__device__ __forceinline__ void st_win2_dispatch(uint32_t L, uint32_t m0, uint32_t m1, uint32_t P_a, uint32_t win_a, const G &gx, double &s0, double &s1)
{
  switch (L) {
  case 1: st_win2_fixed<1>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 2: st_win2_fixed<2>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 3: st_win2_fixed<3>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 4: st_win2_fixed<4>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 5: st_win2_fixed<5>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 6: st_win2_fixed<6>(m0, m1, P_a, win_a, gx, s0, s1); break;
  case 7: st_win2_fixed<7>(m0, m1, P_a, win_a, gx, s0, s1); break;
  default: st_win2_fixed<8>(m0, m1, P_a, win_a, gx, s0, s1); break;
  }
}

template <class Epi>
__global__ void __launch_bounds__(PK_CT + 32, 4) k_spmv_st(CsrDev A, const double *__restrict__ x, Epi epi, int nstages, int stage_bytes, int pats_bytes, int win_ok, int vec_tma,
                                                           TileOrder ord)
{
  pdl_enter();
  if (!epi.active()) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[TMA_MAX_STAGES], empty_bar[TMA_MAX_STAGES];
  const int  nv = epi.nvec();
  const int  vec_off = (int)ST_WIN_OFF + A.st_nwin * PB_ST_WCAP;
  const int  ntiles = (A.n + TR - 1) / TR;
  const int  warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool rev = epi.reverse();
  const typename Epi::Gather gx = epi.gather(x);
  typename Epi::Acc acc;
  epi.init(acc);
  {   // pattern table -> shared memory (a few hundred bytes per pattern)
    const int      nw = A.st_npat * (int)(sizeof(StPattern) / 4);
    const int     *src = reinterpret_cast<const int *>(A.st_pats);
    int           *dst = reinterpret_cast<int *>(smem_raw);
    for (int k = threadIdx.x; k < nw; k += blockDim.x) dst[k] = __ldg(src + k);
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], PK_CT / 32);
    }
    mbar_fence_init();
  }
  __syncthreads();
  unsigned char *stages = smem_raw + pats_bytes;

  if (warp == PK_CT / 32) {
    // ------------------------------ producer warp ------------------------------
    int pidn = 0;
    if (blockIdx.x < ntiles) pidn = __ldg(A.st_pid + tile_at(blockIdx.x, ord.ta, ord.tb, rev));
    int      s = 0, filled = 0;
    uint32_t ph = 0;
    for (int i = blockIdx.x; i < ntiles; i += gridDim.x) {
      const int tile = tile_at(i, ord.ta, ord.tb, rev);
      const int pid = pidn;
      const int ni = i + gridDim.x;
      if (ni < ntiles) pidn = __ldg(A.st_pid + tile_at(ni, ord.ta, ord.tb, rev));   // in flight while this tile is issued
      if (filled >= nstages) mbar_wait(&empty_bar[s], ph ^ 1u);
      else filled++;
      unsigned char   *st = stages + (size_t)s * stage_bytes;
      const StPattern *P = reinterpret_cast<const StPattern *>(smem_raw) + pid;
      const int        r0 = tile * TR, r1 = min(r0 + TR, A.n);
      const bool       fullt = (r1 - r0 == TR) && vec_tma;
      bool             windowed = fullt && win_ok;
      uint32_t         wbytes = 0;
      const int        nwin = P->nwin;
      for (int w = 0; w < nwin; w++) {
        const int lo = r0 + P->wlo[w];
        if (lo < 0 || lo + P->wlen[w] > A.ncols) windowed = false;
        wbytes += (uint32_t)P->wlen[w] * 8u;
      }
      if (lane == 0) {
        reinterpret_cast<int *>(st)[0] = pid;
        reinterpret_cast<int *>(st)[1] = windowed ? 1 : 0;
      }
      if (fullt) {
        if (lane == 0) {
          mbar_arrive_expect_tx(&full_bar[s], (uint32_t)TR + (uint32_t)nv * TR * 8u + (windowed ? wbytes : 0u));
          bulk_g2s(st + ST_MASK_OFF, A.st_masks + r0, (uint32_t)TR, &full_bar[s]);
          if (windowed)
            for (int w = 0; w < nwin; w++) bulk_g2s(st + ST_WIN_OFF + (size_t)w * PB_ST_WCAP, x + (r0 + P->wlo[w]), (uint32_t)P->wlen[w] * 8u, &full_bar[s]);
          for (int v = 0; v < nv; v++) bulk_g2s(st + vec_off + (size_t)v * TR * 8, epi.vsrc(v) + r0, (uint32_t)TR * 8u, &full_bar[s]);
        }
      } else {
        // last (partial) tile, or caller vectors that are not 16-byte aligned: the warp stages masks and vector slices itself
        for (int t = lane; t < TR; t += 32) st[ST_MASK_OFF + t] = (t < r1 - r0) ? __ldg(A.st_masks + r0 + t) : (unsigned char)0;
        for (int v = 0; v < nv; v++) {
          double       *vs = (double *)(st + vec_off) + (size_t)v * TR;
          const double *src = epi.vsrc(v) + r0;
          for (int t = lane; t < r1 - r0; t += 32) vs[t] = src[t];
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full_bar[s]);
      }
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  } else {
    // ------------------------------ consumer warps: two rows (t, t + PK_CT) per thread ------------------------------
    const uint32_t smem_a = smem_u32(smem_raw), stages_a = smem_a + (uint32_t)pats_bytes;
    int            s = 0;
    uint32_t       ph = 0;
    for (int i = blockIdx.x; i < ntiles; i += gridDim.x) {
      const int tile = tile_at(i, ord.ta, ord.tb, rev);
      mbar_wait(&full_bar[s], ph);
      const uint32_t st_a = stages_a + (uint32_t)s * (uint32_t)stage_bytes;
      const uint32_t vs_a = st_a + (uint32_t)vec_off + 8u * threadIdx.x;
      const uint32_t pid = (uint32_t)lds_s32(st_a), windowed = (uint32_t)lds_s32(st_a + 4u);
      const uint32_t P_a = smem_a + pid * (uint32_t)sizeof(StPattern);
      const uint32_t L = (uint32_t)lds_s32(P_a);
      const uint32_t m0 = lds_u8(st_a + ST_MASK_OFF + threadIdx.x), m1 = lds_u8(st_a + ST_MASK_OFF + threadIdx.x + PK_CT);
      const int      r0 = tile * TR + threadIdx.x, r1 = r0 + PK_CT;
      double         s0, s1;
      if (windowed) st_win2_dispatch(L, m0, m1, P_a, st_a + ST_WIN_OFF + 8u * threadIdx.x, gx, s0, s1);
      else st_row2_dispatch(L, m0, m1, P_a + (uint32_t)offsetof(StPattern, v), P_a + (uint32_t)offsetof(StPattern, d), gx, r0, r1, s0, s1);
      if (r0 < A.n) epi.row_s(r0, vs_a, s0, acc);
      if (r1 < A.n) epi.row_s(r1, vs_a + PK_CT * 8u, s1, acc);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
      if (++s == nstages) {
        s = 0;
        ph ^= 1u;
      }
    }
  }
  epi.finalize(acc);
}


// ---- all-stencil matrices, direct form: no staging at all.  With a uniform pattern the gather x[r + d] of the 32 rows of a warp is ONE
// coalesced 256-byte load per pattern entry (served by L1 / L2 for the shifted copies), the presence byte only predicates it, and the
// epilogue operands are plain coalesced loads issued together with the gathers: a row costs ONE memory round trip, like the streaming
// kernels K_B / K_C, and thousands of threads keep the loads in flight -- no producer / consumer ring, no shared-memory traffic.
// LMAX = longest pattern of the matrix (5 / 7 for the Laplacians): tiles with that pattern and no missing entry take the unrolled path.
template <int LMAX, class G>
__device__ __forceinline__ double sd_row(int L, uint32_t m, const StPattern &P, const G &gx, int r)
{
  constexpr uint32_t FULL = (1u << LMAX) - 1u;
  const char        *xr = reinterpret_cast<const char *>(gx.x + r);
  if (__all_sync(0xffffffffu, L == LMAX && m == FULL)) {
    double xv[LMAX];
    int    db[LMAX];
#pragma unroll
    for (int j = 0; j < LMAX; j++) db[j] = P.d[j] * 8;
#pragma unroll
    for (int j = 0; j < LMAX; j++) xv[j] = gx.ld(reinterpret_cast<const double *>(xr + (long long)db[j]));
    __syncwarp();   // scheduling fence (the warp is converged here): every gather is issued before the first multiply-add
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < LMAX; j++) s += P.v[j] * xv[j];
    return s;
  }
  // rows with missing entries (next to a grid boundary) and tiles with a shorter pattern: same order, every load predicated and still
  // issued before the first multiply-add -- the warps that own the boundary rows of a structured grid take this path in every tile
  double xv[LMAX], vv[LMAX];
#pragma unroll
  for (int j = 0; j < LMAX; j++) {
    const bool on = (j < L) && ((m >> j) & 1u);
    xv[j]         = on ? gx.ld(reinterpret_cast<const double *>(xr + (long long)(P.d[j] * 8))) : 0.0;
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < LMAX; j++) vv[j] = P.v[j];
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < LMAX; j++)
    if ((j < L) && ((m >> j) & 1u)) s += vv[j] * xv[j];
  return s;
}

// L2 prefetch of what a future tile of this CTA will read from DRAM: the 2 KB slices of the epilogue vectors and the one gather window
// no earlier row has touched (largest offset on an ascending sweep, smallest on a descending one) -- bulk prefetches issued by one warp
// (cp.async.bulk.prefetch.L2 -> UBLKPF), no registers and no shared memory held while the lines travel.  The loads of the row loop then
// find their lines in L2 (~0.3 us) instead of HBM (~1 us under load), which is what bounds a one-round-trip-per-row kernel.
__device__ __forceinline__ void l2_prefetch_bulk(const double *p, long long e0, long long e1, long long n)
{   // elements [e0, e1) of p, clipped to [0, n) and widened to 16-byte granules inside the array
  if (e0 < 0) e0 = 0;
  if (e1 > n) e1 = n;
  uintptr_t a0 = (uintptr_t)(p + e0), a1 = (uintptr_t)(p + e1);
  a0 = (a0 + 15) & ~(uintptr_t)15;
  a1 &= ~(uintptr_t)15;
  if (a1 > a0) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a0), "r"((uint32_t)(a1 - a0)) : "memory");
}
template <class Epi>
__device__ __forceinline__ void sd_prefetch_tile(const Epi &epi, const double *gx, int tile, int rows, int n, int ncols, bool rev, const TileOrder &ord, int lane)
{
  const long long r0 = (long long)tile * rows;
  const int       nv = epi.nvec();
  if (lane == 0) {
    const int d = rev ? ord.dlo : ord.dhi;
    l2_prefetch_bulk(gx, r0 + d, r0 + d + rows, ncols);
  } else if (lane <= nv) {
    const double *v = epi.vsrc(lane - 1);
    if (v != gx) l2_prefetch_bulk(v, r0, r0 + rows, n);
  }
}

template <class Epi, int LMAX, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_spmv_sd(CsrDev A, const double *__restrict__ x, Epi epi, TileOrder ord)
{
  pdl_enter();
  if (!epi.active()) return;
  __shared__ StPattern s_pats[PB_ST_MAXPAT];
  {
    const int  nw = A.st_npat * (int)(sizeof(StPattern) / 4);
    const int *src = reinterpret_cast<const int *>(A.st_pats);
    int       *dst = reinterpret_cast<int *>(s_pats);
    for (int k = threadIdx.x; k < nw; k += NT) dst[k] = __ldg(src + k);
  }
  __syncthreads();
  const int  ntiles = (A.n + TR - 1) / TR;
  const bool rev = epi.reverse();
  const typename Epi::Gather gx = epi.gather(x);
  typename Epi::Acc acc;
  epi.init(acc);
  // presence byte and pattern id of the next tile are loaded one iteration ahead: the gathers of a row never wait for them
  uint32_t m_next = 0;
  int      pid_next = 0;
  if ((int)blockIdx.x < ntiles) {
    const int t0 = tile_at(blockIdx.x, ord.ta, ord.tb, rev);
    pid_next = __ldg(A.st_pid + t0);
    m_next   = __ldg(A.st_masks + (size_t)t0 * TR + threadIdx.x);   // the mask array is padded to whole tiles
  }
  for (int i = blockIdx.x; i < ntiles; i += gridDim.x) {
    const int      tile = tile_at(i, ord.ta, ord.tb, rev);
    const uint32_t m = m_next;
    const int      pid = pid_next;
    const int      ni = i + gridDim.x;
    const int      r = tile * TR + threadIdx.x;
    const bool     live = r < A.n;
    if (ord.pf > 0 && threadIdx.x < 32) {
      const long long pi = (long long)i + (long long)ord.pf * gridDim.x;
      if (pi < ntiles) sd_prefetch_tile(epi, gx.x, tile_at((int)pi, ord.ta, ord.tb, rev), TR, A.n, A.ncols, rev, ord, (int)threadIdx.x);
    }
    const typename Epi::Pre pre = epi.preload(live ? r : 0);   // epilogue operands: in flight together with the gathers
    if (ni < ntiles) {
      const int tn = tile_at(ni, ord.ta, ord.tb, rev);
      pid_next = __ldg(A.st_pid + tn);
      m_next   = __ldg(A.st_masks + (size_t)tn * TR + threadIdx.x);
    }
    const StPattern &P = s_pats[pid];
    const double     sum = sd_row<LMAX>(P.L, m, P, gx, r);   // rows beyond the end carry an empty mask: nothing is loaded
    if (live) epi.row_p(r, sum, pre, acc);
  }
  epi.finalize(acc);
}


// Two ADJACENT rows per thread (r even): the epilogue operands and results travel as 16-byte accesses, the two gathers of a pattern entry
// share one address computation, and the per-row share of the loop overhead (pattern operands, tile bookkeeping) is halved.  A CTA walks
// "super tiles" of 512 rows = two 256-row tiles (threads 0..127 the first, 128..255 the second: the pattern is still warp-uniform).
// Needs an even row count and 16-byte aligned vectors; k_spmv_sd is the fallback.
template <int LMAX, class G>
__device__ __forceinline__ void sd_row2(int L, uint32_t m0, uint32_t m1, const StPattern &P, const G &gx, int r, double &s0, double &s1)
{
  constexpr uint32_t FULL = (1u << LMAX) - 1u;
  const char        *xr = reinterpret_cast<const char *>(gx.x + r);
  double             x0[LMAX], x1[LMAX], vv[LMAX];
  if (__all_sync(0xffffffffu, L == LMAX && m0 == FULL && m1 == FULL)) {
#pragma unroll
    for (int j = 0; j < LMAX; j++) {
      const double *a = reinterpret_cast<const double *>(xr + (long long)(P.d[j] * 8));
      x0[j]           = gx.ld(a);
      x1[j]           = gx.ld(a + 1);
    }
    __syncwarp();   // scheduling fence: every gather is issued before the first multiply-add
#pragma unroll
    for (int j = 0; j < LMAX; j++) vv[j] = P.v[j];
    s0 = 0.0;
    s1 = 0.0;
#pragma unroll
    for (int j = 0; j < LMAX; j++) s0 += vv[j] * x0[j];
#pragma unroll
    for (int j = 0; j < LMAX; j++) s1 += vv[j] * x1[j];
    return;
  }
#pragma unroll
  for (int j = 0; j < LMAX; j++) {
    const double *a = reinterpret_cast<const double *>(xr + (long long)(P.d[j] * 8));
    const bool    on0 = (j < L) && ((m0 >> j) & 1u), on1 = (j < L) && ((m1 >> j) & 1u);
    x0[j]             = on0 ? gx.ld(a) : 0.0;
    x1[j]             = on1 ? gx.ld(a + 1) : 0.0;
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < LMAX; j++) vv[j] = P.v[j];
  s0 = 0.0;
  s1 = 0.0;
#pragma unroll
  for (int j = 0; j < LMAX; j++)
    if ((j < L) && ((m0 >> j) & 1u)) s0 += vv[j] * x0[j];
#pragma unroll
  for (int j = 0; j < LMAX; j++)
    if ((j < L) && ((m1 >> j) & 1u)) s1 += vv[j] * x1[j];
}

template <class Epi, int LMAX, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_spmv_sd2(CsrDev A, const double *__restrict__ x, Epi epi, TileOrder ord)
{
  pdl_enter();
  if (!epi.active()) return;
  __shared__ StPattern s_pats[PB_ST_MAXPAT];
  {
    const int  nw = A.st_npat * (int)(sizeof(StPattern) / 4);
    const int *src = reinterpret_cast<const int *>(A.st_pats);
    int       *dst = reinterpret_cast<int *>(s_pats);
    for (int k = threadIdx.x; k < nw; k += NT) dst[k] = __ldg(src + k);
  }
  __syncthreads();
  const int  nst = (A.n + 2 * TR - 1) / (2 * TR);   // super tiles (the mask / pattern-id arrays are padded to an even number of tiles)
  const int  half = threadIdx.x >> 7;
  const bool rev = epi.reverse();
  const typename Epi::Gather gx = epi.gather(x);
  typename Epi::Acc acc;
  epi.init(acc);
  uchar2 m_next = make_uchar2(0, 0);
  int    pid_next = 0;
  if ((int)blockIdx.x < nst) {
    const int t0 = tile_at(blockIdx.x, ord.ta, ord.tb, rev);
    pid_next = __ldg(A.st_pid + 2 * t0 + half);
    m_next   = __ldg(reinterpret_cast<const uchar2 *>(A.st_masks + (size_t)t0 * (2 * TR)) + threadIdx.x);
  }
  for (int i = blockIdx.x; i < nst; i += gridDim.x) {
    const int    st = tile_at(i, ord.ta, ord.tb, rev);
    const uchar2 m = m_next;
    const int    pid = pid_next;
    const int    ni = i + gridDim.x;
    const int    r = st * (2 * TR) + 2 * (int)threadIdx.x;
    const bool   live = r < A.n;   // n is even: r + 1 < n as well
    const typename Epi::Pre2 pre = epi.preload2(live ? r : 0);
    if (ni < nst) {
      const int tn = tile_at(ni, ord.ta, ord.tb, rev);
      pid_next = __ldg(A.st_pid + 2 * tn + half);
      m_next   = __ldg(reinterpret_cast<const uchar2 *>(A.st_masks + (size_t)tn * (2 * TR)) + threadIdx.x);
    }
    const StPattern &P = s_pats[pid];
    double           s0, s1;
    sd_row2<LMAX>(P.L, m.x, m.y, P, gx, r, s0, s1);
    if (live) epi.row2_p(r, s0, s1, pre, acc);
  }
  epi.finalize(acc);
}

template <class K>
static int occ_blocks(K kernel, size_t smem)
{
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, NT, smem) != cudaSuccess || nb < 1) nb = 1;
  return nb;
}

template <class Epi, int W>
static void launch_vector(const CsrDev &A, const double *x, const Epi &epi)
{
  static int occ = 0;
  if (!occ) occ = occ_blocks(k_spmv_vector<Epi, W>, 0);
  int64_t need = ((int64_t)A.n * W + NT - 1) / NT;
  int64_t grid = (int64_t)g_ctx.sm_count * occ;
  if (grid > need) grid = need;
  if (grid > max_red_blocks()) grid = max_red_blocks();
  if (grid < 1) grid = 1;
  k_spmv_vector<Epi, W><<<(int)grid, NT, 0, g_ctx.stream>>>(A, x, epi);
}



// ---- long rows (SVM factors: ~1000 non-zeros per row): tile-ELL -----------------------------------------------------------------
// The lanes-per-row kernel reads a row with unit stride but gathers x with one 32-byte sector per non-zero from L2 (2.7x the matrix
// stream at C4).  Here a tile of 256 rows is stored column-major, one thread owns a row: entry t of 32 rows is one 256-byte line of values
// and one 128-byte line of columns, the gathers of a warp at step t fall into the same column neighbourhood when the rows are similar
// (sorted columns: the t-th entry of every row sits near t/len of the column range), and the products are added in storage order.
static constexpr int ELL_U = 8;
template <class Epi>
__global__ void __launch_bounds__(NT, 3) k_spmv_ell(CsrDev A, const double *__restrict__ x, Epi epi)
{
  pdl_enter();
  if (!epi.active()) return;
  typename Epi::Acc acc;
  epi.init(acc);
  const int ntiles = (A.n + TR - 1) / TR;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int     r = tile * TR + threadIdx.x;
    const int     len = (r < A.n) ? __ldg(A.ell_len + r) : 0;
    const int     lt = __ldg(A.ell_lt + tile);
    const double *val = A.ell_val + __ldg(A.ell_off + tile) + threadIdx.x;
    const int    *col = A.ell_col + __ldg(A.ell_off + tile) + threadIdx.x;
    double        s = 0.0;
    for (int t = 0; t < lt; t += ELL_U) {
      int    c[ELL_U];
      double v[ELL_U], xv[ELL_U];
#pragma unroll
      for (int j = 0; j < ELL_U; j++) {
        const bool on = t + j < len;
        c[j]          = on ? __ldcs(col + (size_t)(t + j) * TR) : 0;
        v[j]          = on ? __ldcs(val + (size_t)(t + j) * TR) : 0.0;
      }
#pragma unroll
      for (int j = 0; j < ELL_U; j++) xv[j] = (t + j < len) ? __ldg(x + c[j]) : 0.0;
#pragma unroll
      for (int j = 0; j < ELL_U; j++)
        if (t + j < len) s += v[j] * xv[j];
    }
    if (r < A.n) epi.row(r, s, acc);
  }
  epi.finalize(acc);
}

template <class Epi>
static void launch_ell(const CsrDev &A, const double *x, const Epi &epi)
{
  static int occ = 0;
  if (!occ) occ = occ_blocks(k_spmv_ell<Epi>, 0);
  int ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
  if (grid > ntiles) grid = ntiles;
  if (grid > max_red_blocks()) grid = max_red_blocks();
  if (grid < 1) grid = 1;
  launch_k(k_spmv_ell<Epi>, grid, NT, 0, A, x, epi);
}

// CSR -> tile-ELL on the device: one CTA per tile, thread r walks its row and scatters it into the column-major tile
__global__ void __launch_bounds__(NT) k_csr_to_ell(int n, const int *__restrict__ ia, const int *__restrict__ ja, const double *__restrict__ a, const int64_t *__restrict__ off,
                                                   const int *__restrict__ lt, double *__restrict__ ev, int *__restrict__ ec, int *__restrict__ elen)
{
  const int tile = blockIdx.x, r = tile * TR + threadIdx.x;
  const int L = lt[tile];
  const int k0 = (r < n) ? ia[r] : 0, len = (r < n) ? ia[r + 1] - k0 : 0;
  if (r < n) elen[r] = len;
  double *v = ev + off[tile] + threadIdx.x;
  int    *c = ec + off[tile] + threadIdx.x;
  for (int t = 0; t < L; t++) {
    v[(size_t)t * TR] = (t < len) ? a[k0 + t] : 0.0;
    c[(size_t)t * TR] = (t < len) ? ja[k0 + t] : 0;
  }
}
int csr_to_tile_ell(CsrDev &A, const int *h_ia)
{
  const int        ntiles = (A.n + TR - 1) / TR;
  std::vector<int> maxrow((size_t)ntiles);
  for (int t = 0; t < ntiles; t++) {
    int L = 0;
    for (int r = t * TR; r < std::min(A.n, (t + 1) * TR); r++) L = std::max(L, h_ia[r + 1] - h_ia[r]);
    maxrow[t] = L;
  }
  return csr_to_tile_ell_widths(A, maxrow);
}
int csr_to_tile_ell_widths(CsrDev &A, const std::vector<int> &tile_maxrow)
{
  const int ntiles = (A.n + TR - 1) / TR;
  if (ntiles == 0 || !A.ia || !A.ja || !A.a) return 0;
  std::vector<int64_t> off((size_t)ntiles);
  std::vector<int>     lt((size_t)ntiles);
  int64_t              tot = 0;
  for (int t = 0; t < ntiles; t++) {
    const int L = (tile_maxrow[t] + ELL_U - 1) / ELL_U * ELL_U;
    lt[t]       = L;
    off[t]      = tot;
    tot += (int64_t)L * TR;
  }
  if (tot > (int64_t)(1.3 * (double)A.nnz) + 65536) return 0;   // ragged rows: the padding would cost more than it saves
  double  *ev;
  int     *ec, *el, *dlt;
  int64_t *doff;
  PB_CHK(dmalloc(&ev, (size_t)tot));
  PB_CHK(dmalloc(&ec, (size_t)tot));
  PB_CHK(dmalloc(&el, (size_t)std::max(A.n, 1)));
  PB_CHK(dmalloc(&dlt, (size_t)ntiles));
  PB_CHK(dmalloc(&doff, (size_t)ntiles));
  PB_CUDA(cudaMemcpyAsync(dlt, lt.data(), sizeof(int) * (size_t)ntiles, cudaMemcpyHostToDevice, g_ctx.stream));
  PB_CUDA(cudaMemcpyAsync(doff, off.data(), sizeof(int64_t) * (size_t)ntiles, cudaMemcpyHostToDevice, g_ctx.stream));
  k_csr_to_ell<<<ntiles, NT, 0, g_ctx.stream>>>(A.n, A.ia, A.ja, A.a, doff, dlt, ev, ec, el);
  LAUNCH_CHECK();
  PB_CUDA(cudaStreamSynchronize(g_ctx.stream));   // lt / off are locals
  dfree(A.ia);
  dfree(A.ja);
  dfree(A.a);
  A.ia = A.ja = nullptr;
  A.a  = nullptr;
  A.ell_val   = ev;
  A.ell_col   = ec;
  A.ell_len   = el;
  A.ell_lt    = dlt;
  A.ell_off   = doff;
  A.ell_elems = tot;
  A.kind      = 5;
  return 0;
}

template <class Epi, class = void>
struct EpiHasStaged : std::false_type {};
template <class Epi>
struct EpiHasStaged<Epi, std::void_t<decltype(std::declval<const Epi &>().nvec())>> : std::true_type {};


template <class Epi>
static void launch_tma(const CsrDev &A, const double *x, const Epi &epi)
{
  if constexpr (!EpiHasStaged<Epi>::value) {
    // epilogues without a staged-vector interface (ghost pass) use the plain streamed kernel
    size_t smem = (size_t)A.tile_cap * sizeof(double);
    int    occ = occ_blocks(k_spmv_stream<Epi>, smem);
    int    ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
    if (grid > ntiles) grid = ntiles;
    k_spmv_stream<Epi><<<grid, NT, smem, g_ctx.stream>>>(A, x, epi);
  } else {
    // host mirror of the epilogue's vector list: all sources must be 16-byte aligned for cp.async.bulk
    const int nv = epi.nvec_host();
    bool      ok = aligned16(A.a) && aligned16(A.ja) && aligned16(A.ia);
    for (int v = 0; v < nv && ok; v++) ok = aligned16(epi.vsrc_host(v));
    const int      cap = A.tile_cap;
    const TmaStage L = tma_stage_layout(cap, nv);
    int            nstages = A.stages > 0 ? A.stages : 2;
    if (nstages > TMA_MAX_STAGES) nstages = TMA_MAX_STAGES;
    size_t smem = (size_t)L.bytes * nstages;
    if (!ok || smem > 200 * 1024) {
      size_t sm1 = (size_t)A.tile_cap * sizeof(double);
      int    occ = occ_blocks(k_spmv_stream<Epi>, sm1);
      int    ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
      if (grid > ntiles) grid = ntiles;
      k_spmv_stream<Epi><<<grid, NT, sm1, g_ctx.stream>>>(A, x, epi);
      return;
    }
    static size_t attr_smem = 0;
    if (smem > attr_smem) {
      cudaFuncSetAttribute(k_spmv_tma<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      attr_smem = smem;
    }
    static int    occ = 0;
    static size_t occ_smem = (size_t)-1;
    if (!occ || occ_smem != smem) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_spmv_tma<Epi>, NT + 32, smem) != cudaSuccess || nb < 1) nb = 1;
      occ      = nb;
      occ_smem = smem;
    }
    int ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
    if (grid > ntiles) grid = ntiles;
    if (grid > max_red_blocks()) grid = max_red_blocks();
    k_spmv_tma<Epi><<<grid, NT + 32, smem, g_ctx.stream>>>(A, x, epi, cap, nstages);
  }
}


template <class Epi>
static int launch_pk(const CsrDev &A, const double *x, const Epi &epi, TileOrder ord)
{
  if constexpr (!EpiHasStaged<Epi>::value) {
    set_error("internal: epilogue without staged vectors on a packed matrix");
    return 76;
  } else {
    const int nv = epi.nvec_host();
    int       vec_tma = 1;
    for (int v = 0; v < nv && vec_tma; v++) vec_tma = aligned16(epi.vsrc_host(v));
    const int blob_cap = (A.pk_max + 127) & ~127;
    const size_t stage = (size_t)blob_cap + (size_t)nv * TR * 8;
    int          nstages = A.stages > 0 ? A.stages : 3;
    if (nstages > TMA_MAX_STAGES) nstages = TMA_MAX_STAGES;
    while (nstages > 1 && stage * nstages > 200 * 1024) nstages--;
    const size_t smem = stage * nstages;
    if (smem > 220 * 1024) {
      set_error("packed SpMV tile does not fit in shared memory (%zu bytes)", smem);
      return 76;
    }
    // register budget: 5 CTAs per SM (72 registers) by default, PERMON_B200_PK_OCC=4 lets the compiler use 96 (A/B measurements)
    static int minb = 0;
    if (!minb) {
      const char *e = getenv("PERMON_B200_PK_OCC");
      minb = (e && atoi(e) == 4) ? 4 : 5;
    }
    auto kern = (minb == 4) ? k_spmv_pk<Epi, 4> : k_spmv_pk<Epi, 5>;
    static size_t attr_smem = 0;
    if (smem > attr_smem) {
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      attr_smem = smem;
    }
    static int    occ = 0;
    static size_t occ_smem = (size_t)-1;
    if (!occ || occ_smem != smem) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, PK_CT + 32, smem) != cudaSuccess || nb < 1) nb = 1;
      occ      = nb;
      occ_smem = smem;
    }
    int ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
    if (grid > ntiles) grid = ntiles;
    if (grid > max_red_blocks()) grid = max_red_blocks();
    if (ord.tb <= ord.ta || ord.tb > ntiles) {   // no preference: all tiles in index order
      ord.ta = 0;
      ord.tb = ntiles;
    }
    launch_k(kern, grid, PK_CT + 32, smem, A, x, epi, blob_cap, nstages, vec_tma, ord);
    return 0;
  }
}


template <class Epi>
static int launch_st(const CsrDev &A, const double *x, const Epi &epi, TileOrder ord)
{
  if constexpr (!EpiHasStaged<Epi>::value) {
    set_error("internal: epilogue without staged vectors on a stencil matrix");
    return 76;
  } else {
    const int nv = epi.nvec_host();
    int       vec_tma = aligned16(A.st_masks) ? 1 : 0;
    for (int v = 0; v < nv && vec_tma; v++) vec_tma = aligned16(epi.vsrc_host(v));
    const int    win_ok = aligned16(x) ? 1 : 0;
    const int    pats_bytes = (int)((A.st_npat * sizeof(StPattern) + 127) & ~(size_t)127);
    const size_t stage = ((size_t)ST_WIN_OFF + (size_t)A.st_nwin * PB_ST_WCAP + (size_t)nv * TR * 8 + 127) & ~(size_t)127;
    // stages: as many as leave room for 4 CTAs per SM (the windows make a stage 14-20 KB), at least 2
    int nstages = A.stages > 0 ? A.stages : (int)(((size_t)224 * 1024 / 4 - 1024 - (size_t)pats_bytes) / stage);
    if (nstages > TMA_MAX_STAGES) nstages = TMA_MAX_STAGES;
    if (nstages < 2) nstages = 2;
    const size_t smem = (size_t)pats_bytes + stage * nstages;
    if (smem > 220 * 1024) {
      set_error("stencil SpMV stage does not fit in shared memory (%zu bytes)", smem);
      return 76;
    }
    static size_t attr_smem = 0;
    if (smem > attr_smem) {
      cudaFuncSetAttribute(k_spmv_st<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      attr_smem = smem;
    }
    static int    occ = 0;
    static size_t occ_smem = (size_t)-1;
    if (!occ || occ_smem != smem) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_spmv_st<Epi>, PK_CT + 32, smem) != cudaSuccess || nb < 1) nb = 1;
      occ      = nb;
      occ_smem = smem;
    }
    int ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
    if (grid > ntiles) grid = ntiles;
    if (grid > max_red_blocks()) grid = max_red_blocks();
    if (ord.tb <= ord.ta || ord.tb > ntiles) {
      ord.ta = 0;
      ord.tb = ntiles;
    }
    launch_k(k_spmv_st<Epi>, grid, PK_CT + 32, smem, A, x, epi, nstages, (int)stage, pats_bytes, win_ok, vec_tma, ord);
    return 0;
  }
}


template <class Epi, int LMAX>
static int launch_sd_l(const CsrDev &A, const double *x, const Epi &epi, TileOrder ord)
{
  // CTAs per SM: 5 for one row per thread (48 registers), 4 for two (64).  The other occupancies were measured and lost (4: 0.207 ms, 6:
  // 0.133 ms against 0.127 ms on C2; profiles/r2_ab_kernel_variants.txt) -- only the winners are instantiated, which also halves the build time.
  static int pairs = -1;
  if (pairs < 0) {
    const char *e = getenv("PERMON_B200_SD_PAIRS");   // measured on C2 / C3: one row per thread is 2-10 % faster (more warps in flight); pairs stay selectable
    pairs = (e && e[0] == '1') ? 1 : 0;
  }
  if (pairs && (A.n % 2 == 0) && aligned16(x) && epi.pair_ok()) {
    // two adjacent rows per thread, 16-byte accesses
    auto       k2 = k_spmv_sd2<Epi, LMAX, 4>;
    static int occ2 = 0;
    if (!occ2) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k2, NT, 0) != cudaSuccess || nb < 1) nb = 1;
      occ2 = nb;
    }
    const int ntiles = (A.n + TR - 1) / TR, nst = (ntiles + 1) / 2;
    int       grid = g_ctx.sm_count * occ2;
    if (grid > nst) grid = nst;
    if (grid > max_red_blocks()) grid = max_red_blocks();
    TileOrder o2;
    o2.ta = (ord.ta + 1) / 2;
    o2.tb = ord.tb / 2;
    if (o2.tb <= o2.ta || o2.tb > nst || ord.tb <= ord.ta || ord.tb > ntiles || (ord.ta == 0 && ord.tb == ntiles)) {
      o2.ta = 0;
      o2.tb = nst;
    }
    launch_k(k2, grid, NT, 0, A, x, epi, o2);
    return 0;
  }
  auto kern = k_spmv_sd<Epi, LMAX, 5>;
  static int pf = -1;
  if (pf < 0) {
    // L2 prefetch distance in grid sweeps.  OFF by default: measured on C2 / C3 (profiles/README.md, r2k) the bulk prefetches make K_A
    // 28-40 % SLOWER at every distance tried (1, 2, 4) -- kept as a switch for the record
    const char *e = getenv("PERMON_B200_SD_PF");
    pf = e ? atoi(e) : 0;
    if (pf < 0 || pf > 64) pf = 0;
  }
  ord.pf  = pf;
  ord.dlo = A.st_dlo;
  ord.dhi = A.st_dhi;
  static int occ = 0;
  if (!occ) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, NT, 0) != cudaSuccess || nb < 1) nb = 1;
    occ = nb;
  }
  int ntiles = (A.n + TR - 1) / TR, grid = g_ctx.sm_count * occ;
  if (grid > ntiles) grid = ntiles;
  if (grid > max_red_blocks()) grid = max_red_blocks();
  if (ord.tb <= ord.ta || ord.tb > ntiles) {
    ord.ta = 0;
    ord.tb = ntiles;
  }
  launch_k(kern, grid, NT, 0, A, x, epi, ord);
  return 0;
}
template <class Epi>
static int launch_sd(const CsrDev &A, const double *x, const Epi &epi, TileOrder ord)
{
  // the unrolled path is compiled for the pattern lengths of the common stencils; other lengths run the predicated loop (LMAX = 8 never
  // matches a shorter pattern, so every row takes the generic path)
  switch (A.st_lmax) {
  case 3: return launch_sd_l<Epi, 3>(A, x, epi, ord);
  case 5: return launch_sd_l<Epi, 5>(A, x, epi, ord);
  case 7: return launch_sd_l<Epi, 7>(A, x, epi, ord);
  default: return launch_sd_l<Epi, 8>(A, x, epi, ord);
  }
}

template <class Epi>
static int launch_spmv(const CsrDev &A, const double *x, const Epi &epi, int family, double bytes, TileOrder ord = TileOrder())
{
  prof_pre(family, bytes);
  if (A.n == 0) {
    // still run one CTA so that reductions publish their (identity) record
    k_spmv_vector<Epi, 32><<<1, NT, 0, g_ctx.stream>>>(A, x, epi);
  } else if (A.kind == 5) {
    launch_ell(A, x, epi);
  } else if (A.kind == 4) {
    static int direct = -1;
    if (direct < 0) {
      const char *e = getenv("PERMON_B200_ST_KERNEL");   // "direct" (default) | "windows"
      direct = (e && !strcmp(e, "windows")) ? 0 : 1;
    }
    if (direct) PB_CHK(launch_sd(A, x, epi, ord));
    else PB_CHK(launch_st(A, x, epi, ord));
  } else if (A.kind == 3) {
    PB_CHK(launch_pk(A, x, epi, ord));
  } else if (A.kind == 2) {
    launch_tma(A, x, epi);
  } else if (A.kind == 0) {
    static int    occ = 0;
    static size_t occ_smem = (size_t)-1;
    size_t        smem = (size_t)A.tile_cap * sizeof(double);
    if (!occ || occ_smem != smem) {
      occ      = occ_blocks(k_spmv_stream<Epi>, smem);
      occ_smem = smem;
    }
    int ntiles = (A.n + TR - 1) / TR;
    int grid   = g_ctx.sm_count * occ;
    if (grid > ntiles) grid = ntiles;
    if (grid > max_red_blocks()) grid = max_red_blocks();
    k_spmv_stream<Epi><<<grid, NT, smem, g_ctx.stream>>>(A, x, epi);
  } else {
    switch (A.W) {
    case 2: launch_vector<Epi, 2>(A, x, epi); break;
    case 4: launch_vector<Epi, 4>(A, x, epi); break;
    case 8: launch_vector<Epi, 8>(A, x, epi); break;
    case 16: launch_vector<Epi, 16>(A, x, epi); break;
    default: launch_vector<Epi, 32>(A, x, epi); break;
    }
  }
  prof_post(family);
  LAUNCH_CHECK();
  return 0;
}

double csr_stream_bytes(const CsrDev &A)
{
  if (A.kind == 3 || A.kind == 4) return (double)A.pk_bytes;
  if (A.kind == 5) return 12.0 * (double)A.ell_elems + 4.0 * A.n;
  return 12.0 * (double)A.nnz + 4.0 * (A.n + 1);
}

// decide the kernel flavour from the row pointer (host copy); the device re-coder computes the same statistics on the device
void spmv_stats(int n, const int *h_ia, int *maxrow_out, int *cap_out)
{
  int maxrow = 0, cap = 0;
  for (int r0 = 0; r0 < n; r0 += TR) {
    int r1 = (r0 + TR < n) ? r0 + TR : n;
    int t  = h_ia[r1] - h_ia[r0];
    if (t > cap) cap = t;
  }
#pragma omp parallel for reduction(max : maxrow) schedule(static)
  for (int r = 0; r < n; r++) {
    int l = h_ia[r + 1] - h_ia[r];
    if (l > maxrow) maxrow = l;
  }
  *maxrow_out = maxrow;
  *cap_out    = cap;
}
int spmv_config(CsrDev &A, const int *h_ia)
{
  int maxrow, cap;
  spmv_stats(A.n, h_ia, &maxrow, &cap);
  spmv_decide(A, maxrow, cap);
  return 0;
}
void spmv_decide(CsrDev &A, int maxrow, int cap)
{
  const int n = A.n;
  const double avg = n ? (double)A.nnz / n : 0.0;
  const char  *force = getenv("PERMON_B200_SPMV");   // "stream" | "vector" (A/B measurements)
  bool         stream = (cap <= 5632 && maxrow <= 64);   // <= 44 KB of products per tile
  if (force && !strcmp(force, "vector")) stream = false;
  if (stream) {
    A.kind     = 2;   // TMA-staged; "stream" forces the plain-load variant for A/B measurements
    if ((force && !strcmp(force, "stream")) || A.rows) A.kind = 0;
    A.tile_cap = (cap + 3 + 31) & ~31;   // +3: the tile copy starts at a 16-byte aligned element
    if (A.tile_cap < 32) A.tile_cap = 32;
    const char *st = getenv("PERMON_B200_STAGES");
    A.stages = st ? atoi(st) : 2;
  } else {
    A.kind = 1;
    int W  = 32;
    if (avg <= 3) W = 2;
    else if (avg <= 6) W = 4;
    else if (avg <= 12) W = 8;
    else if (avg <= 24) W = 16;
    A.W = W;
  }
}

// ---- epilogues ---------------------------------------------------------------------------------------
struct EpiPlain {
  typedef GatherPlain Gather;
  __device__ Gather gather(const double *x) const { return Gather{x}; }
  double *y;
  int     accumulate;
  struct Acc {};
  __device__ bool active() const { return true; }
  __device__ bool reverse() const { return false; }
  __device__ void init(Acc &) const {}
  __device__ void row(int r, double ax, Acc &) const { y[r] = accumulate ? y[r] + ax : ax; }
  struct Pre {};
  __device__ Pre preload(int) const { return Pre{}; }
  __device__ void row_p(int r, double ax, const Pre &, Acc &a) const { row(r, ax, a); }
  __device__ void finalize(Acc &) const {}
  __host__ __device__ int  nvec() const { return 0; }
  __host__ __device__ const double *vsrc(int) const { return nullptr; }
  int nvec_host() const { return nvec(); }
  const double *vsrc_host(int i) const { return vsrc(i); }
  __device__ void row_s(int r, uint32_t, double ax, Acc &a) const { row(r, ax, a); }

  struct Pre2 {};
  __device__ Pre2 preload2(int) const { return Pre2{}; }
  __device__ void row2_p(int r, double a0, double a1, const Pre2 &, Acc &a) const
  {
    row(r, a0, a);
    row(r + 1, a1, a);
  }
  bool pair_ok() const { return true; }
};

struct EpiGated {
  typedef GatherPlain Gather;
  __device__ Gather gather(const double *x) const { return Gather{x}; }   // plain SpMV that only runs in the right phase of the device-driven iteration
  double        *y;
  const MpgpCtl *S;
  int            phase;
  struct Acc {};
  __device__ bool active() const
  {
    if (S->reason != 0) return false;
    return phase == 0 ? true : (S->step == 'e' || S->init);
  }
  __device__ bool reverse() const { return false; }
  __device__ void init(Acc &) const {}
  __device__ void row(int r, double ax, Acc &) const { y[r] = ax; }
  struct Pre {};
  __device__ Pre preload(int) const { return Pre{}; }
  __device__ void row_p(int r, double ax, const Pre &, Acc &a) const { row(r, ax, a); }
  struct Pre2 {};
  __device__ Pre2 preload2(int) const { return Pre2{}; }
  __device__ void row2_p(int r, double a0, double a1, const Pre2 &, Acc &a) const
  {
    row(r, a0, a);
    row(r + 1, a1, a);
  }
  bool pair_ok() const { return true; }
  __device__ void finalize(Acc &) const {}
  __host__ __device__ int  nvec() const { return 0; }
  __host__ __device__ const double *vsrc(int) const { return nullptr; }
  int nvec_host() const { return nvec(); }
  const double *vsrc_host(int i) const { return vsrc(i); }
  __device__ void row_s(int r, uint32_t, double ax, Acc &a) const { row(r, ax, a); }
};

struct AccRed {
  double v[PB_NRED];
  int    halo_ok;   // this thread has seen every neighbour's halo flag (GhostMerge)
};

// off-diagonal part of row r (multi-GPU): MatMultAdd order, the ghost products are added one by one to the diagonal-block sum.
// Out of line: it runs for the few rows next to a partition boundary only and must not cost the streaming loop any registers.
struct GhostRet {
  double ax;
  int    ok;
};
__device__ __noinline__ GhostRet ghost_slow(const GhostMerge &gm, int r, double ax, int halo_ok)
{
  GhostRet  out{ax, halo_ok};
  const int k = __ldg(gm.row_map + (r < gm.lo ? r : r - gm.hi + gm.lo));
  if (k < 0) return out;
  if (!halo_ok) {
    for (int q = 0; q < gm.nflags; q++) wait_flag(gm.flags + (size_t)q * PB_FLAG_STRIDE, gm.seq);
    out.ok = 1;
  }
  const int e0 = __ldg(gm.oia + k), e1 = __ldg(gm.oia + k + 1);
  for (int e = e0; e < e1; e++) out.ax += __ldg(gm.oa + e) * __ldcg(gm.ghost + __ldg(gm.oja + e));
  return out;
}
__device__ __forceinline__ double ghost_apply(const GhostMerge &gm, int r, double ax, int &halo_ok)
{
  if (gm.row_map == nullptr || (r >= gm.lo && r < gm.hi)) return ax;
  const GhostRet g = ghost_slow(gm, r, ax, halo_ok);   // by value: the accumulators stay in registers
  halo_ok = g.ok;
  return g.ax;
}

// K_A epilogue: Ap_r = (A p)_r ; p.Ap ; B p ; max feasible step (QPCFeas).  (g.p comes from the kernel that wrote p, see mpgp_ctl.h.)
// MODE 1: lower bound only, no equality rows (the obstacle problems); MODE 2: lower and upper bound arrays, no equality rows
// (two-sided boxes, C5); MODE 0: anything.  In modes 1 and 2 the staged path sheds every run-time flag.
template <int MODE, bool GHOST>
struct EpiAT {
  typedef GatherPlain Gather;
  __device__ Gather gather(const double *x) const { return Gather{x}; }
  const double        *p, *x;
  double              *Ap;
  BoxDev               bx;
  const double        *B;
  int                  m, n;
  const MpgpCtl       *S;
  RedBuf               rb;
  GhostMerge           gm;
  typedef AccRed       Acc;
  __device__ bool active() const { return S->reason == 0; }
  __device__ bool reverse() const { return S->sweep != 0; }
  __device__ void init(Acc &a) const
  {
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) a.v[k] = 0.0;
    a.v[RA_FEAS] = HUGE_VAL;
    a.halo_ok    = 0;
  }
  __device__ void row(int r, double ax, Acc &a) const
  {
    if constexpr (GHOST) ax = ghost_apply(gm, r, ax, a.halo_ok);
    Ap[r] = ax;
    const double pr = __ldg(p + r);
    a.v[RA_PAP] += pr * ax;
    if constexpr (MODE != 0) {
      BoxVal b;
      b.has_lb = true;
      b.has_ub = (MODE == 2);
      b.lb     = __ldg(bx.lb + r);
      b.ub     = (MODE == 2) ? __ldg(bx.ub + r) : 0.0;
      a.v[RA_FEAS] = box_feas_lazy(__ldg(x + r), pr, b, a.v[RA_FEAS]);
    } else {
#pragma unroll
      for (int j = 0; j < PB_MAXEQ; j++)
        if (j < m) a.v[RA_BP + j] += B[(size_t)j * n + r] * pr;
      a.v[RA_FEAS] = box_feas_lazy(x[r], pr, load_box(bx, r), a.v[RA_FEAS]);
    }
  }
  // direct kernels: the row's epilogue operands are loaded BEFORE the gathers are consumed, so that a row costs one memory round trip
  struct Pre {
    double p, x, lb, ub;
  };
  __device__ Pre preload(int r) const
  {
    Pre q;
    q.p  = __ldg(p + r);
    q.x  = __ldg(x + r);
    q.lb = (MODE != 0 || bx.lb) ? __ldg(bx.lb + r) : 0.0;
    q.ub = (MODE == 2 || (MODE == 0 && bx.ub)) ? __ldg(bx.ub + r) : 0.0;
    return q;
  }
  __device__ void row_p(int r, double ax, const Pre &q, Acc &a) const
  {
    if constexpr (GHOST) ax = ghost_apply(gm, r, ax, a.halo_ok);
    Ap[r] = ax;
    a.v[RA_PAP] += q.p * ax;
    BoxVal b;
    b.has_lb = (MODE != 0) || bx.lb != nullptr;
    b.has_ub = (MODE == 2) || (MODE == 0 && bx.ub != nullptr);
    b.lb     = q.lb;
    b.ub     = q.ub;
    if constexpr (MODE == 0) {
#pragma unroll
      for (int j = 0; j < PB_MAXEQ; j++)
        if (j < m) a.v[RA_BP + j] += B[(size_t)j * n + r] * q.p;
    }
    a.v[RA_FEAS] = box_feas_lazy(q.x, q.p, b, a.v[RA_FEAS]);
  }
  struct Pre2 {
    double2 p, x, lb, ub;
  };
  __device__ Pre2 preload2(int r) const
  {
    Pre2 q;
    q.p  = __ldg(reinterpret_cast<const double2 *>(p + r));
    q.x  = __ldg(reinterpret_cast<const double2 *>(x + r));
    q.lb = (MODE != 0 || bx.lb) ? __ldg(reinterpret_cast<const double2 *>(bx.lb + r)) : make_double2(0.0, 0.0);
    q.ub = (MODE == 2 || (MODE == 0 && bx.ub)) ? __ldg(reinterpret_cast<const double2 *>(bx.ub + r)) : make_double2(0.0, 0.0);
    return q;
  }
  __device__ void row2_p(int r, double a0, double a1, const Pre2 &q, Acc &a) const
  {
    if constexpr (GHOST) {
      a0 = ghost_apply(gm, r, a0, a.halo_ok);
      a1 = ghost_apply(gm, r + 1, a1, a.halo_ok);
    }
    *reinterpret_cast<double2 *>(Ap + r) = make_double2(a0, a1);
    a.v[RA_PAP] += q.p.x * a0;
    a.v[RA_PAP] += q.p.y * a1;
    BoxVal b0, b1;
    b0.has_lb = b1.has_lb = (MODE != 0) || bx.lb != nullptr;
    b0.has_ub = b1.has_ub = (MODE == 2) || (MODE == 0 && bx.ub != nullptr);
    b0.lb = q.lb.x; b1.lb = q.lb.y;
    b0.ub = q.ub.x; b1.ub = q.ub.y;
    if constexpr (MODE == 0) {
#pragma unroll
      for (int j = 0; j < PB_MAXEQ; j++)
        if (j < m) {
          a.v[RA_BP + j] += B[(size_t)j * n + r] * q.p.x;
          a.v[RA_BP + j] += B[(size_t)j * n + r + 1] * q.p.y;
        }
    }
    a.v[RA_FEAS] = box_feas_lazy(q.x.x, q.p.x, b0, a.v[RA_FEAS]);
    a.v[RA_FEAS] = box_feas_lazy(q.x.y, q.p.y, b1, a.v[RA_FEAS]);
  }
  bool pair_ok() const { return aligned16(p) && aligned16(x) && aligned16(Ap) && aligned16(bx.lb) && aligned16(bx.ub); }
  __device__ void finalize(Acc &a) const { grid_reduce8<(1 << RA_FEAS)>(a.v, rb, nullptr); }
  // staged row vectors for the TMA kernels: p, x, [lb], [ub], [B_0..B_{m-1}]
  __host__ __device__ int nvec() const { return 2 + (bx.lb ? 1 : 0) + (bx.ub ? 1 : 0) + m; }
  int nvec_host() const { return nvec(); }
  const double *vsrc_host(int i) const { return vsrc(i); }
  __host__ __device__ const double *vsrc(int i) const
  {
    if (i == 0) return p;
    if (i == 1) return x;
    int k = 2;
    if (bx.lb) {
      if (i == k) return bx.lb;
      k++;
    }
    if (bx.ub) {
      if (i == k) return bx.ub;
      k++;
    }
    return B + (size_t)(i - k) * n;
  }
  // va: shared-memory address of this row's slot in the first staged vector; vector k sits k * TR * 8 bytes further
  __device__ void row_s(int r, uint32_t va, double ax, Acc &a) const
  {
    if constexpr (GHOST) ax = ghost_apply(gm, r, ax, a.halo_ok);
    Ap[r] = ax;
    const double pr = lds_f64(va);
    a.v[RA_PAP] += pr * ax;
    const double xr = lds_f64(va + TR * 8);
    if constexpr (MODE != 0) {
      BoxVal b;
      b.has_lb = true;
      b.has_ub = (MODE == 2);
      b.lb     = lds_f64(va + 2 * TR * 8);
      b.ub     = (MODE == 2) ? lds_f64(va + 3 * TR * 8) : 0.0;
      a.v[RA_FEAS] = box_feas_lazy(xr, pr, b, a.v[RA_FEAS]);
    } else {
      BoxVal   b;
      uint32_t k = 2;
      b.has_lb = bx.lb != nullptr;
      b.has_ub = bx.ub != nullptr;
      b.lb     = b.has_lb ? lds_f64(va + (k++) * TR * 8) : 0.0;
      b.ub     = b.has_ub ? lds_f64(va + (k++) * TR * 8) : 0.0;
#pragma unroll
      for (int j = 0; j < PB_MAXEQ; j++)
        if (j < m) a.v[RA_BP + j] += lds_f64(va + (k + j) * TR * 8) * pr;
      a.v[RA_FEAS] = box_feas_lazy(xr, pr, b, a.v[RA_FEAS]);
    }
  }
};

// K_A' epilogue: g_r = (A x)_r + rho (B^T Bu)_r - b_r ; split ; p = gf ; |gP|^2 |gc|^2 |gf|^2
template <int MODE, bool GHOST>
struct EpiA2T {
  typedef GatherPlain Gather;
  __device__ Gather gather(const double *x) const { return Gather{x}; }
  const double        *x, *b;
  double              *g, *p;
  BoxDev               bx;
  const double        *B;
  int                  m, n;
  const MpgpCtl       *S;
  RedBuf               rb;
  GhostMerge           gm;
  typedef AccRed       Acc;
  __device__ bool active() const { return S->reason == 0 && (S->step == 'e' || S->init); }
  __device__ bool reverse() const { return S->sweep != 0; }
  __device__ void init(Acc &a) const
  {
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) a.v[k] = 0.0;
    a.halo_ok = 0;
  }
  __device__ void row(int r, double ax, Acc &a) const
  {
    double gr = ax;
    if constexpr (GHOST) gr = ghost_apply(gm, r, ax, a.halo_ok);
    BoxVal bv;
    if constexpr (MODE != 0) {
      bv.has_lb = true;
      bv.has_ub = (MODE == 2);
      bv.lb     = __ldg(bx.lb + r);
      bv.ub     = (MODE == 2) ? __ldg(bx.ub + r) : 0.0;
    } else {
      bv = load_box(bx, r);
      if (m > 0) {
        double t = 0.0;
        for (int j = 0; j < m; j++) t += B[(size_t)j * n + r] * S->Bu[j];
        gr += S->rho * t;
      }
    }
    gr -= __ldg(b + r);
    double gf, gc;
    box_split(x[r], gr, bv, bx.astol, gf, gc);
    g[r] = gr;
    p[r] = gf;
    const double gP = gf + gc;
    a.v[RB_GP2] += gP * gP;
    a.v[RB_GC2] += gc * gc;
    a.v[RB_GF2] += gf * gf;
  }
  struct Pre {
    double x, b, lb, ub;
  };
  __device__ Pre preload(int r) const
  {
    Pre q;
    q.x  = __ldg(x + r);
    q.b  = __ldg(b + r);
    q.lb = (MODE != 0 || bx.lb) ? __ldg(bx.lb + r) : 0.0;
    q.ub = (MODE == 2 || (MODE == 0 && bx.ub)) ? __ldg(bx.ub + r) : 0.0;
    return q;
  }
  __device__ void row_p(int r, double ax, const Pre &q, Acc &a) const
  {
    double gr = ax;
    if constexpr (GHOST) gr = ghost_apply(gm, r, ax, a.halo_ok);
    BoxVal bv;
    bv.has_lb = (MODE != 0) || bx.lb != nullptr;
    bv.has_ub = (MODE == 2) || (MODE == 0 && bx.ub != nullptr);
    bv.lb     = q.lb;
    bv.ub     = q.ub;
    if constexpr (MODE == 0) {
      if (m > 0) {
        double t = 0.0;
        for (int j = 0; j < m; j++) t += B[(size_t)j * n + r] * S->Bu[j];
        gr += S->rho * t;
      }
    }
    gr -= q.b;
    double gf, gc;
    box_split(q.x, gr, bv, bx.astol, gf, gc);
    g[r] = gr;
    p[r] = gf;
    const double gP = gf + gc;
    a.v[RB_GP2] += gP * gP;
    a.v[RB_GC2] += gc * gc;
    a.v[RB_GF2] += gf * gf;
  }
  struct Pre2 {
    double2 x, b, lb, ub;
  };
  __device__ Pre2 preload2(int r) const
  {
    Pre2 q;
    q.x  = __ldg(reinterpret_cast<const double2 *>(x + r));
    q.b  = __ldg(reinterpret_cast<const double2 *>(b + r));
    q.lb = (MODE != 0 || bx.lb) ? __ldg(reinterpret_cast<const double2 *>(bx.lb + r)) : make_double2(0.0, 0.0);
    q.ub = (MODE == 2 || (MODE == 0 && bx.ub)) ? __ldg(reinterpret_cast<const double2 *>(bx.ub + r)) : make_double2(0.0, 0.0);
    return q;
  }
  __device__ void row2_p(int r, double a0, double a1, const Pre2 &q, Acc &a) const
  {
    double gr0 = a0, gr1 = a1;
    if constexpr (GHOST) {
      gr0 = ghost_apply(gm, r, a0, a.halo_ok);
      gr1 = ghost_apply(gm, r + 1, a1, a.halo_ok);
    }
    BoxVal b0, b1;
    b0.has_lb = b1.has_lb = (MODE != 0) || bx.lb != nullptr;
    b0.has_ub = b1.has_ub = (MODE == 2) || (MODE == 0 && bx.ub != nullptr);
    b0.lb = q.lb.x; b1.lb = q.lb.y;
    b0.ub = q.ub.x; b1.ub = q.ub.y;
    if constexpr (MODE == 0) {
      if (m > 0) {
        double t0 = 0.0, t1 = 0.0;
        for (int j = 0; j < m; j++) {
          t0 += B[(size_t)j * n + r] * S->Bu[j];
          t1 += B[(size_t)j * n + r + 1] * S->Bu[j];
        }
        gr0 += S->rho * t0;
        gr1 += S->rho * t1;
      }
    }
    gr0 -= q.b.x;
    gr1 -= q.b.y;
    double gf0, gc0, gf1, gc1;
    box_split(q.x.x, gr0, b0, bx.astol, gf0, gc0);
    box_split(q.x.y, gr1, b1, bx.astol, gf1, gc1);
    *reinterpret_cast<double2 *>(g + r) = make_double2(gr0, gr1);
    *reinterpret_cast<double2 *>(p + r) = make_double2(gf0, gf1);
    const double gP0 = gf0 + gc0, gP1 = gf1 + gc1;
    a.v[RB_GP2] += gP0 * gP0;
    a.v[RB_GC2] += gc0 * gc0;
    a.v[RB_GF2] += gf0 * gf0;
    a.v[RB_GP2] += gP1 * gP1;
    a.v[RB_GC2] += gc1 * gc1;
    a.v[RB_GF2] += gf1 * gf1;
  }
  bool pair_ok() const { return aligned16(x) && aligned16(b) && aligned16(g) && aligned16(p) && aligned16(bx.lb) && aligned16(bx.ub); }
  __device__ void finalize(Acc &a) const { grid_reduce8<0>(a.v, rb, nullptr); }
  // staged row vectors for the TMA kernels: x, b, [lb], [ub], [B_0..B_{m-1}]
  __host__ __device__ int nvec() const { return 2 + (bx.lb ? 1 : 0) + (bx.ub ? 1 : 0) + m; }
  int nvec_host() const { return nvec(); }
  const double *vsrc_host(int i) const { return vsrc(i); }
  __host__ __device__ const double *vsrc(int i) const
  {
    if (i == 0) return x;
    if (i == 1) return b;
    int k = 2;
    if (bx.lb) {
      if (i == k) return bx.lb;
      k++;
    }
    if (bx.ub) {
      if (i == k) return bx.ub;
      k++;
    }
    return B + (size_t)(i - k) * n;
  }
  __device__ void row_s(int r, uint32_t va, double ax, Acc &a) const
  {
    BoxVal bv;
    double gr = ax;
    if constexpr (GHOST) gr = ghost_apply(gm, r, ax, a.halo_ok);
    if constexpr (MODE != 0) {
      bv.has_lb = true;
      bv.has_ub = (MODE == 2);
      bv.lb     = lds_f64(va + 2 * TR * 8);
      bv.ub     = (MODE == 2) ? lds_f64(va + 3 * TR * 8) : 0.0;
    } else {
      uint32_t k = 2;
      bv.has_lb = bx.lb != nullptr;
      bv.has_ub = bx.ub != nullptr;
      bv.lb     = bv.has_lb ? lds_f64(va + (k++) * TR * 8) : 0.0;
      bv.ub     = bv.has_ub ? lds_f64(va + (k++) * TR * 8) : 0.0;
      if (m > 0) {
        double tt = 0.0;
#pragma unroll
        for (int j = 0; j < PB_MAXEQ; j++)
          if (j < m) tt += lds_f64(va + (k + j) * TR * 8) * S->Bu[j];
        gr += S->rho * tt;
      }
    }
    gr -= lds_f64(va + TR * 8);
    double gf, gc;
    box_split(lds_f64(va), gr, bv, bx.astol, gf, gc);
    g[r] = gr;
    p[r] = gf;
    const double gP = gf + gc;
    a.v[RB_GP2] += gP * gP;
    a.v[RB_GC2] += gc * gc;
    a.v[RB_GF2] += gf * gf;
  }
};

// power-method step (MatGetMaxEigenvalue, permonmatutils.c:484-511) in ONE pass: the normalised iterate v = s * w is formed on the
// fly (the same product VecScale would have stored), y = A v, and the two dot products of VecMDot(v, {Av, v}) ride in the epilogue
struct EpiPower {
  typedef GatherScaled Gather;
  const double *w;
  double        s;
  double       *y;
  RedBuf        rb;
  __device__ Gather gather(const double *x) const { return Gather{x, s}; }
  typedef AccRed Acc;
  __device__ bool active() const { return true; }
  __device__ bool reverse() const { return false; }
  __device__ void init(Acc &a) const
  {
#pragma unroll
    for (int k = 0; k < PB_NRED; k++) a.v[k] = 0.0;
    a.halo_ok = 0;
  }
  __device__ void row(int r, double ax, Acc &a) const
  {
    y[r] = ax;
    const double vr = w[r] * s;
    a.v[0] += ax * vr;
    a.v[1] += vr * vr;
  }
  struct Pre {
    double w;
  };
  __device__ Pre preload(int r) const { return Pre{__ldg(w + r)}; }
  __device__ void row_p(int r, double ax, const Pre &q, Acc &a) const
  {
    y[r] = ax;
    const double vr = q.w * s;
    a.v[0] += ax * vr;
    a.v[1] += vr * vr;
  }
  struct Pre2 {
    double2 w;
  };
  __device__ Pre2 preload2(int r) const { return Pre2{__ldg(reinterpret_cast<const double2 *>(w + r))}; }
  __device__ void row2_p(int r, double a0, double a1, const Pre2 &q, Acc &a) const
  {
    *reinterpret_cast<double2 *>(y + r) = make_double2(a0, a1);
    const double v0 = q.w.x * s, v1 = q.w.y * s;
    a.v[0] += a0 * v0;
    a.v[1] += v0 * v0;
    a.v[0] += a1 * v1;
    a.v[1] += v1 * v1;
  }
  bool pair_ok() const { return aligned16(w) && aligned16(y); }
  __device__ void finalize(Acc &a) const { grid_reduce8<0>(a.v, rb, nullptr); }
  __host__ __device__ int nvec() const { return 1; }
  __host__ __device__ const double *vsrc(int) const { return w; }
  int nvec_host() const { return 1; }
  const double *vsrc_host(int) const { return w; }
  __device__ void row_s(int r, uint32_t va, double ax, Acc &a) const
  {
    y[r] = ax;
    const double vr = lds_f64(va) * s;
    a.v[0] += ax * vr;
    a.v[1] += vr * vr;
  }
};
int k_power_step(const CsrDev &A, const double *w, double s, double *y, RedBuf rb)
{
  if (A.kind != 3 && A.kind != 4) {
    set_error("internal: fused power step needs a packed matrix");
    return 76;
  }
  EpiPower e{w, s, y, rb};
  return launch_spmv(A, w, e, KF_SPMV_PLAIN, csr_stream_bytes(A) + 16.0 * A.n);
}

int k_spmv(const CsrDev &A, const double *x, double *y, int accumulate)
{
  EpiPlain e{y, accumulate};
  return launch_spmv(A, x, e, KF_SPMV_PLAIN, csr_stream_bytes(A) + 16.0 * A.n);
}

int k_spmv_gated(const CsrDev &A, const double *x, double *y, const MpgpCtl *S, int phase)
{
  EpiGated e{y, S, phase};
  return launch_spmv(A, x, e, KF_SPMV_PLAIN, csr_stream_bytes(A) + 16.0 * A.n);
}

static double bytes_A(const CsrDev &A, const MpgpVecs &v)
{   // matrix + p (gather; its row slice comes from the same lines) + x + lb[+ub] + B rows, write Ap
  return csr_stream_bytes(A) + 8.0 * v.n * (3 + (v.bx.lb ? 1 : 0) + (v.bx.ub ? 1 : 0) + v.m);
}
static double bytes_A2(const CsrDev &A, const MpgpVecs &v)
{   // matrix + x (gather) + b + lb[+ub] + B rows, write g, p
  return csr_stream_bytes(A) + 8.0 * v.n * (4 + (v.bx.lb ? 1 : 0) + (v.bx.ub ? 1 : 0) + v.m);
}
// tiles that lie entirely inside the rows without ghost columns go first (multi-GPU); otherwise index order
static TileOrder tile_order(const CsrDev &A, const GhostMerge &gm)
{
  TileOrder o;
  const int ntiles = (A.n + TR - 1) / TR;
  o.ta = 0;
  o.tb = ntiles;
  if (gm.row_map) {
    int ta = (gm.lo + TR - 1) / TR, tb = gm.hi / TR;
    if (tb > ta) {
      o.ta = ta;
      o.tb = tb;
    }
  }
  return o;
}

template <int MODE, bool GHOST>
static int fused_A_t(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm, TileOrder ord)
{
  EpiAT<MODE, GHOST> e{v.p, v.x, v.Ap, v.bx, v.B, v.m, v.n, S, rb, gm};
  return launch_spmv(A, xin, e, KF_SPMV_A, bytes_A(A, v), ord);
}
template <int MODE, bool GHOST>
static int fused_A2_t(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm, TileOrder ord)
{
  EpiA2T<MODE, GHOST> e{v.x, v.b, v.g, v.p, v.bx, v.B, v.m, v.n, S, rb, gm};
  return launch_spmv(A, xin, e, KF_SPMV_A2, bytes_A2(A, v), ord);
}
// MODE: 1 lower bound only, 2 both bounds (no equality rows), 0 anything; the ghost-column code exists only in the multi-GPU instantiations
static int box_mode(const MpgpVecs &v) { return (v.m == 0 && v.bx.lb) ? (v.bx.ub ? 2 : 1) : 0; }

int k_fused_A(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm)
{
  const TileOrder ord = tile_order(A, gm);
  const int       mode = box_mode(v);
  if (gm.row_map) {
    if (mode == 1) return fused_A_t<1, true>(A, xin, v, S, rb, gm, ord);
    if (mode == 2) return fused_A_t<2, true>(A, xin, v, S, rb, gm, ord);
    return fused_A_t<0, true>(A, xin, v, S, rb, gm, ord);
  }
  if (mode == 1) return fused_A_t<1, false>(A, xin, v, S, rb, gm, ord);
  if (mode == 2) return fused_A_t<2, false>(A, xin, v, S, rb, gm, ord);
  return fused_A_t<0, false>(A, xin, v, S, rb, gm, ord);
}

int k_fused_A2(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm)
{
  const TileOrder ord = tile_order(A, gm);
  const int       mode = box_mode(v);
  if (gm.row_map) {
    if (mode == 1) return fused_A2_t<1, true>(A, xin, v, S, rb, gm, ord);
    if (mode == 2) return fused_A2_t<2, true>(A, xin, v, S, rb, gm, ord);
    return fused_A2_t<0, true>(A, xin, v, S, rb, gm, ord);
  }
  if (mode == 1) return fused_A2_t<1, false>(A, xin, v, S, rb, gm, ord);
  if (mode == 2) return fused_A2_t<2, false>(A, xin, v, S, rb, gm, ord);
  return fused_A2_t<0, false>(A, xin, v, S, rb, gm, ord);
}

// peer-memory halo push: dst_q[k] = vec[send_idx[k]] written straight into the neighbours' ghost buffers, then a
// sequence flag per neighbour once every CTA's stores are fenced (threadfence + ticket, last CTA signals)
__global__ void __launch_bounds__(NT) k_halo_push_kernel(HaloPush hp, const double *__restrict__ vec, int gated, unsigned long long seq, const MpgpCtl *__restrict__ S)
{
  if (S) {
    if (S->reason != 0) return;
    if (gated && !(S->step == 'e' || S->init)) return;
  }
  __shared__ int s_last;
  const int      stride = gridDim.x * NT;
  for (int k = blockIdx.x * NT + threadIdx.x; k < hp.total; k += stride) {
    int q = 0;
    while (q + 1 < hp.nneigh && k >= hp.send_off[q + 1]) q++;
    hp.dst[q][k - hp.send_off[q]] = vec[hp.send_idx[k]];
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = atomicAdd(hp.counter, 1u);
    s_last     = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence_system();
    if ((int)threadIdx.x < hp.nneigh) *(volatile unsigned long long *)hp.flag[threadIdx.x] = seq;
    if (threadIdx.x == 0) *hp.counter = 0u;
  }
}
int k_halo_push(const HaloPush &hp, const double *vec, int gated, unsigned long long seq, const MpgpCtl *S)
{
  int grid = (hp.total + NT - 1) / NT;
  if (grid < 1) grid = 1;
  if (grid > g_ctx.sm_count * 2) grid = g_ctx.sm_count * 2;
  prof_pre(KF_HALO, 20.0 * hp.total);
  k_halo_push_kernel<<<grid, NT, 0, g_ctx.stream>>>(hp, vec, gated, seq, S);
  prof_post(KF_HALO);
  LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// K_B: fused step  (mpgp.c:553-555 CG, :633-638 proportioning, :316-321 expansion std/fixed)
// =====================================================================================================
// control-step prologues, kept out of line so that their register needs do not set the budget of the streaming loops
__device__ __noinline__ void fold_ctrl_A(const CtrlFold &cf, MpgpCtl *sS)
{
  *sS = *cf.Sin;
  mpgp_ctrl_A(sS, cf.rec0);
  if (blockIdx.x == 0) *cf.Sout = *sS;
}
__device__ __noinline__ void fold_ctrl_B(const CtrlFold &cf, MpgpCtl *sS, bool second)
{
  *sS = *cf.Sin;
  mpgp_ctrl_B(sS, second ? cf.rec1 : cf.rec0);
  if (blockIdx.x == 0) *cf.Sout = *sS;
}

// fused halo push helpers: the thread that produces a boundary value also stores it into the neighbours' ghost windows
__device__ __forceinline__ void push_boundary(const PushRanges *hp, int r, double val)
{
  const int n = hp->n;
  for (int q = 0; q < n; q++) {
    const int lo = hp->lo[q];
    if (r >= lo && r < hp->hi[q]) hp->dst[q][r - lo] = val;
  }
}
// rows in [gap_lo, gap_hi) belong to no send range (the interior of the block): two register compares per element keep the
// fused push off the hot loop
// after all CTAs fenced their peer stores, the last one raises the neighbours' flags (called by every thread of every CTA)
__device__ __forceinline__ void push_signal(const PushRanges *hp, unsigned long long seq, int *s_last)
{
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = atomicAdd(hp->counter, 1u);
    *s_last    = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (*s_last) {
    __threadfence_system();
    if ((int)threadIdx.x < hp->n) *(volatile unsigned long long *)hp->flag[threadIdx.x] = seq;
    if (threadIdx.x == 0) *hp->counter = 0u;
  }
}

// one element of the c / p update (mpgp.c:553-558 CG, :633-638 proportioning)
template <bool EQ>
__device__ __forceinline__ void update_cp_elem(int step, double acg, double astol, double xr, double pr, double g0, double apr, const BoxVal &b, const double *brow, int m,
                                               double &xn, double &gn, double &gf, double *acc)
{
  double gc;
  xn = xr - acg * pr;
  gn = g0 - acg * apr;
  box_split(xn, gn, b, astol, gf, gc);
  if (step == 'c') acc[RB_APGF] += apr * gf;
  const double gP = gf + gc;
  acc[RB_GP2] += gP * gP;
  acc[RB_GC2] += gc * gc;
  acc[RB_GF2] += gf * gf;
  if (EQ) {
#pragma unroll
    for (int j = 0; j < PB_MAXEQ; j++)
      if (j < m) acc[RB_BU + j] += brow[j] * xn;
  }
}
// one element of the expansion half step + reduced-gradient step (mpgp.c:316-321, std / fixed length)
template <bool EQ>
__device__ __forceinline__ double update_e_elem(double afeas, double alpha, double astol, double xr, double pr, double g0, double apr, const BoxVal &b, const double *brow, int m,
                                                double *acc)
{
  const double xh = xr - afeas * pr;
  const double gh = g0 - afeas * apr;
  double       gf, gc;
  box_split(xh, gh, b, astol, gf, gc);
  const double grd = box_reduced(xh, gf, b, alpha);
  const double xn  = xh - alpha * grd;
  if (EQ) {
#pragma unroll
    for (int j = 0; j < PB_MAXEQ; j++)
      if (j < m) acc[RB_BU + j] += brow[j] * xn;
  }
  return xn;
}
template <bool EQ>
__device__ __forceinline__ double penal_apr(double apr, double rho, const double *B, int n, int r, int m, const double *bp, double *brow)
{   // A_rho p = A p + rho B^T (B p)   (matpenalized.c:12-22)
  if (!EQ) return apr;
  double t = 0.0;
#pragma unroll
  for (int j = 0; j < PB_MAXEQ; j++) {
    brow[j] = (j < m) ? B[(size_t)j * n + r] : 0.0;
    t += brow[j] * bp[j];
  }
  return apr + rho * t;
}

// K_B.  EQ: equality rows present (SMALXE inner solve).  VEC2: 16-byte accesses (n even, pointers 16-byte aligned).
template <bool EQ, bool VEC2, bool PUSH>
__global__ void __launch_bounds__(NT, EQ ? 3 : 4) k_update_B(MpgpVecs v, CtrlFold cf, RedBuf rb, const PushRanges *__restrict__ hp, unsigned long long push_seq)
{
  __shared__ MpgpCtl sS;
  __shared__ int     s_plast;
  pdl_enter();
  const MpgpCtl     *S = cf.Sin;
  if (cf.fold) {   // ctrl_A in the prologue: step selection from the K_A records (mpgp.c:541-547,617-621)
    if (cf.Sin->reason != 0) {
      if (blockIdx.x == 0 && threadIdx.x == 0) *cf.Sout = *cf.Sin;   // hand the stop on to K_A' / K_C
      return;
    }
    if (cf.flags0) {
      if ((int)threadIdx.x < cf.size) wait_flag(cf.flags0 + (size_t)threadIdx.x * PB_FLAG_STRIDE, cf.seq0);
      __syncthreads();
    }
    if (threadIdx.x == 0) fold_ctrl_A(cf, &sS);
    __syncthreads();
    S = &sS;
  } else if (S->reason != 0) {
    return;
  }
  const int    step = S->step;
  const bool   pushx = PUSH && (step == 'e');
  const double acg = S->acg, afeas = S->afeas, alpha = S->alpha, rho = S->rho, astol = v.bx.astol;
  const int    m = v.m, n = v.n;
  double       bp[PB_MAXEQ] = {0.0, 0.0, 0.0, 0.0};
  if (EQ) {
#pragma unroll
    for (int j = 0; j < PB_MAXEQ; j++) bp[j] = (j < m) ? S->Bp[j] : 0.0;
  }
  double acc[PB_NRED];
#pragma unroll
  for (int k = 0; k < PB_NRED; k++) acc[k] = 0.0;
  const bool has_lb = v.bx.lb != nullptr, has_ub = v.bx.ub != nullptr;
  const int  stride = gridDim.x * NT;
  // serpentine sweeps: K_B walks the rows against the direction K_A just used, so that the tail of K_A's stream (the last
  // Ap / p / x / lb lines it touched) is still in L2 when K_B starts there
  const bool rev = S->serp && (S->sweep == 0);

  if (VEC2) {
    const int      n2 = n >> 1;
    const double2 *x2 = reinterpret_cast<const double2 *>(v.x), *p2 = reinterpret_cast<const double2 *>(v.p), *g2 = reinterpret_cast<const double2 *>(v.g),
                  *A2 = reinterpret_cast<const double2 *>(v.Ap), *l2 = reinterpret_cast<const double2 *>(v.bx.lb), *u2 = reinterpret_cast<const double2 *>(v.bx.ub);
    double2 *xo = reinterpret_cast<double2 *>(v.x), *go = reinterpret_cast<double2 *>(v.g), *po = reinterpret_cast<double2 *>(v.p);
    int glo = INT_MAX, ghi = INT_MAX;
    if (PUSH && pushx) {
      glo = hp->gap_lo;
      ghi = hp->gap_hi;
    }
    for (int i0 = blockIdx.x * NT + threadIdx.x; i0 < n2; i0 += stride) {
      const int     i = rev ? n2 - 1 - i0 : i0;
      const double2 xr = x2[i], pr = p2[i], g0 = g2[i], ap = A2[i];
      BoxVal        b0, b1;
      b0.has_lb = b1.has_lb = has_lb;
      b0.has_ub = b1.has_ub = has_ub;
      b0.lb = b1.lb = b0.ub = b1.ub = 0.0;
      if (has_lb) {
        const double2 t = l2[i];
        b0.lb = t.x;
        b1.lb = t.y;
      }
      if (has_ub) {
        const double2 t = u2[i];
        b0.ub = t.x;
        b1.ub = t.y;
      }
      double br0[PB_MAXEQ], br1[PB_MAXEQ];
      const double a0 = penal_apr<EQ>(ap.x, rho, v.B, n, 2 * i, m, bp, br0);
      const double a1 = penal_apr<EQ>(ap.y, rho, v.B, n, 2 * i + 1, m, bp, br1);
      if (step == 'e') {
        double2 xn;
        xn.x  = update_e_elem<EQ>(afeas, alpha, astol, xr.x, pr.x, g0.x, a0, b0, br0, m, acc);
        xn.y  = update_e_elem<EQ>(afeas, alpha, astol, xr.y, pr.y, g0.y, a1, b1, br1, m, acc);
        xo[i] = xn;
        if (PUSH && (2 * i < glo || 2 * i + 1 >= ghi)) {
          push_boundary(hp, 2 * i, xn.x);
          push_boundary(hp, 2 * i + 1, xn.y);
        }
      } else {
        double2 xn, gn, gf;
        update_cp_elem<EQ>(step, acg, astol, xr.x, pr.x, g0.x, a0, b0, br0, m, xn.x, gn.x, gf.x, acc);
        update_cp_elem<EQ>(step, acg, astol, xr.y, pr.y, g0.y, a1, b1, br1, m, xn.y, gn.y, gf.y, acc);
        xo[i] = xn;
        go[i] = gn;
        if (step == 'c') {             // mpgp.c:555: gf is needed once more, by the direction update: K_C rebuilds it from g
          uchar2 am;                   // and this byte mask (gf = active ? 0 : g), 1/8 of the bytes of writing gf itself
          am.x = gf_differs(gf.x, gn.x);
          am.y = gf_differs(gf.y, gn.y);
          reinterpret_cast<uchar2 *>(v.gf)[i] = am;
        } else {
          po[i] = gf;                  // mpgp.c:638: p = gf
        }
      }
    }
  } else {
    int glo = INT_MAX, ghi = INT_MAX;
    if (PUSH && pushx) {
      glo = hp->gap_lo;
      ghi = hp->gap_hi;
    }
    for (int r0 = blockIdx.x * NT + threadIdx.x; r0 < n; r0 += stride) {
      const int    r = rev ? n - 1 - r0 : r0;
      const double xr = v.x[r], pr = v.p[r], g0 = v.g[r];
      double       brow[PB_MAXEQ];
      const double apr = penal_apr<EQ>(v.Ap[r], rho, v.B, n, r, m, bp, brow);
      const BoxVal b = load_box(v.bx, r);
      if (step == 'e') {
        const double xn = update_e_elem<EQ>(afeas, alpha, astol, xr, pr, g0, apr, b, brow, m, acc);
        v.x[r]          = xn;
        if (PUSH && (r < glo || r >= ghi)) push_boundary(hp, r, xn);
      } else {
        double xn, gn, gf;
        update_cp_elem<EQ>(step, acg, astol, xr, pr, g0, apr, b, brow, m, xn, gn, gf, acc);
        v.x[r] = xn;
        v.g[r] = gn;
        if (step == 'c') reinterpret_cast<unsigned char *>(v.gf)[r] = gf_differs(gf, gn);
        else v.p[r] = gf;
      }
    }
  }
  grid_reduce8<0>(acc, rb, nullptr);
  if (PUSH && pushx) push_signal(hp, push_seq, &s_plast);
}

template <bool EQ, bool VEC2>
static void launch_B(int grid, const MpgpVecs &v, const CtrlFold &cf, RedBuf rb, const PushRanges *hp, unsigned long long seq)
{
  if (hp) launch_k(k_update_B<EQ, VEC2, true>, grid, NT, 0, v, cf, rb, hp, seq);
  else launch_k(k_update_B<EQ, VEC2, false>, grid, NT, 0, v, cf, rb, (const PushRanges *)nullptr, 0ull);
}
int k_fused_B(const MpgpVecs &v, const CtrlFold &cf, RedBuf rb, const PushRanges *hp, unsigned long long push_seq)
{
  const bool vec2 = (v.n % 2 == 0) && aligned16(v.x) && aligned16(v.p) && aligned16(v.g) && aligned16(v.Ap) && aligned16(v.gf) && aligned16(v.bx.lb) && aligned16(v.bx.ub) &&
                    !getenv("PERMON_B200_NOVEC");
  // one resident wave: K_B holds 64 registers per thread (4 CTAs / SM, 3 with equality rows), so the generic 8-per-SM grid would run as two
  // waves -- the prologue (step selection), the block reduction and the ticket would be paid twice per SM slot
  static int occ_b[2] = {0, 0};
  const int  eqi = v.m > 0 ? 1 : 0;
  if (!occ_b[eqi]) {
    int nb = 0;
    cudaError_t e = (eqi ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_update_B<true, true, false>, NT, 0)
                         : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_update_B<false, true, false>, NT, 0));
    occ_b[eqi] = (e == cudaSuccess && nb >= 1) ? nb : 4;
    if (getenv("PERMON_B200_KB_TWO_WAVES")) occ_b[eqi] = 8;   // A/B: the former grid
  }
  int        grid = g_ctx.sm_count * occ_b[eqi];
  int        need = ((vec2 ? v.n / 2 : v.n) + NT - 1) / NT;
  if (need < 1) need = 1;
  if (grid > need) grid = need;
  // x p g Ap lb[ub] read, x g + the gf byte mask written (CG step)
  prof_pre(KF_UPDATE_B, 8.0 * v.n * (6.125 + (v.bx.lb ? 1 : 0) + (v.bx.ub ? 1 : 0) + v.m));
  if (v.m > 0) {
    if (vec2) launch_B<true, true>(grid, v, cf, rb, hp, push_seq);
    else launch_B<true, false>(grid, v, cf, rb, hp, push_seq);
  } else {
    if (vec2) launch_B<false, true>(grid, v, cf, rb, hp, push_seq);
    else launch_B<false, false>(grid, v, cf, rb, hp, push_seq);
  }
  prof_post(KF_UPDATE_B);
  LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// K_C: direction update  (mpgp.c:560 p = gf - bcg p ; :623 p = gc)
// =====================================================================================================
template <bool PUSH>
__global__ void __launch_bounds__(NT, 8) k_direction_C(MpgpVecs v, CtrlFold cf, RedBuf rc, const PushRanges *__restrict__ hp, unsigned long long push_seq, int vec2)
{
  __shared__ MpgpCtl sS;
  __shared__ int     s_plast;
  pdl_enter();
  const MpgpCtl     *S = cf.Sin;
  if (cf.fold) {   // ctrl_B in the prologue: norms, stopping test, beta, next step kind (mpgp.c:514-535,558-559)
    if (cf.Sin->reason != 0) return;
    const bool                second = (cf.Sin->step == 'e' || cf.Sin->init);   // record of K_A' or of K_B
    const unsigned long long *fl = second ? cf.flags1 : cf.flags0;
    if (fl) {
      if ((int)threadIdx.x < cf.size) wait_flag(fl + (size_t)threadIdx.x * PB_FLAG_STRIDE, second ? cf.seq1 : cf.seq0);
      __syncthreads();
    }
    if (threadIdx.x == 0) fold_ctrl_B(cf, &sS, second);
    __syncthreads();
    S = &sS;
  }
  if (S->reason != 0) return;
  const int    pmode = S->pmode;
  const double bcg = S->bcg, astol = v.bx.astol;
  const int    stride = gridDim.x * NT;
  const bool   rev = S->serp && (S->sweep == 0);   // the direction of this iteration's K_A (ctrl_B has already flipped `sweep`)
  if (pmode == 1) {
    double gp = 0.0;   // g.p of the new direction (mpgp.c:541 of the coming iteration): K_A's record carries it
    if (vec2) {
      const double2 *g2 = reinterpret_cast<const double2 *>(v.g);
      const uchar2  *a2 = reinterpret_cast<const uchar2 *>(v.gf);   // K_B's byte mask lives in the gf array
      double2       *p2 = reinterpret_cast<double2 *>(v.p);
      const int      n2 = v.n >> 1;
      int            glo = INT_MAX, ghi = INT_MAX;
      if (PUSH) {
        glo = hp->gap_lo;
        ghi = hp->gap_hi;
      }
      for (int i0 = blockIdx.x * NT + threadIdx.x; i0 < n2; i0 += stride) {
        const int     i = rev ? n2 - 1 - i0 : i0;
        const double2 gg = g2[i], q = p2[i];
        const uchar2  am = a2[i];
        double2       pn;
        pn.x  = (am.x ? 0.0 : gg.x) - bcg * q.x;
        pn.y  = (am.y ? 0.0 : gg.y) - bcg * q.y;
        p2[i] = pn;
        gp += gg.x * pn.x;
        gp += gg.y * pn.y;
        if (PUSH && (2 * i < glo || 2 * i + 1 >= ghi)) {
          push_boundary(hp, 2 * i, pn.x);
          push_boundary(hp, 2 * i + 1, pn.y);
        }
      }
    } else {
      for (int r0 = blockIdx.x * NT + threadIdx.x; r0 < v.n; r0 += stride) {
        const int    r = rev ? v.n - 1 - r0 : r0;
        const double gg = v.g[r];
        const double pn = (reinterpret_cast<const unsigned char *>(v.gf)[r] ? 0.0 : gg) - bcg * v.p[r];
        v.p[r]          = pn;
        gp += gg * pn;
        if (PUSH) push_boundary(hp, r, pn);
      }
    }
    block_partial1(gp, rc.partials);
  } else if (pmode == 2) {
    for (int r = blockIdx.x * NT + threadIdx.x; r < v.n; r += stride) {
      double gf, gc;
      box_split(v.x[r], v.g[r], load_box(v.bx, r), astol, gf, gc);
      v.p[r] = gc;
      if (PUSH) push_boundary(hp, r, gc);
    }
  } else if (PUSH) {   // p is already final (written by K_B or K_A'): only the boundary values travel
    const int nq = hp->n;
    for (int q = 0; q < nq; q++) {
      const int lo = hp->lo[q], hi = hp->hi[q];
      double   *dst = hp->dst[q];
      for (int r = lo + blockIdx.x * NT + threadIdx.x; r < hi; r += stride) dst[r - lo] = v.p[r];
    }
  }
  if (PUSH) push_signal(hp, push_seq, &s_plast);
}

int fused_C_grid(int n)
{
  int grid = elementwise_grid();
  int need = (n + NT - 1) / NT;
  if (need < 1) need = 1;
  return grid > need ? need : grid;
}
int k_fused_C(const MpgpVecs &v, const CtrlFold &cf, RedBuf rc, const PushRanges *hp, unsigned long long push_seq)
{
  const int grid = fused_C_grid(v.n);
  const int vec2 = (v.n % 2 == 0) && aligned16(v.gf) && aligned16(v.g) && aligned16(v.p) && !getenv("PERMON_B200_NOVEC");
  prof_pre(KF_DIR_C, 8.0 * v.n * 3.125);
  if (hp) launch_k(k_direction_C<true>, grid, NT, 0, v, cf, rc, hp, push_seq, vec2);
  else launch_k(k_direction_C<false>, grid, NT, 0, v, cf, rc, (const PushRanges *)nullptr, 0ull, vec2);
  prof_post(KF_DIR_C);
  LAUNCH_CHECK();
  return 0;
}

// initial projection x = P(x) (mpgp.c:497) + B u of the projected iterate
__global__ void __launch_bounds__(NT) k_project_init(MpgpVecs v, const MpgpCtl *__restrict__ S, RedBuf rb)
{
  pdl_enter();
  if (S->reason != 0) return;
  double acc[PB_NRED];
#pragma unroll
  for (int k = 0; k < PB_NRED; k++) acc[k] = 0.0;
  const int stride = gridDim.x * NT;
  for (int r = blockIdx.x * NT + threadIdx.x; r < v.n; r += stride) {
    const double xn = box_project(v.x[r], load_box(v.bx, r));
    v.x[r]          = xn;
    for (int j = 0; j < v.m; j++) acc[RB_BU + j] += v.B[(size_t)j * v.n + r] * xn;
  }
  grid_reduce8<0>(acc, rb, nullptr);
}

int k_fused_project(const MpgpVecs &v, const MpgpCtl *S, RedBuf rb)
{
  int grid = elementwise_grid();
  int need = (v.n + NT - 1) / NT;
  if (need < 1) need = 1;
  if (grid > need) grid = need;
  prof_pre(KF_QPC, 8.0 * v.n * 3);
  k_project_init<<<grid, NT, 0, g_ctx.stream>>>(v, S, rb);
  prof_post(KF_QPC);
  LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// ctrl kernels
// =====================================================================================================
__global__ void k_ctrl_A_kernel(MpgpCtl *S, const double *ra) { mpgp_ctrl_A(S, ra); }
__global__ void k_ctrl_E_kernel(MpgpCtl *S, const double *rb) { mpgp_ctrl_E(S, rb); }
__global__ void k_ctrl_B_kernel(MpgpCtl *S, const double *rb) { mpgp_ctrl_B(S, rb); }

// peer-memory variants: one warp; lane q waits for rank q's record, lane 0 then runs the control step
__global__ void k_ctrl_A_p2p_kernel(MpgpCtl *S, int size, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq)
{
  if (S->reason != 0) return;
  if ((int)threadIdx.x < size) wait_flag(my_flag + p2p_flag_index(0, threadIdx.x), seq);
  __syncwarp();
  if (threadIdx.x == 0) mpgp_ctrl_A(S, my_slot + p2p_slot_index(0, seq, 0));
}
__global__ void k_ctrl_E_p2p_kernel(MpgpCtl *S, int size, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq)
{
  if (S->reason != 0) return;
  if (!(S->step == 'e' || S->init)) return;
  if ((int)threadIdx.x < size) wait_flag(my_flag + p2p_flag_index(1, threadIdx.x), seq);
  __syncwarp();
  if (threadIdx.x == 0) mpgp_ctrl_E(S, my_slot + p2p_slot_index(1, seq, 0));
}
__global__ void k_ctrl_B_p2p_kernel(MpgpCtl *S, int size, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq1, unsigned long long seq2)
{
  if (S->reason != 0) return;
  const bool second = (S->step == 'e' || S->init);   // the record comes from K_A' (kind 2) or from K_B (kind 1)
  const int  kind = second ? 2 : 1;
  const unsigned long long seq = second ? seq2 : seq1;
  if ((int)threadIdx.x < size) wait_flag(my_flag + p2p_flag_index(kind, threadIdx.x), seq);
  __syncwarp();
  if (threadIdx.x == 0) mpgp_ctrl_B(S, my_slot + p2p_slot_index(kind, seq, 0));
}
int k_ctrl_A_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq)
{
  (void)win;
  prof_pre(KF_CTRL, 0);
  k_ctrl_A_p2p_kernel<<<1, 32, 0, g_ctx.stream>>>(S, g_p2p_size, my_slot, my_flag, seq);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}
int k_ctrl_E_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq)
{
  (void)win;
  prof_pre(KF_CTRL, 0);
  k_ctrl_E_p2p_kernel<<<1, 32, 0, g_ctx.stream>>>(S, g_p2p_size, my_slot, my_flag, seq);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}
int k_ctrl_B_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq1, unsigned long long seq2)
{
  (void)win;
  prof_pre(KF_CTRL, 0);
  k_ctrl_B_p2p_kernel<<<1, 32, 0, g_ctx.stream>>>(S, g_p2p_size, my_slot, my_flag, seq1, seq2);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}

int k_ctrl_A(MpgpCtl *S, const double *ra)
{
  prof_pre(KF_CTRL, 0);
  k_ctrl_A_kernel<<<1, 1, 0, g_ctx.stream>>>(S, ra);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}
int k_ctrl_E(MpgpCtl *S, const double *rb)
{
  prof_pre(KF_CTRL, 0);
  k_ctrl_E_kernel<<<1, 1, 0, g_ctx.stream>>>(S, rb);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}
int k_ctrl_B(MpgpCtl *S, const double *rb)
{
  prof_pre(KF_CTRL, 0);
  k_ctrl_B_kernel<<<1, 1, 0, g_ctx.stream>>>(S, rb);
  prof_post(KF_CTRL);
  LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// generic vector kernels
// =====================================================================================================
template <class F>
__global__ void __launch_bounds__(NT) k_elementwise(int n, F f)
{
  const int stride = gridDim.x * NT;
  for (int i = blockIdx.x * NT + threadIdx.x; i < n; i += stride) f(i);
}
template <class F>
static int launch_ew(int n, F f, int family, double bytes)
{
  if (n <= 0) return 0;
  int grid = elementwise_grid();
  int need = (n + NT - 1) / NT;
  if (grid > need) grid = need;
  prof_pre(family, bytes);
  k_elementwise<<<grid, NT, 0, g_ctx.stream>>>(n, f);
  prof_post(family);
  LAUNCH_CHECK();
  return 0;
}

int k_set(int n, double *x, double a)
{
  return launch_ew(n, [=] __device__(int i) { x[i] = a; }, KF_VEC, 8.0 * n);
}
int k_copy(int n, const double *x, double *y)
{
  if (x == y) return 0;
  return launch_ew(n, [=] __device__(int i) { y[i] = x[i]; }, KF_VEC, 16.0 * n);
}
int k_scale(int n, double *x, double a)
{
  return launch_ew(n, [=] __device__(int i) { x[i] *= a; }, KF_VEC, 16.0 * n);
}
int k_filter(int n, double *x, double tol)
{   // PETSc VecFilter: entries with |x_i| < tol become 0
  return launch_ew(n, [=] __device__(int i) { const double v = x[i]; if (fabs(v) < tol) x[i] = 0.0; }, KF_VEC, 16.0 * n);
}
int k_scale_to(int n, double *y, double a, const double *x)
{   // y = a x : VecCopy + VecScale in one pass (same products, same rounding)
  return launch_ew(n, [=] __device__(int i) { y[i] = x[i] * a; }, KF_VEC, 16.0 * n);
}
int k_axpy(int n, double *y, double a, const double *x)
{
  return launch_ew(n, [=] __device__(int i) { y[i] += a * x[i]; }, KF_VEC, 24.0 * n);
}
int k_aypx(int n, double *y, double a, const double *x)
{
  return launch_ew(n, [=] __device__(int i) { y[i] = x[i] + a * y[i]; }, KF_VEC, 24.0 * n);
}
int k_waxpy(int n, double *w, double a, const double *x, const double *y)
{
  return launch_ew(n, [=] __device__(int i) { w[i] = a * x[i] + y[i]; }, KF_VEC, 24.0 * n);
}
int k_pmax(int n, double *w, const double *x, const double *y)
{
  return launch_ew(n, [=] __device__(int i) { double a = x[i], b = y[i]; w[i] = (a < b) ? b : a; }, KF_VEC, 24.0 * n);
}
int k_pmin(int n, double *w, const double *x, const double *y)
{
  return launch_ew(n, [=] __device__(int i) { double a = x[i], b = y[i]; w[i] = (a < b) ? a : b; }, KF_VEC, 24.0 * n);
}
int k_scatter_is(int nis, const int *is, const double *sub, double fill, int n, double *full)
{
  PB_CHK(k_set(n, full, fill));
  return launch_ew(nis, [=] __device__(int k) { full[is[k]] = sub[k]; }, KF_VEC, 20.0 * nis);
}
int k_pack(int n, const int *idx, const double *x, double *buf)
{
  return launch_ew(n, [=] __device__(int k) { buf[k] = x[idx[k]]; }, KF_HALO, 20.0 * n);
}
int k_dense_rows_multT_add(int n, int m, const double *B, const double *t, double scale, double *y, int accumulate)
{
  return launch_ew(n, [=] __device__(int i) {
    double s = 0.0;
    for (int j = 0; j < m; j++) s += B[(size_t)j * n + i] * t[j];
    y[i] = accumulate ? y[i] + scale * s : scale * s;
  }, KF_VEC, 8.0 * n * (m + 2));
}
int k_qpc_project(int n, const double *x, BoxDev bx, double *Px)
{
  return launch_ew(n, [=] __device__(int i) { Px[i] = box_project(x[i], load_box(bx, i)); }, KF_QPC, 32.0 * n);
}
// MatOrthColumns_Cholesky_Default (permonmatorth.c:97-110): every column of G is forward-solved with the Cholesky factor of G G^T
struct SmallLower {
  double v[PB_MAXEQ * PB_MAXEQ];
};
int k_rows_forward_solve(int n, int m, const double *L, const double *G, double *TB)
{
  SmallLower Ls;
  for (int i = 0; i < m * m; i++) Ls.v[i] = L[i];
  return launch_ew(
    n,
    [=] __device__(int col) {
      double y[PB_MAXEQ];
#pragma unroll
      for (int i = 0; i < PB_MAXEQ; i++) {
        if (i < m) {
          double v = G[(size_t)i * n + col];
          for (int k = 0; k < i; k++) v -= Ls.v[i * m + k] * y[k];
          y[i]                   = v / Ls.v[i * m + i];
          TB[(size_t)i * n + col] = y[i];
        }
      }
    },
    KF_VEC, 16.0 * n * m);
}

int k_qpc_grads(int n, const double *x, const double *g, BoxDev bx, double *gf, double *gc)
{
  return launch_ew(n, [=] __device__(int i) {
    double a, c;
    box_split(x[i], g[i], load_box(bx, i), bx.astol, a, c);
    gf[i] = a;
    gc[i] = c;
  }, KF_QPC, 48.0 * n);
}
int k_qpc_gradreduced(int n, const double *x, const double *gf, double alpha, BoxDev bx, double *gr)
{
  return launch_ew(n, [=] __device__(int i) { gr[i] = box_reduced(x[i], gf[i], load_box(bx, i), alpha); }, KF_QPC, 40.0 * n);
}
int k_box_mult(int n, const double *r, int has_lb, int has_ub, double *llb, double *lub)
{   // QPComputeMissingBoxMultipliers qp.c:858-881
  return launch_ew(n, [=] __device__(int i) {
    const double ri = r[i];
    if (has_lb) llb[i] = (has_ub && ri < 0.0) ? 0.0 : ri;
    if (has_ub) {
      const double u = -1.0 * ri;
      lub[i]         = (has_lb && u < 0.0) ? 0.0 : u;
    }
  }, KF_VEC, 24.0 * n);
}

// reductions ---------------------------------------------------------------------------------------------
template <int MINMASK, class F>
__global__ void __launch_bounds__(NT) k_reduce(int n, F f, RedBuf rb)
{
  double acc[PB_NRED];
#pragma unroll
  for (int k = 0; k < PB_NRED; k++) acc[k] = red_identity<MINMASK>(k);
  const int stride = gridDim.x * NT;
  for (int i = blockIdx.x * NT + threadIdx.x; i < n; i += stride) f(i, acc);
  grid_reduce8<MINMASK>(acc, rb, nullptr);
}
template <int MINMASK, class F>
static int launch_red(int n, F f, RedBuf rb, int family, double bytes)
{
  int grid = elementwise_grid();
  int need = (n + NT - 1) / NT;
  if (need < 1) need = 1;
  if (grid > need) grid = need;
  prof_pre(family, bytes);
  k_reduce<MINMASK><<<grid, NT, 0, g_ctx.stream>>>(n, f, rb);
  prof_post(family);
  LAUNCH_CHECK();
  return 0;
}
int k_dot(int n, const double *x, const double *y, RedBuf rb)
{
  return launch_red<0>(n, [=] __device__(int i, double(&a)[PB_NRED]) { a[0] += x[i] * y[i]; }, rb, KF_VEC, 16.0 * n);
}
// CG update in one pass (KSPSolve_CG: VecAXPY(X, a, P); VecAXPY(R, -a, W); dp = VecNorm(R); beta = VecDot(R, R)): x += a p, r -= a w,
// out[0] = r.r of the new residual -- the norm and the dot product of the reference are the same sum
int k_cg_update(int n, double a, const double *p, const double *w, double *x, double *r, RedBuf rb)
{
  return launch_red<0>(n, [=] __device__(int i, double(&acc)[PB_NRED]) {
    x[i] += a * p[i];
    const double ri = r[i] + (-a) * w[i];
    r[i]            = ri;
    acc[0] += ri * ri;
  }, rb, KF_VEC, 48.0 * n);
}
int k_mdot2(int n, const double *x, const double *y0, const double *y1, RedBuf rb)
{
  return launch_red<0>(n, [=] __device__(int i, double(&a)[PB_NRED]) {
    const double xi = x[i];
    a[0] += xi * y0[i];
    a[1] += xi * y1[i];
  }, rb, KF_VEC, 24.0 * n);
}
int k_dense_rows_mult(int n, int m, const double *B, const double *x, RedBuf rb)
{
  return launch_red<0>(n, [=] __device__(int i, double(&a)[PB_NRED]) {
    const double xi = x[i];
    for (int j = 0; j < m; j++) a[j] += B[(size_t)j * n + i] * xi;
  }, rb, KF_VEC, 8.0 * n * (m + 1));
}
int k_qpc_feas(int n, const double *x, const double *d, BoxDev bx, RedBuf rb)
{
  return launch_red<(1 << RA_FEAS)>(n, [=] __device__(int i, double(&a)[PB_NRED]) { a[RA_FEAS] = box_feas_lazy(x[i], d[i], load_box(bx, i), a[RA_FEAS]); }, rb, KF_QPC, 32.0 * n);
}
// QPCViewKKT_Box numbers (qpcbox.c:333-427): out[0]=sum min(x-lb,0)^2 | max(x-ub,0)^2, out[1]=sum min(lam,0)^2,
// out[2]=lam'(lb-x) | lam'(x-ub) with the infinite-bound convention of the reference
int k_kkt_box(int n, const double *x, const double *bound, const double *lam, int upper, RedBuf rb)
{
  const double PINF = 1.7976931348623157e+308 / 4.0;
  return launch_red<0>(n, [=] __device__(int i, double(&a)[PB_NRED]) {
    const double xi = x[i], bi = bound[i], li = lam[i];
    double       d, t;
    if (!upper) {
      d = xi - bi;
      d = (d < 0.0) ? d : 0.0;
      t = bi - xi;
      if (bi <= -PINF) t = -1.0;
    } else {
      d = xi - bi;
      d = (d < 0.0) ? 0.0 : d;
      t = xi - bi;
      if (bi >= PINF) t = 1.0;
    }
    const double lm = (li < 0.0) ? li : 0.0;
    a[0] += d * d;
    a[1] += lm * lm;
    a[2] += li * t;
  }, rb, KF_QPC, 24.0 * n);
}

}  // namespace pb
