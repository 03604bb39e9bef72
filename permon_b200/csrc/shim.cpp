// shim.cpp -- the PETSc stand-in behind include/permon_b200.h: communicator (one process per GPU, NCCL),
// options database, viewers, IS, Vec and Mat with host<->device validity tracking, the row-partitioned AIJ
// matrix with its halo plan, and the generic (un-fused) Mat/Vec operations built on the CUDA kernels.
// There is no CPU arithmetic here: every numerical operation launches a kernel from kernels.cu.
#include <time.h>
#include <cuda_runtime.h>
#include <math.h>
#include <nccl.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <omp.h>

#include <algorithm>
#include <fstream>
#include <sstream>

#include "objects.h"

using namespace pb;

static _p_PermonComm g_world, g_self;
MPI_Comm             PETSC_COMM_WORLD = &g_world;
MPI_Comm             PETSC_COMM_SELF  = &g_self;

static std::map<std::string, std::string> g_opts;
static std::map<MPI_Comm, Reducer>        g_reducers;

namespace pb {

int err(int code, const char *fmt, ...)
{
  char    buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  set_error("%s", buf);
  return code;
}

#define PB_NCCL(call)                                                                          \
  do {                                                                                         \
    ncclResult_t r_ = (call);                                                                  \
    if (r_ != ncclSuccess) return pb::err(PETSC_ERR_LIB, "NCCL error %d (%s) in %s at %s:%d", (int)r_, ncclGetErrorString(r_), #call, __FILE__, __LINE__); \
  } while (0)

// ---------------------------------------------------------------------------------------------------
// options
// ---------------------------------------------------------------------------------------------------
int options_get(const std::string &prefix, const char *name, std::string *val)
{
  std::string key = std::string("-") + prefix + (name[0] == '-' ? name + 1 : name);
  auto        it = g_opts.find(key);
  if (it == g_opts.end()) return 0;
  if (val) *val = it->second;
  return 1;
}
bool options_real(const std::string &prefix, const char *name, double *v)
{
  std::string s;
  if (!options_get(prefix, name, &s)) return false;
  if (s == "PETSC_DECIDE" || s == "decide") *v = PETSC_DECIDE;
  else *v = atof(s.c_str());
  return true;
}
bool options_int(const std::string &prefix, const char *name, PetscInt *v)
{
  std::string s;
  if (!options_get(prefix, name, &s)) return false;
  *v = (PetscInt)atol(s.c_str());
  return true;
}
bool options_bool(const std::string &prefix, const char *name, bool *v)
{
  std::string s;
  if (!options_get(prefix, name, &s)) return false;
  std::string t = s;
  std::transform(t.begin(), t.end(), t.begin(), ::tolower);
  *v = (t.empty() || t == "1" || t == "true" || t == "yes" || t == "on");
  return true;
}
bool options_string(const std::string &prefix, const char *name, std::string *v) { return options_get(prefix, name, v) != 0; }

void vprintf_viewer(PetscViewer v, const char *fmt, ...)
{
  if (PETSC_COMM_WORLD->rank != 0) return;
  FILE *f = (v && v->f) ? v->f : stdout;
  int   tab = v ? v->tab : 0;
  for (int i = 0; i < tab; i++) fputs("  ", f);
  va_list ap;
  va_start(ap, fmt);
  vfprintf(f, fmt, ap);
  va_end(ap);
  fflush(f);
}

// ---------------------------------------------------------------------------------------------------
// reducer
// ---------------------------------------------------------------------------------------------------
int Reducer::init(MPI_Comm c)
{
  comm = c;
  PB_CHK(dev_init());
  const int size = c->size;
  cudaStream_t s = ctx().stream;
  PB_CHK(dmalloc(&rb.partials, PB_NRED * (size_t)max_red_blocks()));
  PB_CHK(dmalloc(&rb.counter, 4));   // 16 bytes: the counter and its padding
  PB_CUDA(cudaMemsetAsync(rb.counter, 0, sizeof(unsigned), s));
  PB_CHK(dmalloc(&d_all, (size_t)PB_NRED * size));
  PB_CUDA(cudaMemsetAsync(d_all, 0, sizeof(double) * PB_NRED * size, s));
  if (size > 1) {
    PB_CHK(dmalloc(&d_local, (size_t)PB_NRED));
    PB_CUDA(cudaMemsetAsync(d_local, 0, sizeof(double) * PB_NRED, s));
  } else {
    d_local = d_all;
  }
  h_all = (double *)pinned_get(sizeof(double) * PB_NRED * size);
  if (!h_all) return err(PETSC_ERR_MEM, "out of pinned host memory");
  rb.out = d_local;
  return 0;
}
void Reducer::destroy()
{
  if (!rb.partials) return;
  dfree(rb.partials);
  dfree(rb.counter);
  if (d_local != d_all) dfree(d_local);
  dfree(d_all);
  pinned_put(h_all, sizeof(double) * PB_NRED * comm->size);
  rb = RedBuf();
  d_local = d_all = h_all = nullptr;
}
int Reducer::gather() { return comm_allgather_records(comm, d_local, d_all); }
int Reducer::fetch()
{
  PB_CUDA(cudaMemcpyAsync(h_all, d_all, sizeof(double) * PB_NRED * comm->size, cudaMemcpyDeviceToHost, ctx().stream));
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  return 0;
}
double Reducer::sum(int slot) const
{
  double s = 0.0;
  for (int r = 0; r < comm->size; r++) s += h_all[r * PB_NRED + slot];
  return s;
}
double Reducer::min(int slot) const
{
  double s = HUGE_VAL;
  for (int r = 0; r < comm->size; r++)
    if (h_all[r * PB_NRED + slot] < s) s = h_all[r * PB_NRED + slot];
  return s;
}
Reducer &reducer(MPI_Comm comm)
{
  Reducer &r = g_reducers[comm];
  if (!r.rb.partials) r.init(comm);
  return r;
}

int comm_allgather_records(MPI_Comm comm, const double *d_local, double *d_all)
{
  if (comm->size == 1) return 0;
  if (!comm->nccl) return err(PETSC_ERR_ARG_WRONGSTATE, "multi-rank communicator without NCCL (call PermonB200CommInitRank on a GPU box)");
  ctx().launches++;
  PB_NCCL(ncclAllGather(d_local, d_all, PB_NRED, ncclDouble, (ncclComm_t)comm->nccl, ctx().stream));
  return 0;
}

// ---------------------------------------------------------------------------------------------------
// Vec internals
// ---------------------------------------------------------------------------------------------------
int vec_layout(MPI_Comm comm, PetscInt n, PetscInt *N, PetscInt *rstart)
{
  if (comm->size == 1) {
    *N      = n;
    *rstart = 0;
    return 0;
  }
  if (!comm->agi) return err(PETSC_ERR_ARG_WRONGSTATE, "communicator has no host exchange");
  std::vector<int64_t> all(comm->size);
  if (comm->agi(comm->agctx, (int64_t)n, all.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  int64_t s = 0, tot = 0;
  for (int r = 0; r < comm->size; r++) {
    if (r < comm->rank) s += all[r];
    tot += all[r];
  }
  *N      = (PetscInt)tot;
  *rstart = (PetscInt)s;
  return 0;
}

int vec_create(MPI_Comm comm, PetscInt n, PetscInt N, Vec *v)
{
  _p_Vec *w = new _p_Vec;
  w->comm   = comm;
  w->n      = n;
  if (N == PETSC_DECIDE || comm->size > 1) {
    PetscInt NN = 0, rs = 0;
    int      ierr = vec_layout(comm, n, &NN, &rs);
    if (ierr) {
      delete w;
      return ierr;
    }
    w->N      = NN;
    w->rstart = rs;
  } else {
    w->N      = N;
    w->rstart = 0;
  }
  *v = w;
  return 0;
}

static int vec_alloc_dev(Vec v)
{
  if (v->d) return 0;
  PB_CHK(dev_init());
  PB_CHK(dmalloc(&v->d, (size_t)std::max<PetscInt>(v->n, 1)));
  v->d_owned = true;
  return 0;
}
static int vec_alloc_host(Vec v)
{
  if (v->h) return 0;
  v->h = (double *)malloc(sizeof(double) * (size_t)std::max<PetscInt>(v->n, 1));
  if (!v->h) return err(PETSC_ERR_MEM, "out of host memory");
  v->h_owned = true;
  return 0;
}
// a prefetch in flight: device users wait on the stream, host users on the host
static int vec_settle(Vec v, bool host_side)
{
  if (!v->up_ev) return 0;
  if (host_side) PB_CUDA(cudaEventSynchronize(v->up_ev));
  else PB_CUDA(cudaStreamWaitEvent(ctx().stream, v->up_ev, 0));
  PB_CUDA(cudaEventDestroy(v->up_ev));
  v->up_ev = nullptr;
  return 0;
}
int vec_prefetch(Vec v)
{
  if (!v || v->d_valid || !v->h_valid || v->n == 0 || v->up_ev || getenv("PERMON_B200_NOPREFETCH")) return 0;
  PB_CHK(vec_alloc_dev(v));
  DevCtx     &c = ctx();
  cudaEvent_t ea;
  PB_CUDA(cudaEventCreateWithFlags(&ea, cudaEventDisableTiming));
  PB_CUDA(cudaEventRecord(ea, c.stream));   // the (stream-ordered) allocation precedes the copy
  PB_CUDA(cudaStreamWaitEvent(c.copy_stream, ea, 0));
  PB_CUDA(cudaEventDestroy(ea));
  PB_CUDA(cudaMemcpyAsync(v->d, v->h, sizeof(double) * (size_t)v->n, cudaMemcpyHostToDevice, c.copy_stream));
  PB_CUDA(cudaEventCreateWithFlags(&v->up_ev, cudaEventDisableTiming));
  PB_CUDA(cudaEventRecord(v->up_ev, c.copy_stream));
  v->d_valid = true;
  return 0;
}
int vec_dev_read(Vec v, const double **d)
{
  PB_CHK(vec_settle(v, false));
  PB_CHK(vec_alloc_dev(v));
  if (!v->d_valid) {
    if (v->h_valid) {
      PB_CUDA(cudaMemcpyAsync(v->d, v->h, sizeof(double) * (size_t)v->n, cudaMemcpyHostToDevice, ctx().stream));
      v->h2d_inflight = true;   // pinned host buffers: the DMA really is asynchronous
    } else {
      PB_CUDA(cudaMemsetAsync(v->d, 0, sizeof(double) * (size_t)v->n, ctx().stream));
    }
    v->d_valid = true;
  }
  *d = v->d;
  return 0;
}
int vec_dev_write(Vec v, double **d)
{
  PB_CHK(vec_settle(v, false));
  PB_CHK(vec_alloc_dev(v));
  v->d_valid = true;
  v->h_valid = false;
  v->state++;
  *d = v->d;
  return 0;
}
int vec_dev_rw(Vec v, double **d)
{
  const double *c;
  PB_CHK(vec_dev_read(v, &c));
  v->h_valid = false;
  v->state++;
  *d = v->d;
  return 0;
}
int vec_host_read(Vec v, const double **h)
{
  PB_CHK(vec_settle(v, true));
  PB_CHK(vec_alloc_host(v));
  if (!v->h_valid) {
    if (v->d_valid) {
      PhaseTimer pt("Vec download (D2H)");
      PB_CUDA(cudaMemcpyAsync(v->h, v->d, sizeof(double) * (size_t)v->n, cudaMemcpyDeviceToHost, ctx().stream));
      PB_CUDA(cudaStreamSynchronize(ctx().stream));
    } else {
      memset(v->h, 0, sizeof(double) * (size_t)v->n);
    }
    v->h_valid = true;
  }
  *h = v->h;
  return 0;
}
int vec_host_write(Vec v, double **h)
{
  PB_CHK(vec_settle(v, true));
  PB_CHK(vec_alloc_host(v));
  if ((v->d_valid || v->h2d_inflight) && ctx().ready) PB_CUDA(cudaStreamSynchronize(ctx().stream));   // pending device readers / an upload still reading the host buffer
  v->h2d_inflight = false;
  v->h_valid = true;
  v->d_valid = false;
  v->state++;
  *h = v->h;
  return 0;
}
int vec_host_rw(Vec v, double **h)
{
  const double *c;
  PB_CHK(vec_host_read(v, &c));
  if (v->h2d_inflight && ctx().ready) {   // the caller is about to WRITE the buffer an asynchronous upload may still be reading
    PB_CUDA(cudaStreamSynchronize(ctx().stream));
    v->h2d_inflight = false;
  }
  v->d_valid = false;
  v->state++;
  *h = v->h;
  return 0;
}

int dense_rows_mult_host(MPI_Comm comm, int n, int m, const double *Bd, const double *x, double *t)
{
  Reducer &R = reducer(comm);
  for (int c = 0; c < m; c += PB_NRED) {
    const int mc = std::min(PB_NRED, m - c);
    PB_CHK(k_dense_rows_mult(n, mc, Bd + (size_t)c * n, x, R.rb));
    PB_CHK(R.gather());
    PB_CHK(R.fetch());
    for (int j = 0; j < mc; j++) t[c + j] = R.sum(j);
  }
  return 0;
}
int dense_rows_multT_host(MPI_Comm comm, int n, int m, const double *Bd, const double *t, double scale, double *y, int accumulate)
{
  Reducer &R = reducer(comm);
  if (m == 0 && !accumulate) return k_set(n, y, 0.0);
  for (int c = 0; c < m; c += PB_NRED) {
    const int mc = std::min(PB_NRED, m - c);
    // t is pageable host memory: the copy is staged before the call returns, the chunk buffer can be reused right away on the stream
    PB_CUDA(cudaMemcpyAsync(R.d_all, t + c, sizeof(double) * mc, cudaMemcpyHostToDevice, ctx().stream));
    PB_CHK(k_dense_rows_multT_add(n, mc, Bd + (size_t)c * n, R.d_all, scale, y, (accumulate || c > 0) ? 1 : 0));
  }
  return 0;
}
int vec_dot(Vec x, Vec y, double *val)
{
  if (x->n != y->n) return err(PETSC_ERR_ARG_INCOMP, "VecDot: local sizes differ (%d vs %d)", (int)x->n, (int)y->n);
  const double *dx, *dy;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(y, &dy));
  Reducer &R = reducer(x->comm);
  PB_CHK(k_dot(x->n, dx, dy, R.rb));
  PB_CHK(R.gather());
  PB_CHK(R.fetch());
  *val = R.sum(0);
  return 0;
}
int vec_norm2(Vec x, double *val)
{
  double d;
  PB_CHK(vec_dot(x, x, &d));
  *val = sqrt(d);
  return 0;
}
int vec_mdot2(Vec x, Vec y0, Vec y1, double *v0, double *v1)
{
  const double *dx, *d0, *d1;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(y0, &d0));
  PB_CHK(vec_dev_read(y1, &d1));
  Reducer &R = reducer(x->comm);
  PB_CHK(k_mdot2(x->n, dx, d0, d1, R.rb));
  PB_CHK(R.gather());
  PB_CHK(R.fetch());
  *v0 = R.sum(0);
  *v1 = R.sum(1);
  return 0;
}

}  // namespace pb

_p_Vec::~_p_Vec()
{
  if (up_ev) {
    cudaEventSynchronize(up_ev);
    cudaEventDestroy(up_ev);
  }
  if (h_owned && h) free(h);
  if (d_owned && d) pb::dfree(d);
}

// =====================================================================================================
// life cycle and B200 helpers
// =====================================================================================================
static bool g_initialized = false;

static void options_insert_tokens(const std::vector<std::string> &tok)
{
  for (size_t i = 0; i < tok.size(); i++) {
    const std::string &t = tok[i];
    if (t.size() < 2 || t[0] != '-' || (t[1] >= '0' && t[1] <= '9')) continue;
    std::string val;
    if (i + 1 < tok.size()) {
      const std::string &nx = tok[i + 1];
      bool is_key = nx.size() >= 2 && nx[0] == '-' && !((nx[1] >= '0' && nx[1] <= '9') || nx[1] == '.');
      if (!is_key) {
        val = nx;
        i++;
      }
    }
    g_opts[t] = val;
  }
}
static void options_insert_file(const std::string &path)
{
  std::ifstream f(path);
  if (!f) return;
  std::string              line;
  std::vector<std::string> tok;
  while (std::getline(f, line)) {
    size_t h = line.find('#');
    if (h != std::string::npos) line = line.substr(0, h);
    std::istringstream is(line);
    std::string        w;
    while (is >> w) tok.push_back(w);
  }
  options_insert_tokens(tok);
}

PetscErrorCode PermonInitialize(int *argc, char ***args, const char file[], const char help[])
{
  (void)help;
  if (g_initialized) return 0;
  // rc files exactly as src/sys/permoninit.c:62-73: ~/.permonrc, ./permonrc, ./.permonrc, then argv
  const char *home = getenv("HOME");
  if (home) options_insert_file(std::string(home) + "/.permonrc");
  options_insert_file("permonrc");
  options_insert_file(".permonrc");
  if (file) options_insert_file(file);
  if (argc && args && *args) {
    std::vector<std::string> tok;
    for (int i = 1; i < *argc; i++) tok.push_back((*args)[i]);
    options_insert_tokens(tok);
  }
  g_initialized = true;
  return 0;
}

PetscErrorCode PermonFinalize(void)
{
  for (auto &kv : g_reducers) kv.second.destroy();
  g_reducers.clear();
  if (g_world.p2p) {
    for (int q = 0; q < g_world.size; q++)
      if (q != g_world.rank && g_world.peer_bases[q]) cudaIpcCloseMemHandle(g_world.peer_bases[q]);
    cudaFree(g_world.d_win);
    g_world.p2p = false;
  }
  if (g_world.win_base) {
    cudaFree(g_world.win_base);
    g_world.win_base = nullptr;
  }
  if (g_world.nccl) {
    ncclCommDestroy((ncclComm_t)g_world.nccl);
    g_world.nccl = nullptr;
  }
  g_initialized = false;
  return 0;
}

PetscErrorCode PermonB200GetDeviceCount(int *count)
{
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) c = 0;
  *count = c;
  return 0;
}
PetscErrorCode PermonB200SetDevice(int device)
{
  if (ctx().ready && ctx().device != device) return err(PETSC_ERR_ARG_WRONGSTATE, "device already initialised as %d", ctx().device);
  ctx().device = device;
  return 0;
}
PetscErrorCode PermonB200SetStream(void *s)
{
  PB_CHK(dev_init());
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  ctx().stream = s ? (cudaStream_t)s : ctx().own_stream;
  return 0;
}
PetscErrorCode PermonB200GetStream(void **s)
{
  PB_CHK(dev_init());
  *s = (void *)ctx().stream;
  return 0;
}
PetscErrorCode PermonB200Synchronize(void)
{
  PB_CHK(dev_init());
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  PB_CUDA(cudaStreamSynchronize(ctx().comm_stream));
  return 0;
}
PetscErrorCode PermonB200GetUniqueId(void *id128)
{
  ncclUniqueId id;
  PB_NCCL(ncclGetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, 128);
  return 0;
}

// default host exchange over NCCL (device staging); only used at set-up time
static int nccl_agi(void *vctx, int64_t value, int64_t *all)
{
  MPI_Comm c = (MPI_Comm)vctx;
  int64_t *d = nullptr;
  if (cudaMalloc(&d, sizeof(int64_t) * (c->size + 1)) != cudaSuccess) return 1;
  cudaMemcpyAsync(d + c->size, &value, sizeof(int64_t), cudaMemcpyHostToDevice, ctx().stream);
  if (ncclAllGather(d + c->size, d, 1, ncclInt64, (ncclComm_t)c->nccl, ctx().stream) != ncclSuccess) return 1;
  cudaMemcpyAsync(all, d, sizeof(int64_t) * c->size, cudaMemcpyDeviceToHost, ctx().stream);
  if (cudaStreamSynchronize(ctx().stream) != cudaSuccess) return 1;
  cudaFree(d);
  return 0;
}
static int nccl_agv(void *vctx, const void *sendbuf, int64_t sendbytes, void *recvbuf, const int64_t *recvbytes)
{
  MPI_Comm c = (MPI_Comm)vctx;
  int64_t  mx = 0;
  for (int r = 0; r < c->size; r++) mx = std::max(mx, recvbytes[r]);
  mx = (mx + 15) & ~(int64_t)15;
  if (mx == 0) return 0;
  char *d = nullptr;
  if (cudaMalloc(&d, (size_t)mx * (c->size + 1)) != cudaSuccess) return 1;
  char *mine = d + (size_t)mx * c->size;
  cudaMemcpyAsync(mine, sendbuf, (size_t)sendbytes, cudaMemcpyHostToDevice, ctx().stream);
  if (ncclAllGather(mine, d, (size_t)mx, ncclChar, (ncclComm_t)c->nccl, ctx().stream) != ncclSuccess) return 1;
  std::vector<char> h((size_t)mx * c->size);
  cudaMemcpyAsync(h.data(), d, h.size(), cudaMemcpyDeviceToHost, ctx().stream);
  if (cudaStreamSynchronize(ctx().stream) != cudaSuccess) return 1;
  char *out = (char *)recvbuf;
  for (int r = 0; r < c->size; r++) {
    memcpy(out, h.data() + (size_t)mx * r, (size_t)recvbytes[r]);
    out += recvbytes[r];
  }
  cudaFree(d);
  return 0;
}

// Peer-memory window of the communicator: one small cudaMalloc per rank, mapped by every peer through CUDA IPC.
static const size_t kWinSlotBytes = sizeof(double) * PB_NKINDS * 2 * PB_MAXRANKS * PB_NRED;
static const size_t kWinFlagBytes = sizeof(unsigned long long) * PB_NKINDS * PB_MAXRANKS * PB_FLAG_STRIDE;
static int comm_p2p_setup(MPI_Comm c)
{
  const int size = c->size, rank = c->rank;
  PB_CUDA(cudaMalloc(&c->win_base, kWinSlotBytes + kWinFlagBytes));
  PB_CUDA(cudaMemset(c->win_base, 0, kWinSlotBytes + kWinFlagBytes));
  PB_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t mine;
  int                ok = (cudaIpcGetMemHandle(&mine, c->win_base) == cudaSuccess);
  std::vector<cudaIpcMemHandle_t> all(size);
  std::vector<int64_t>            bytes(size, (int64_t)sizeof(cudaIpcMemHandle_t));
  if (c->agv(c->agctx, &mine, sizeof mine, all.data(), bytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  c->peer_bases.assign(size, nullptr);
  for (int q = 0; q < size && ok; q++) {
    if (q == rank) {
      c->peer_bases[q] = c->win_base;
      continue;
    }
    if (cudaIpcOpenMemHandle(&c->peer_bases[q], all[q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      ok = 0;
    }
  }
  std::vector<int64_t> oks(size);
  if (c->agi(c->agctx, ok, oks.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  for (int q = 0; q < size; q++) ok = ok && oks[q];
  if (!ok) {   // no peer access between some pair of devices: keep the NCCL path
    c->p2p = false;
    return 0;
  }
  P2PWin W;
  W.rank = rank;
  W.size = size;
  for (int q = 0; q < PB_MAXRANKS; q++) {
    W.slot[q] = q < size ? (double *)c->peer_bases[q] : nullptr;
    W.flag[q] = q < size ? (unsigned long long *)((char *)c->peer_bases[q] + kWinSlotBytes) : nullptr;
  }
  PB_CUDA(cudaMalloc(&c->d_win, sizeof(P2PWin)));
  PB_CUDA(cudaMemcpy(c->d_win, &W, sizeof W, cudaMemcpyHostToDevice));
  c->my_slot = (double *)c->win_base;
  c->my_flag = (unsigned long long *)((char *)c->win_base + kWinSlotBytes);
  g_p2p_size = size;
  c->p2p     = true;
  return 0;
}

PetscErrorCode PermonB200CommInitRank(int nranks, int rank, const void *id128)
{
  if (nranks < 1 || rank < 0 || rank >= nranks) return err(PETSC_ERR_ARG_OUTOFRANGE, "bad rank %d of %d", rank, nranks);
  if (nranks > PB_MAXRANKS) return err(PETSC_ERR_SUP, "at most %d ranks", PB_MAXRANKS);
  g_world.rank = rank;
  g_world.size = nranks;
  if (nranks == 1) return 0;
  // one process per GPU on one node: the ranks' OpenMP regions (host split of the matrix, packer) share the host cores instead of
  // every rank starting one thread per core
  if (!getenv("OMP_NUM_THREADS")) {
    const int per = omp_get_num_procs() / nranks;
    omp_set_num_threads(per > 1 ? per : 1);
  }
  PB_CHK(dev_init());
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclComm_t c;
  PB_NCCL(ncclCommInitRank(&c, nranks, id, rank));
  g_world.nccl  = (ncclComm *)c;
  g_world.agi   = nccl_agi;
  g_world.agv   = nccl_agv;
  g_world.agctx = &g_world;
  const char *pe = getenv("PERMON_B200_P2P");
  if (!pe || strcmp(pe, "0")) PB_CHK(comm_p2p_setup(&g_world));
  return 0;
}

PetscErrorCode PermonB200CommSetHostExchange(int nranks, int rank, PermonB200AllGatherI64 agi, PermonB200AllGatherV agv, void *cctx)
{
  g_world.rank  = rank;
  g_world.size  = nranks;
  g_world.agi   = agi;
  g_world.agv   = agv;
  g_world.agctx = cctx;
  return 0;
}

PetscErrorCode PermonB200ProfileBegin(void)
{
  PB_CHK(dev_init());
  prof_begin();
  return 0;
}
PetscErrorCode PermonB200ProfileEnd(int *nfamilies)
{
  int n = prof_end();
  if (nfamilies) *nfamilies = n;
  return 0;
}
PetscErrorCode PermonB200ProfileGet(int family, const char **name, int64_t *launches, double *total_ms, double *bytes_per_launch)
{
  if (name) *name = family_name(family);
  return prof_get(family, launches, total_ms, bytes_per_launch);
}
PetscErrorCode PermonB200ProfileGetWorking(int family, int64_t *launches, double *total_ms)
{
  if (!launches || !total_ms) return err(PETSC_ERR_ARG_NULL, "null output");
  return prof_get_working(family, launches, total_ms);
}
PetscErrorCode PermonB200ProfileDump(const char *path) { return prof_dump(path); }
PetscErrorCode PermonB200GetLaunchCount(int64_t *launches)
{
  *launches = ctx().launches;
  return 0;
}
const char *PermonB200GetLastErrorMessage(void) { return last_error(); }

// ---- options -----------------------------------------------------------------------------------------
PetscErrorCode PetscOptionsSetValue(void *, const char name[], const char value[])
{
  if (!name || name[0] != '-') return err(PETSC_ERR_ARG_WRONG, "option name must start with '-'");
  g_opts[name] = value ? value : "";
  return 0;
}
PetscErrorCode PetscOptionsClearValue(void *, const char name[])
{
  g_opts.erase(name);
  return 0;
}
PetscErrorCode PetscOptionsClear(void *)
{
  g_opts.clear();
  return 0;
}
PetscErrorCode PetscOptionsInsertString(void *, const char in_str[])
{
  std::istringstream       is(in_str ? in_str : "");
  std::vector<std::string> tok;
  std::string              w;
  while (is >> w) tok.push_back(w);
  options_insert_tokens(tok);
  return 0;
}
PetscErrorCode PetscOptionsHasName(void *, const char pre[], const char name[], PetscBool *set)
{
  *set = options_get(pre ? pre : "", name, nullptr) ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}

// ---- viewers ----------------------------------------------------------------------------------------
PetscErrorCode PetscViewerASCIIOpen(MPI_Comm comm, const char name[], PetscViewer *viewer)
{
  _p_PetscViewer *v = new _p_PetscViewer;
  v->comm = comm;
  if (name && strcmp(name, "stdout")) {
    v->f = (comm->rank == 0) ? fopen(name, "w") : nullptr;
    v->own = true;
    if (comm->rank == 0 && !v->f) {
      delete v;
      return err(PETSC_ERR_ARG_WRONG, "cannot open %s", name);
    }
  }
  *viewer = v;
  return 0;
}
PetscErrorCode PetscViewerDestroy(PetscViewer *viewer)
{
  if (!viewer || !*viewer) return 0;
  if ((*viewer)->own && (*viewer)->f) fclose((*viewer)->f);
  delete *viewer;
  *viewer = nullptr;
  return 0;
}

// ---- IS ------------------------------------------------------------------------------------------------
PetscErrorCode ISCreateStride(MPI_Comm comm, PetscInt n, PetscInt first, PetscInt step, IS *is)
{
  _p_IS *s = new _p_IS;
  s->comm = comm;
  s->idx.resize(n);
  for (PetscInt i = 0; i < n; i++) s->idx[i] = first + i * step;
  *is = s;
  return 0;
}
PetscErrorCode ISCreateGeneral(MPI_Comm comm, PetscInt n, const PetscInt idx[], int, IS *is)
{
  _p_IS *s = new _p_IS;
  s->comm = comm;
  s->idx.assign(idx, idx + n);
  *is = s;
  return 0;
}
PetscErrorCode ISGetLocalSize(IS is, PetscInt *n)
{
  *n = (PetscInt)is->idx.size();
  return 0;
}
PetscErrorCode ISDestroy(IS *is)
{
  if (!is || !*is) return 0;
  if (--(*is)->refct == 0) {
    if ((*is)->d_local) cudaFree((*is)->d_local);
    delete *is;
  }
  *is = nullptr;
  return 0;
}

// ---- Vec -----------------------------------------------------------------------------------------------
PetscErrorCode VecCreateSeq(MPI_Comm comm, PetscInt n, Vec *v) { return vec_create(comm, n, n, v); }
PetscErrorCode VecCreateMPI(MPI_Comm comm, PetscInt n, PetscInt N, Vec *v) { return vec_create(comm, n, N, v); }
PetscErrorCode VecCreateSeqWithArray(MPI_Comm comm, PetscInt, PetscInt n, const PetscScalar array[], Vec *v)
{
  PB_CHK(vec_create(comm, n, n, v));
  if (array) {
    (*v)->h       = const_cast<double *>(array);
    (*v)->h_valid = true;
  }
  return 0;
}
PetscErrorCode VecCreateMPIWithArray(MPI_Comm comm, PetscInt, PetscInt n, PetscInt N, const PetscScalar array[], Vec *v)
{
  PB_CHK(vec_create(comm, n, N, v));
  if (array) {
    (*v)->h       = const_cast<double *>(array);
    (*v)->h_valid = true;
  }
  return 0;
}
PetscErrorCode VecCreateSeqCUDAWithArray(MPI_Comm comm, PetscInt, PetscInt n, const PetscScalar darray[], Vec *v)
{
  PB_CHK(dev_init());
  PB_CHK(vec_create(comm, n, n, v));
  if (darray) {
    (*v)->d       = const_cast<double *>(darray);
    (*v)->d_valid = true;
  }
  return 0;
}
PetscErrorCode VecCreateMPICUDAWithArray(MPI_Comm comm, PetscInt, PetscInt n, PetscInt N, const PetscScalar darray[], Vec *v)
{
  PB_CHK(dev_init());
  PB_CHK(vec_create(comm, n, N, v));
  if (darray) {
    (*v)->d       = const_cast<double *>(darray);
    (*v)->d_valid = true;
  }
  return 0;
}
PetscErrorCode VecDuplicate(Vec v, Vec *newv)
{
  _p_Vec *w = new _p_Vec;
  w->comm   = v->comm;
  w->n      = v->n;
  w->N      = v->N;
  w->rstart = v->rstart;
  *newv     = w;
  return 0;
}
PetscErrorCode VecDestroy(Vec *v)
{
  if (!v || !*v) return 0;
  unref(*v);
  return 0;
}
PetscErrorCode VecGetSize(Vec v, PetscInt *N)
{
  *N = v->N;
  return 0;
}
PetscErrorCode VecGetLocalSize(Vec v, PetscInt *n)
{
  *n = v->n;
  return 0;
}
PetscErrorCode VecGetOwnershipRange(Vec v, PetscInt *low, PetscInt *high)
{
  if (low) *low = v->rstart;
  if (high) *high = v->rstart + v->n;
  return 0;
}
PetscErrorCode VecGetArray(Vec v, PetscScalar **a) { return vec_host_rw(v, a); }
PetscErrorCode VecRestoreArray(Vec, PetscScalar **a)
{
  if (a) *a = nullptr;
  return 0;
}
PetscErrorCode VecGetArrayRead(Vec v, const PetscScalar **a) { return vec_host_read(v, a); }
PetscErrorCode VecRestoreArrayRead(Vec, const PetscScalar **a)
{
  if (a) *a = nullptr;
  return 0;
}
PetscErrorCode VecCUDAGetArray(Vec v, PetscScalar **d) { return vec_dev_rw(v, d); }
PetscErrorCode VecCUDARestoreArray(Vec, PetscScalar **d)
{
  if (d) *d = nullptr;
  return 0;
}
PetscErrorCode VecCUDAGetArrayRead(Vec v, const PetscScalar **d) { return vec_dev_read(v, d); }
PetscErrorCode VecCUDARestoreArrayRead(Vec, const PetscScalar **d)
{
  if (d) *d = nullptr;
  return 0;
}
PetscErrorCode VecSet(Vec v, PetscScalar alpha)
{
  double *d;
  PB_CHK(vec_dev_write(v, &d));
  v->invalidated = false;
  return k_set(v->n, d, alpha);
}
PetscErrorCode VecZeroEntries(Vec v) { return VecSet(v, 0.0); }
PetscErrorCode VecCopy(Vec x, Vec y)
{
  if (x == y) return 0;
  if (x->n != y->n) return err(PETSC_ERR_ARG_INCOMP, "VecCopy: local sizes differ");
  const double *dx;
  double       *dy;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_write(y, &dy));
  pb::vec_mark_invalid(y, pb::vec_invalid(x));
  return k_copy(x->n, dx, dy);
}
PetscErrorCode VecScale(Vec x, PetscScalar alpha)
{
  double *d;
  PB_CHK(vec_dev_rw(x, &d));
  return k_scale(x->n, d, alpha);
}
PetscErrorCode VecAXPY(Vec y, PetscScalar alpha, Vec x)
{
  if (x->n != y->n) return err(PETSC_ERR_ARG_INCOMP, "VecAXPY: local sizes differ");
  const double *dx;
  double       *dy;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_rw(y, &dy));
  return k_axpy(y->n, dy, alpha, dx);
}
PetscErrorCode VecAYPX(Vec y, PetscScalar beta, Vec x)
{
  if (x->n != y->n) return err(PETSC_ERR_ARG_INCOMP, "VecAYPX: local sizes differ");
  const double *dx;
  double       *dy;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_rw(y, &dy));
  return k_aypx(y->n, dy, beta, dx);
}
PetscErrorCode VecWAXPY(Vec w, PetscScalar alpha, Vec x, Vec y)
{
  const double *dx, *dy;
  double       *dw;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(y, &dy));
  if (w == x || w == y) PB_CHK(vec_dev_rw(w, &dw));
  else PB_CHK(vec_dev_write(w, &dw));
  return k_waxpy(w->n, dw, alpha, dx, dy);
}
PetscErrorCode VecPointwiseMax(Vec w, Vec x, Vec y)
{
  const double *dx, *dy;
  double       *dw;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(y, &dy));
  if (w == x || w == y) PB_CHK(vec_dev_rw(w, &dw));
  else PB_CHK(vec_dev_write(w, &dw));
  return k_pmax(w->n, dw, dx, dy);
}
PetscErrorCode VecPointwiseMin(Vec w, Vec x, Vec y)
{
  const double *dx, *dy;
  double       *dw;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(y, &dy));
  if (w == x || w == y) PB_CHK(vec_dev_rw(w, &dw));
  else PB_CHK(vec_dev_write(w, &dw));
  return k_pmin(w->n, dw, dx, dy);
}
PetscErrorCode VecDot(Vec x, Vec y, PetscScalar *val) { return vec_dot(x, y, val); }
PetscErrorCode VecNorm(Vec x, NormType type, PetscReal *val)
{
  if (type != NORM_2) return err(PETSC_ERR_SUP, "only NORM_2 is on the path");
  return vec_norm2(x, val);
}
// VecInvalidate / VecIsInvalidated: src/vec/interface/permonvecutils.c:266,303 ("this multiplier is not computed")
// The reference also fills an invalidated vector with +inf (VecFlag, what src/tests/ex4.c prints); here only the flag is kept -- nothing on the
// path reads an invalidated vector -- together with the rule that any later write (VecSet, VecCopy into it, VecGetArray ...) validates it again.
PetscErrorCode VecInvalidate(Vec vec)
{
  pb::vec_mark_invalid(vec, true);
  return 0;
}
PetscErrorCode VecIsInvalidated(Vec vec, PetscBool *flg)
{
  *flg = pb::vec_invalid(vec) ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}

// =====================================================================================================
// Mat
// =====================================================================================================
_p_Mat::~_p_Mat()
{
  if (kind == MK_AIJ && d_owned) {
    pb::dfree(Ad.ia);
    pb::dfree(Ad.ja);
    pb::dfree(Ad.a);
    pb::dfree(Ad.pk);
    pb::dfree(Ad.pk_off);
    pb::dfree(Ad.st_masks);
    pb::dfree(Ad.st_pid);
    pb::dfree(Ad.st_pats);
    pb::dfree(Ad.ell_val);
    pb::dfree(Ad.ell_col);
    pb::dfree(Ad.ell_len);
    pb::dfree(Ad.ell_lt);
    pb::dfree(Ad.ell_off);
  }
  if (kind == MK_DENSEROWS || eq_host) pb::dfree(rows_d);
  if (kind == MK_DENSE) {
    pb::dfree(dn_own);
    pb::dfree(Ad.dn_part);
  }
  delete eq_host;
  if (kind == MK_AIJ) {
    pb::dfree(Ao.ia);
    pb::dfree(Ao.ja);
    pb::dfree(Ao.a);
    pb::dfree(Ao.rows);
  }
  if (halo) {
    pb::dfree(halo->d_send_idx);
    pb::dfree(halo->d_send);
    pb::dfree(halo->d_ghost);
    pb::dfree(halo->d_row_map);
    if (halo->ev_packed) cudaEventDestroy(halo->ev_packed);
    if (halo->ev_arrived) cudaEventDestroy(halo->ev_arrived);
    if (halo->ev_consumed) cudaEventDestroy(halo->ev_consumed);
    for (void *pw : halo->peer_gwins)
      if (pw) cudaIpcCloseMemHandle(pw);
    if (halo->push[0].counter) cudaFree(halo->push[0].counter);
    if (halo->gwin) cudaFree(halo->gwin);
    if (halo->d_ranges) cudaFree(halo->d_ranges);
    delete halo->host;
    delete halo;
  }
  pb::unref(row);
  pb::unref(M1);
  pb::unref(M2);
  pb::unref(twork);
  pb::unref(A);
  if (pf && --pf->refct == 0) delete pf;
}

namespace pb {
int pk_build(int n, const int *ia, const int *ja, const double *a, RawBuf &blob, std::vector<unsigned> &h_off, int &max_tile_bytes,
             int64_t &ncoded, bool &packed, StencilHost *st, bool want_blob);
int pk_stencil_windowed(int n, const int *ia, const int *ja, const double *a, int coff, int ncols, StencilHost &st, OffDiagEntries &off, int64_t &nnz_diag);
}

static double wall_now()
{
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}
static bool verbose_timing() { return getenv("PERMON_B200_VERBOSE") != nullptr; }

// all-stencil form (device.h): presence bytes + pattern ids + pattern table
static int upload_stencil(pb::CsrDev &C, pb::StencilHost &st, int64_t nnz, double t_build)
{
  cudaStream_t   s = ctx().stream;
  const double   t0 = wall_now();
  unsigned char *dm, *dp;
  pb::StPattern *dt;
  // one spare (zero) tile behind both arrays: the two-rows-per-thread kernel walks pairs of tiles
  PB_CHK(dmalloc(&dm, st.masks.size() + TR));
  PB_CHK(dmalloc(&dp, st.pid.size() + 16));
  PB_CUDA(cudaMemsetAsync(dm + st.masks.size(), 0, TR, s));
  PB_CUDA(cudaMemsetAsync(dp + st.pid.size(), 0, 16, s));
  PB_CHK(dmalloc(&dt, st.pats.size()));
  PB_CUDA(cudaMemcpyAsync(dm, st.masks.data(), st.masks.size(), cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(dp, st.pid.data(), st.pid.size(), cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(dt, st.pats.data(), sizeof(pb::StPattern) * st.pats.size(), cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaStreamSynchronize(s));   // st may be a local
  if (verbose_timing())
    fprintf(stderr, "[permon_b200] matrix %d rows, %lld nnz: all-stencil form (%d patterns, %d windows) built in %.1f ms, %.1f MB uploaded in %.1f ms\n", C.n,
            (long long)nnz, (int)st.pats.size(), st.nwin, 1e3 * t_build, (st.masks.size() + st.pid.size()) / 1e6, 1e3 * (wall_now() - t0));
  C.st_masks = dm;
  C.st_pid   = dp;
  C.st_pats  = dt;
  stencil_set_fields(C, st.pats, st.nwin, st.masks.size(), st.pid.size());
  return 0;
}

namespace pb {
void stencil_set_fields(CsrDev &C, const std::vector<StPattern> &pats, int nwin, size_t masks_bytes, size_t npid)
{
  C.st_npat = (int)pats.size();
  C.st_nwin = nwin;
  C.st_lmax = 0;
  for (const pb::StPattern &P : pats) C.st_lmax = std::max(C.st_lmax, P.L);
  C.st_dlo = C.st_dhi = 0;
  for (const pb::StPattern &P : pats)
    for (int j = 0; j < P.L; j++) {
      C.st_dlo = std::min(C.st_dlo, P.d[j]);
      C.st_dhi = std::max(C.st_dhi, P.d[j]);
    }
  C.pk_bytes = (int64_t)masks_bytes + (int64_t)npid + (int64_t)(sizeof(pb::StPattern) * pats.size());
  C.pk_coded = (int64_t)npid;
  C.kind     = 4;
  const char *stg = getenv("PERMON_B200_STAGES");
  C.stages = stg ? atoi(stg) : 0;   // 0: as many as fit
}
}  // namespace pb

static int upload_csr(pb::CsrDev &C, int nrows, int ncols, const int *ia, const int *ja, const double *a, const int *rows)
{
  const int64_t nnz = ia[nrows];
  C.n     = nrows;
  C.ncols = ncols;
  C.nnz   = nnz;
  cudaStream_t s = ctx().stream;
  if (rows) {
    int *dr;
    PB_CHK(dmalloc(&dr, (size_t)std::max(nrows, 1)));
    PB_CUDA(cudaMemcpyAsync(dr, rows, sizeof(int) * (size_t)nrows, cudaMemcpyHostToDevice, s));
    C.rows = dr;
  }
  PB_CHK(spmv_config(C, ia));
  // Tile-streamable matrices are re-coded into packed tiles (pack.cpp) and only that form goes to the device;
  // PERMON_B200_SPMV=tma|stream|vector keeps plain CSR for A/B measurements.  Tiny matrices (equality rows) stay CSR.
  if (C.kind == 2 && !rows && nrows >= 64 && !getenv("PERMON_B200_SPMV")) {
    pb::RawBuf            blob;
    std::vector<unsigned> off;
    int                        max_tile = 0;
    int64_t                    ncoded = 0;
    bool                       packed = false;
    const double t_pk0 = wall_now();
    pb::StencilHost st;
    const char     *env_w = getenv("PERMON_B200_ST_WINDOWS");
    const bool      want_st = !(env_w && env_w[0] == '0') && nrows == ncols;
    PB_CHK(pb::pk_build(nrows, ia, ja, a, blob, off, max_tile, ncoded, packed, want_st ? &st : nullptr, false));
    const double t_pk1 = wall_now();
    if (packed && st.valid) {
      PB_CHK(upload_stencil(C, st, nnz, t_pk1 - t_pk0));
      C.pk_coded = ncoded;
      return 0;
    }
    // Incompressible matrices (every value distinct: FEM, scaled operators): a raw tile costs 12 B per non-zero in the blob format as
    // well, and the CSR ring (k_spmv_tma: three unit-stride streams, 0.90 of the HBM roof on C2r) beats the blob kernel on raw tiles
    // (0.64) -- measured 1942 vs 1349 it/s on C2r (profiles/README.md).  Break-even is about one third of the tiles coded.
    const int64_t ntiles_pk = ((int64_t)nrows + TR - 1) / TR;
    if (packed && !getenv("PERMON_B200_KEEP_RAW_TILES") && ncoded * 3 < ntiles_pk) packed = false;
    if (packed) {
      unsigned char *dblob;
      unsigned      *doff;
      PB_CHK(dmalloc(&dblob, blob.size()));
      PB_CHK(dmalloc(&doff, off.size()));
      PB_CUDA(cudaMemcpyAsync(dblob, blob.data(), blob.size(), cudaMemcpyHostToDevice, s));
      PB_CUDA(cudaMemcpyAsync(doff, off.data(), sizeof(unsigned) * off.size(), cudaMemcpyHostToDevice, s));
      PB_CUDA(cudaStreamSynchronize(s));   // blob / off are locals
      if (verbose_timing())
        fprintf(stderr, "[permon_b200] matrix %d rows, %lld nnz: re-coded into packed tiles in %.1f ms, %.1f MB uploaded in %.1f ms\n", nrows, (long long)nnz,
                1e3 * (t_pk1 - t_pk0), blob.size() / 1e6, 1e3 * (wall_now() - t_pk1));
      C.pk       = dblob;
      C.pk_off   = doff;
      C.pk_max   = max_tile;
      C.pk_bytes = (int64_t)off.back() * 16 + (int64_t)sizeof(unsigned) * (int64_t)off.size();
      C.pk_coded = ncoded;
      C.kind     = 3;
      const char *st = getenv("PERMON_B200_STAGES");
      C.stages = st ? atoi(st) : 3;
      return 0;
    }
  }
  int *dia, *dja;
  double *da;
  // 8 elements of padding: the TMA kernel copies 16-byte aligned, 16-byte granular tile ranges
  PB_CHK(dmalloc(&dia, (size_t)(nrows + 1 + 8)));
  PB_CHK(dmalloc(&dja, (size_t)(nnz + 8)));
  PB_CHK(dmalloc(&da, (size_t)(nnz + 8)));
  PB_CUDA(cudaMemsetAsync(dia + nrows + 1, 0, sizeof(int) * 8, s));
  PB_CUDA(cudaMemsetAsync(dja + nnz, 0, sizeof(int) * 8, s));
  PB_CUDA(cudaMemsetAsync(da + nnz, 0, sizeof(double) * 8, s));
  C.nnz_alloc = nnz + 8;
  C.ia_alloc  = nrows + 1 + 8;
  PB_CUDA(cudaMemcpyAsync(dia, ia, sizeof(int) * (size_t)(nrows + 1), cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(dja, ja, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(da, a, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, s));
  C.ia = dia;
  C.ja = dja;
  C.a  = da;
  // long rows (vector kind): tile-ELL when the rows of a tile are of similar length; PERMON_B200_SPMV=vector keeps the lanes-per-row kernel
  if (C.kind == 1 && !rows && nnz >= (1 << 20) && !getenv("PERMON_B200_SPMV") && !getenv("PERMON_B200_NOELL")) PB_CHK(pb::csr_to_tile_ell(C, ia));
  return 0;
}

PetscErrorCode MatCreateSeqAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt i[], PetscInt j[], PetscScalar a[], Mat *mat)
{
  if (comm->size > 1) return MatCreateMPIAIJWithArrays(comm, m, n, PETSC_DECIDE, PETSC_DECIDE, i, j, a, mat);
  PB_CHK(dev_init());
  if (!i || (i[m] > 0 && (!j || !a))) return err(PETSC_ERR_ARG_NULL, "null CSR array");
  PhaseTimer pt("MatCreateSeqAIJWithArrays");
  _p_Mat *A = new _p_Mat;
  A->comm = comm;
  A->kind = MK_AIJ;
  A->m = A->M = m;
  A->n = A->N = n;
  int ierr = upload_csr(A->Ad, m, n, i, j, a, nullptr);
  if (ierr) {
    delete A;
    return ierr;
  }
  // the host arrays belong to the caller and may be pageable: make sure the copies have left them
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  *mat = A;
  return 0;
}

PetscErrorCode MatCreateSeqAIJCUSPARSEWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, const PetscInt di[], const PetscInt dj[], const PetscScalar da[], Mat *mat)
{
  if (comm->size > 1) return err(PETSC_ERR_SUP, "device-array constructor is sequential");
  PB_CHK(dev_init());
  _p_Mat *A = new _p_Mat;
  A->comm = comm;
  A->kind = MK_AIJ;
  A->m = A->M = m;
  A->n = A->N = n;
  A->d_owned  = false;
  std::vector<int> hia((size_t)m + 1);
  PB_CUDA(cudaMemcpy(hia.data(), di, sizeof(int) * (size_t)(m + 1), cudaMemcpyDeviceToHost));
  A->Ad.n = m;
  A->Ad.ncols = n;
  A->Ad.nnz = hia[m];
  A->Ad.ia = di;
  A->Ad.ja = dj;
  A->Ad.a  = da;
  A->Ad.nnz_alloc = hia[m];   // caller-owned arrays: nothing beyond the last entry may be touched
  A->Ad.ia_alloc  = m + 1;
  PB_CHK(spmv_config(A->Ad, hia.data()));
  *mat = A;
  return 0;
}

// whether a row-partitioned constructor first tries the all-stencil form of the diagonal block straight from the caller's arrays (one
// pass, no copy of the block); shared by the host and the device constructor so that both build the same form
static bool windowed_stencil_first(PetscInt m, PetscInt n)
{
  const char *e1 = getenv("PERMON_B200_ST_WINDOWS"), *e2 = getenv("PERMON_B200_PACK_STENCIL");
  return m == n && m >= 64 && !getenv("PERMON_B200_EAGER_SPLIT") && !getenv("PERMON_B200_SPMV") && !(e1 && e1[0] == '0') && !(e2 && e2[0] == '0');
}

// the off-diagonal block from the ghost entries of a row block (row order, storage order within a row): ghost list (sorted unique global
// columns), compressed rows with ghost-buffer columns, and the per-row "has ghosts" flags
static void split_from_ghosts(const pb::OffDiagEntries &off, PetscInt m, std::vector<PetscInt> &gh, std::vector<int> &oia, std::vector<int> &oja,
                            std::vector<double> &oa, std::vector<int> &orow, std::vector<unsigned char> &skip)
{
  skip.assign(std::max<PetscInt>(m, 1), 0);
  gh.assign(off.gcol.begin(), off.gcol.end());
  std::sort(gh.begin(), gh.end());
  gh.erase(std::unique(gh.begin(), gh.end()), gh.end());
  oja.resize(off.row.size());
  oa.assign(off.val.begin(), off.val.end());
  oia.assign(1, 0);
  for (size_t k = 0; k < off.row.size(); k++) {
    if (orow.empty() || orow.back() != off.row[k]) {
      if (!orow.empty()) oia.push_back((int)k);
      orow.push_back(off.row[k]);
      skip[off.row[k]] = 1;
    }
    oja[k] = (int)(std::lower_bound(gh.begin(), gh.end(), (PetscInt)off.gcol[k]) - gh.begin());
  }
  if (!orow.empty()) oia.push_back((int)off.row.size());
}

// the rest of the halo plan once the ghost list (garray) and the off-diagonal rows are known: the widest ghost-free run of rows, the
// neighbours that own the ghosts and, through the host exchange, the send lists (collective).  On a non-symmetric pattern the matrix is
// destroyed on every rank and an error returned.
static int halo_plan_finish(Mat A, const std::vector<int> &orow, const std::vector<int64_t> &cs)
{
  MPI_Comm                     comm = A->comm;
  HaloPlan                    *H = A->halo;
  const int                    size = comm->size, rank = comm->rank;
  const PetscInt               m = A->m, c0 = A->cstart, c1 = A->cstart + A->n;
  const std::vector<PetscInt> &gh = H->garray;
  H->nboundary = (PetscInt)orow.size();
  {   // widest run of interior rows: kernels skip the per-row flag lookup inside it
    int best_lo = 0, best_hi = 0, cur = 0;
    for (int r : orow) {
      if (r - cur > best_hi - best_lo) best_lo = cur, best_hi = r;
      cur = r + 1;
    }
    if ((int)m - cur > best_hi - best_lo) best_lo = cur, best_hi = (int)m;
    H->skip_lo = best_lo;
    H->skip_hi = best_hi;
  }
  // neighbours that own my ghosts
  H->recv_off.push_back(0);
  for (size_t g = 0; g < gh.size();) {
    int owner = (int)(std::upper_bound(cs.begin(), cs.end(), (int64_t)gh[g]) - cs.begin()) - 1;
    size_t e = g;
    while (e < gh.size() && gh[e] < cs[owner + 1]) e++;
    H->neigh.push_back(owner);
    H->recv_off.push_back((PetscInt)e);
    g = e;
  }
  // everybody publishes its ghost list; I pick what I own => my send lists (in the requester's ghost order)
  std::vector<int64_t> gbytes(size);
  if (comm->agi(comm->agctx, (int64_t)(gh.size() * sizeof(PetscInt)), gbytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  int64_t tot = 0;
  for (int r = 0; r < size; r++) tot += gbytes[r];
  std::vector<PetscInt> allg((size_t)(tot / sizeof(PetscInt)) + 1);
  if (comm->agv(comm->agctx, gh.data(), (int64_t)(gh.size() * sizeof(PetscInt)), allg.data(), gbytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  {
    std::vector<PetscInt> sneigh, soff(1, 0), sidx;
    size_t                off = 0;
    for (int r = 0; r < size; r++) {
      size_t cnt = (size_t)(gbytes[r] / sizeof(PetscInt));
      if (r != rank) {
        size_t before = sidx.size();
        for (size_t k = 0; k < cnt; k++) {
          PetscInt g = allg[off + k];
          if (g >= c0 && g < c1) sidx.push_back(g - c0);
        }
        if (sidx.size() > before) {
          sneigh.push_back(r);
          soff.push_back((PetscInt)sidx.size());
        }
      }
      off += cnt;
    }
    // symmetric sparsity is assumed (Hessians are symmetric); every rank must take the same exit, or the others would hang in the next
    // collective: agree on the flag first, then free the object through the normal destructor (halo plan and host split included)
    std::vector<int64_t> oks(size);
    if (comm->agi(comm->agctx, (int64_t)(sneigh == H->neigh), oks.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
    bool all_ok = true;
    for (int r = 0; r < size; r++) all_ok = all_ok && oks[r];
    if (!all_ok) {
      Mat tmp = A;
      MatDestroy(&tmp);
      return err(PETSC_ERR_SUP, "non-symmetric halo pattern (send and receive neighbour sets differ on some rank)");
    }
    H->send_off = soff;
    H->send_idx = sidx;
  }
  return 0;
}

// Row-partitioned AIJ: split into the diagonal block (local columns) and the off-diagonal block (ghost
// columns, compressed rows), and build the halo plan -- the layout of PETSc's Mat_MPIAIJ
// (include/permon/private/petsc/mpiaij.h:49-83: A, B, garray, lvec, Mvctx).
PetscErrorCode MatCreateMPIAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt M, PetscInt N, const PetscInt i[], const PetscInt j[], const PetscScalar a[], Mat *mat)
{
  (void)M;
  (void)N;
  if (n == PETSC_DECIDE) n = m;
  if (comm->size == 1) {
    // one rank: no ghosts possible
    return MatCreateSeqAIJWithArrays(comm, m, n, const_cast<PetscInt *>(i), const_cast<PetscInt *>(j), const_cast<PetscScalar *>(a), mat);
  }
  if (!comm->agi || !comm->agv) return err(PETSC_ERR_ARG_WRONGSTATE, "communicator has no host exchange");
  PhaseTimer pt("MatCreateMPIAIJWithArrays (host split + plan)");
  const int size = comm->size, rank = comm->rank;
  std::vector<int64_t> rows_all(size), cols_all(size);
  if (comm->agi(comm->agctx, m, rows_all.data()) || comm->agi(comm->agctx, n, cols_all.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  std::vector<int64_t> rs(size + 1, 0), cs(size + 1, 0);
  for (int r = 0; r < size; r++) {
    rs[r + 1] = rs[r] + rows_all[r];
    cs[r + 1] = cs[r] + cols_all[r];
  }
  _p_Mat *A = new _p_Mat;
  A->comm   = comm;
  A->kind   = MK_AIJ;
  A->m      = m;
  A->n      = n;
  A->M      = (PetscInt)rs[size];
  A->N      = (PetscInt)cs[size];
  A->rstart = (PetscInt)rs[rank];
  A->cstart = (PetscInt)cs[rank];
  if (A->M <= PB_MAXEQ_ALL && A->M != A->N) {
    // a short and wide matrix: equality rows B_E (qp.c: QPSetEq).  No diagonal / off-diagonal split and no halo plan: the local rows are
    // kept as they came and re-distributed by COLUMNS (the layout of the vectors) when the QPPF or a MatMult first needs them.
    A->eq_host = new _p_Mat::EqHost;
    A->eq_host->ia.assign(i, i + m + 1);
    A->eq_host->ja.assign(j, j + i[m]);
    A->eq_host->a.assign(a, a + i[m]);
    A->Ad.n = m;
    A->Ad.ncols = n;
    A->Ad.nnz = i[m];
    *mat = A;
    return 0;
  }
  const PetscInt c0 = A->cstart, c1 = A->cstart + n;
  const int64_t  nnz = i[m];
  const double   t_s0 = wall_now();
  HaloPlan      *H = new HaloPlan;
  A->halo          = H;
  // pass 1 (host threads: the split is O(nnz) and sits inside the e2e path of multi-GPU runs): per row, how many entries fall into the
  // diagonal block / outside it, and which columns outside it occur (the ghosts)
  H->host = new HaloPlan::HostSplit;
  std::vector<int>       &dia = H->host->dia, &oia = H->host->oia, &oja = H->host->oja, &orow = H->host->orow;
  std::vector<double>    &oa = H->host->oa;
  HaloPlan::UVec<int>    &dja = H->host->dja;
  HaloPlan::UVec<double> &da = H->host->da;
  std::vector<unsigned char> &skip = H->host->skip;
  std::vector<PetscInt>       gh;
  double t_s1 = t_s0;
  // Fast path: the diagonal block of a constant-coefficient stencil goes straight from the caller's arrays (global columns) into the
  // all-stencil form -- one pass, no intermediate copy of the block; the ghost entries fall out of the same pass.
  bool fast = false;
  {
    if (windowed_stencil_first(m, n)) {
      pb::OffDiagEntries off;
      int64_t            nd = 0;
      PB_CHK(pb::pk_stencil_windowed((int)m, i, j, a, (int)c0, (int)n, H->host->st, off, nd));
      if (H->host->st.valid) {
        fast = true;
        t_s1 = wall_now();
        H->host->nnz_diag = nd;
        H->host->ui = i;
        H->host->uj = j;
        H->host->ua = a;
        H->host->c0 = c0;
        split_from_ghosts(off, m, gh, oia, oja, oa, orow, skip);
        H->garray = gh;
      }
    }
  }
  if (!fast) {
  dia.assign(m + 1, 0);
  skip.assign(std::max<PetscInt>(m, 1), 0);
  std::vector<int>      ocnt(m + 1, 0);
  {
    std::vector<std::vector<PetscInt>> part;
#pragma omp parallel
    {
#pragma omp single
      part.resize(omp_get_num_threads());
      std::vector<PetscInt> &mine = part[omp_get_thread_num()];
#pragma omp for schedule(static)
      for (PetscInt r = 0; r < m; r++) {
        int nd = 0, no = 0;
        for (PetscInt k = i[r]; k < i[r + 1]; k++) {
          if (j[k] >= c0 && j[k] < c1) {
            nd++;
          } else {
            no++;
            mine.push_back(j[k]);
          }
        }
        dia[r + 1]  = nd;
        ocnt[r + 1] = no;
        skip[r]     = no > 0;
      }
      std::sort(mine.begin(), mine.end());
      mine.erase(std::unique(mine.begin(), mine.end()), mine.end());
    }
    for (auto &v : part) gh.insert(gh.end(), v.begin(), v.end());
  }
  std::sort(gh.begin(), gh.end());
  gh.erase(std::unique(gh.begin(), gh.end()), gh.end());
  H->garray = gh;
  t_s1 = wall_now();
  // prefix sums, then pass 2 fills both blocks
  for (PetscInt r = 0; r < m; r++) {
    dia[r + 1] += dia[r];
    ocnt[r + 1] += ocnt[r];
  }
  dja.resize(dia[m]);
  da.resize(dia[m]);
  oja.resize(ocnt[m]);
  oa.resize(ocnt[m]);
  for (PetscInt r = 0; r < m; r++)
    if (skip[r]) orow.push_back(r);
  oia.assign(orow.size() + 1, 0);
  for (size_t q = 0; q < orow.size(); q++) oia[q + 1] = ocnt[orow[q] + 1];
#pragma omp parallel for schedule(static)
  for (PetscInt r = 0; r < m; r++) {
    int pd = dia[r], po = ocnt[r];
    for (PetscInt k = i[r]; k < i[r + 1]; k++) {
      if (j[k] >= c0 && j[k] < c1) {
        dja[pd] = j[k] - c0;
        da[pd++] = a[k];
      } else {
        oja[po] = (int)(std::lower_bound(gh.begin(), gh.end(), j[k]) - gh.begin());
        oa[po++] = a[k];
      }
    }
  }
  }
  const double t_s2 = wall_now();
  PB_CHK(halo_plan_finish(A, orow, cs));
  if (verbose_timing())
    fprintf(stderr, "[permon_b200] rank %d host split of %d rows / %lld nnz: count + ghosts %.1f ms, fill %.1f ms, plan exchange %.1f ms\n", rank, (int)m,
            (long long)nnz, 1e3 * (t_s1 - t_s0), 1e3 * (t_s2 - t_s1), 1e3 * (wall_now() - t_s2));
  A->Ad.n = m;   // sizes are known; the arrays reach the device on first use (mat_ensure_device)
  A->Ad.ncols = n;
  A->Ad.nnz = fast ? H->host->nnz_diag : (int64_t)dja.size();
  *mat = A;
  return 0;
}

// Peer-memory halo: every rank allocates a ghost window (ghosts of p, ghosts of x, one flag per neighbour and vector),
// publishes its IPC handle + neighbour table, and resolves where in each neighbour's window its own boundary values go.
struct HaloExch {
  cudaIpcMemHandle_t h;
  int                nneigh, ng_pad;
  int                neigh[PB_MAXNEIGH];
  int                recv_off[PB_MAXNEIGH + 1];
};
static int halo_p2p_setup(Mat A)
{
  HaloPlan *H = A->halo;
  MPI_Comm  c = A->comm;
  const int size = c->size, rank = c->rank;
  int       ok = ((int)H->neigh.size() <= PB_MAXNEIGH);
  const int ng = (int)H->garray.size(), ng_pad = ((ng + 15) / 16) * 16 + 16;
  const size_t gbytes = sizeof(double) * 2 * (size_t)ng_pad, fbytes = sizeof(unsigned long long) * 2 * PB_MAXNEIGH * PB_FLAG_STRIDE;
  PB_CUDA(cudaMalloc(&H->gwin, gbytes + fbytes));
  PB_CUDA(cudaMemset(H->gwin, 0, gbytes + fbytes));
  PB_CUDA(cudaDeviceSynchronize());
  HaloExch me;
  memset(&me, 0, sizeof me);
  if (cudaIpcGetMemHandle(&me.h, H->gwin) != cudaSuccess) ok = 0;
  me.nneigh = ok ? (int)H->neigh.size() : 0;
  me.ng_pad = ng_pad;
  for (int q = 0; q < me.nneigh; q++) me.neigh[q] = H->neigh[q];
  for (int q = 0; q <= me.nneigh; q++) me.recv_off[q] = H->recv_off[q];
  std::vector<HaloExch> all(size);
  std::vector<int64_t>  bytes(size, (int64_t)sizeof(HaloExch));
  if (c->agv(c->agctx, &me, sizeof me, all.data(), bytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  H->peer_gwins.assign(H->neigh.size(), nullptr);
  for (int w = 0; w < 2; w++) {
    H->push[w]          = HaloPush();
    H->push[w].nneigh   = (int)H->neigh.size();
    H->push[w].total    = (int)H->send_idx.size();
    H->push[w].send_idx = H->d_send_idx;
    for (size_t q = 0; q <= H->neigh.size() && q <= PB_MAXNEIGH; q++) H->push[w].send_off[q] = H->send_off[q];
  }
  for (size_t iq = 0; iq < H->neigh.size() && ok; iq++) {
    const int       q = H->neigh[iq];
    const HaloExch &E = all[q];
    int             jq = -1;
    for (int t = 0; t < E.nneigh; t++)
      if (E.neigh[t] == rank) jq = t;
    if (jq < 0 || E.recv_off[jq + 1] - E.recv_off[jq] != H->send_off[iq + 1] - H->send_off[iq]) {
      ok = 0;
      break;
    }
    if (cudaIpcOpenMemHandle(&H->peer_gwins[iq], E.h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      ok = 0;
      break;
    }
    char *base = (char *)H->peer_gwins[iq];
    for (int w = 0; w < 2; w++) {
      H->push[w].dst[iq]  = (double *)base + (size_t)w * E.ng_pad + E.recv_off[jq];
      H->push[w].flag[iq] = (unsigned long long *)(base + sizeof(double) * 2 * (size_t)E.ng_pad) + ((size_t)w * PB_MAXNEIGH + jq) * PB_FLAG_STRIDE;
    }
  }
  std::vector<int64_t> oks(size);
  if (c->agi(c->agctx, ok, oks.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  for (int q = 0; q < size; q++) ok = ok && oks[q];
  if (!ok) {
    H->p2p = false;
    return 0;
  }
  unsigned *cnt;
  PB_CUDA(cudaMalloc(&cnt, 2 * sizeof(unsigned)));
  PB_CUDA(cudaMemset(cnt, 0, 2 * sizeof(unsigned)));
  for (int w = 0; w < 2; w++) {
    H->push[w].counter = cnt + w;
    H->d_ghost2[w]     = (double *)H->gwin + (size_t)w * ng_pad;
    H->my_hflags[w]    = (unsigned long long *)((char *)H->gwin + gbytes) + (size_t)w * PB_MAXNEIGH * PB_FLAG_STRIDE;
  }
  // contiguous pack lists (slab partitions): the producing kernels can push the boundary values themselves
  H->contig = true;
  H->send_lo.assign(H->neigh.size(), 0);
  for (size_t q = 0; q < H->neigh.size(); q++) {
    const PetscInt a = H->send_off[q], b = H->send_off[q + 1];
    H->send_lo[q] = (b > a) ? H->send_idx[a] : 0;
    for (PetscInt k = a + 1; k < b; k++)
      if (H->send_idx[k] != H->send_idx[k - 1] + 1) H->contig = false;
  }
  if (H->contig) {
    PushRanges R[2];
    for (int w = 0; w < 2; w++) {
      R[w].n = (int)H->neigh.size();
      for (int q = 0; q < R[w].n; q++) {
        R[w].lo[q]   = H->send_lo[q];
        R[w].hi[q]   = H->send_lo[q] + (H->send_off[q + 1] - H->send_off[q]);
        R[w].dst[q]  = H->push[w].dst[q];
        R[w].flag[q] = H->push[w].flag[q];
      }
      R[w].counter = H->push[w].counter;
      // widest run of rows that no range covers: the kernels' cheap "interior" test
      std::vector<std::pair<int, int>> iv;
      for (int q = 0; q < R[w].n; q++)
        if (R[w].hi[q] > R[w].lo[q]) iv.push_back({R[w].lo[q], R[w].hi[q]});
      std::sort(iv.begin(), iv.end());
      int best_lo = 0, best_hi = 0, cur = 0;
      for (auto &I : iv) {
        if (I.first - cur > best_hi - best_lo) best_lo = cur, best_hi = I.first;
        cur = std::max(cur, I.second);
      }
      if ((int)A->m - cur > best_hi - best_lo) best_lo = cur, best_hi = (int)A->m;
      R[w].gap_lo = best_lo;
      R[w].gap_hi = best_hi;
    }
    PB_CUDA(cudaMalloc(&H->d_ranges, sizeof R));
    PB_CUDA(cudaMemcpy(H->d_ranges, R, sizeof R, cudaMemcpyHostToDevice));
  }
  H->p2p = true;
  return 0;
}

// device side of the halo plan: send list, row map of the ghost rows, events (the off-diagonal rows `orow` of the split)
static int halo_device_setup(Mat A, const std::vector<int> &orow)
{
  HaloPlan      *H = A->halo;
  const PetscInt m = A->m;
  PB_CHK(dmalloc(&H->d_send_idx, std::max<size_t>(H->send_idx.size(), 1)));
  PB_CHK(dmalloc(&H->d_send, std::max<size_t>(H->send_idx.size(), 1)));
  PB_CHK(dmalloc(&H->d_ghost, std::max<size_t>(H->garray.size(), 1)));
  // rows outside the ghost-free run [skip_lo, skip_hi) -> their row in the compressed off-diagonal block (GhostMerge)
  std::vector<int> row_map((size_t)std::max<PetscInt>(H->skip_lo + (m - H->skip_hi), 1), -1);
  for (size_t q = 0; q < orow.size(); q++) {
    const int r = orow[q];
    row_map[r < H->skip_lo ? r : r - H->skip_hi + H->skip_lo] = (int)q;
  }
  PB_CHK(dmalloc(&H->d_row_map, row_map.size()));
  PB_CUDA(cudaMemcpyAsync(H->d_send_idx, H->send_idx.data(), sizeof(int) * H->send_idx.size(), cudaMemcpyHostToDevice, ctx().stream));
  PB_CUDA(cudaMemcpyAsync(H->d_row_map, row_map.data(), sizeof(int) * row_map.size(), cudaMemcpyHostToDevice, ctx().stream));
  PB_CUDA(cudaEventCreateWithFlags(&H->ev_packed, cudaEventDisableTiming));
  PB_CUDA(cudaEventCreateWithFlags(&H->ev_arrived, cudaEventDisableTiming));
  PB_CUDA(cudaEventCreateWithFlags(&H->ev_consumed, cudaEventDisableTiming));
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  return 0;
}

// First use of a dense matrix: a device array whose base is 16-byte aligned and whose lda is even (every column start 16-byte aligned,
// what the bulk copies of k_dense need) is adopted as it is; anything else -- host arrays, odd lda, offset device pointers -- goes into
// one library-owned device copy with an even lda.
static int dense_ensure_device(Mat A)
{
  if (A->dn_ready) return 0;
  PB_CHK(dev_init());
  PhaseTimer     pt("dense matrix: adopt / upload");
  cudaStream_t   s = ctx().stream;
  const int64_t  m = A->m, n = A->n, lda = A->dn_src_lda;
  pb::CsrDev    &C = A->Ad;
  C.n     = (int)m;
  C.ncols = (int)n;
  C.nnz   = m * n;
  if (A->dn_src_dev && (((uintptr_t)A->dn_src) & 15) == 0 && lda % 2 == 0) {
    C.dn_a        = A->dn_src;
    C.dn_lda      = lda;
    A->dn_adopted = true;
  } else {
    const int64_t ldp = (m + 1) / 2 * 2;
    PB_CHK(dmalloc(&A->dn_own, (size_t)std::max<int64_t>(ldp * n, 1)));
    if (m > 0 && n > 0)
      PB_CUDA(cudaMemcpy2DAsync(A->dn_own, (size_t)ldp * 8, A->dn_src, (size_t)lda * 8, (size_t)m * 8, (size_t)n,
                                A->dn_src_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
    if (ldp > m && n > 0) PB_CUDA(cudaMemset2DAsync(A->dn_own + m, (size_t)ldp * 8, 0, 8, (size_t)n, s));   // the pad row is never summed
    PB_CUDA(cudaStreamSynchronize(s));   // the host array may be pageable and may change after this call
    C.dn_a   = A->dn_own;
    C.dn_lda = ldp;
  }
  pb::dense_config(C);
  if (C.dn_split > 0) PB_CHK(dmalloc(&C.dn_part, (size_t)std::max<int64_t>(m * ((n + C.dn_split - 1) / C.dn_split), 1)));
  A->dn_ready = true;
  return 0;
}

namespace pb {
int mat_ensure_device(Mat A)
{
  if (A->kind == MK_PROD) {
    PB_CHK(mat_ensure_device(A->M1));
    return mat_ensure_device(A->M2);
  }
  if (A->kind == MK_PENALIZED) return mat_ensure_device(A->A);
  if (A->kind == MK_DENSE) return dense_ensure_device(A);
  if (A->kind != MK_AIJ || !A->halo || !A->halo->host) return 0;
  HaloPlan            *H = A->halo;
  HaloPlan::HostSplit *S = H->host;
  PB_CHK(dev_init());
  PhaseTimer pt("mat_ensure_device (pack + upload + halo set-up)");
  const PetscInt m = A->m;
  if (S->st.valid) {
    A->Ad.n     = m;
    A->Ad.ncols = A->n;
    A->Ad.nnz   = S->nnz_diag;
    PB_CHK(upload_stencil(A->Ad, S->st, S->nnz_diag, 0.0));
  } else {
    PB_CHK(upload_csr(A->Ad, m, A->n, S->dia.data(), S->dja.data(), S->da.data(), nullptr));
  }
  PB_CHK(upload_csr(A->Ao, (int)S->orow.size(), (int)H->garray.size(), S->oia.data(), S->oja.data(), S->oa.data(), S->orow.data()));
  PB_CHK(halo_device_setup(A, S->orow));
  delete S;
  H->host = nullptr;
  if (A->comm->p2p) PB_CHK(halo_p2p_setup(A));
  return 0;
}
}  // namespace pb

PetscErrorCode MatB200GetHaloInfo(Mat A, PetscInt *nghost, const PetscInt **garray, PetscInt *nneigh, const PetscInt **neigh_rank, const PetscInt **recv_off,
                                  const PetscInt **send_off, const PetscInt **send_idx, PetscInt *nboundary_rows)
{
  static const PetscInt zero = 0;
  HaloPlan             *H = A->halo;
  if (nghost) *nghost = H ? (PetscInt)H->garray.size() : 0;
  if (garray) *garray = H ? H->garray.data() : nullptr;
  if (nneigh) *nneigh = H ? (PetscInt)H->neigh.size() : 0;
  if (neigh_rank) *neigh_rank = H ? H->neigh.data() : nullptr;
  if (recv_off) *recv_off = H ? H->recv_off.data() : &zero;
  if (send_off) *send_off = H ? H->send_off.data() : &zero;
  if (send_idx) *send_idx = H ? H->send_idx.data() : nullptr;
  if (nboundary_rows) *nboundary_rows = H ? H->nboundary : 0;
  return 0;
}

PetscErrorCode MatB200GetHostSplit(Mat A, const PetscInt **dia, const PetscInt **dja, const PetscScalar **da, PetscInt *noffrows, const PetscInt **oia,
                                   const PetscInt **oja, const PetscScalar **oa, const PetscInt **orow)
{
  if (!A || A->kind != MK_AIJ || !A->halo || !A->halo->host) return err(PETSC_ERR_ARG_WRONGSTATE, "no host split (sequential matrix, or already on the device)");
  HaloPlan::HostSplit *S = A->halo->host;
  if (S->st.valid && S->dia.empty()) {
    // fast path: the diagonal-block copy was never made; rebuild it from the arrays the matrix was created from (this accessor is a
    // test hook: it must be called while those arrays are still alive)
    const PetscInt m = A->m, c0 = S->c0, c1 = S->c0 + A->n;
    S->dia.assign((size_t)m + 1, 0);
    for (PetscInt r = 0; r < m; r++) {
      int nd = 0;
      for (PetscInt k = S->ui[r]; k < S->ui[r + 1]; k++) nd += (S->uj[k] >= c0 && S->uj[k] < c1);
      S->dia[(size_t)r + 1] = S->dia[(size_t)r] + nd;
    }
    S->dja.resize((size_t)S->dia[(size_t)m]);
    S->da.resize((size_t)S->dia[(size_t)m]);
    for (PetscInt r = 0, p = 0; r < m; r++)
      for (PetscInt k = S->ui[r]; k < S->ui[r + 1]; k++)
        if (S->uj[k] >= c0 && S->uj[k] < c1) {
          S->dja[(size_t)p] = S->uj[k] - c0;
          S->da[(size_t)p++] = S->ua[k];
        }
  }
  if (dia) *dia = S->dia.data();
  if (dja) *dja = S->dja.data();
  if (da) *da = S->da.data();
  if (noffrows) *noffrows = (PetscInt)S->orow.size();
  if (oia) *oia = S->oia.data();
  if (oja) *oja = S->oja.data();
  if (oa) *oa = S->oa.data();
  if (orow) *orow = S->orow.data();
  return 0;
}

PetscErrorCode MatB200GetStorageInfo(Mat A, PetscInt *kind, PetscReal *stream_bytes, PetscInt *coded_tiles, PetscInt *tiles)
{
  if (!A || (A->kind != MK_AIJ && A->kind != MK_DENSE)) return err(PETSC_ERR_ARG_WRONG, "MatB200GetStorageInfo: AIJ or dense matrix expected");
  PB_CHK(pb::mat_ensure_device(A));
  if (A->kind == MK_DENSE) {
    if (kind) *kind = A->Ad.kind;
    if (stream_bytes) *stream_bytes = pb::csr_stream_bytes(A->Ad);
    if (coded_tiles) *coded_tiles = 0;
    if (tiles) *tiles = A->Ad.dn_rpb ? (A->Ad.n + A->Ad.dn_rpb - 1) / A->Ad.dn_rpb : 0;   // row blocks
    return 0;
  }
  if (kind) *kind = A->Ad.kind;
  if (stream_bytes) *stream_bytes = pb::csr_stream_bytes(A->Ad) + (A->halo ? pb::csr_stream_bytes(A->Ao) : 0.0);
  if (coded_tiles) *coded_tiles = (PetscInt)A->Ad.pk_coded;
  if (tiles) *tiles = (A->Ad.n + pb::TR - 1) / pb::TR;
  return 0;
}

static int check_device_array(const void *p, const char *what)
{
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return err(PETSC_ERR_ARG_WRONG, "%s: not a CUDA pointer", what);
  }
  if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) return err(PETSC_ERR_ARG_WRONG, "%s: host memory, a device pointer is required", what);
  if (at.device != ctx().device) return err(PETSC_ERR_ARG_WRONG, "%s: memory of device %d, the library runs on device %d", what, at.device, ctx().device);
  return 0;
}

// Row-partitioned (or one-rank) AIJ from a CSR in device memory, re-coded on the device into the form upload_csr builds from a host CSR
// (recode.cu).  On several ranks the split into the diagonal and off-diagonal block runs on the device too; only the ghost entries reach
// the host, where the halo plan is built exactly as for MatCreateMPIAIJWithArrays.  Nothing of the caller's arrays is kept.
PetscErrorCode MatB200CreateAIJWithDeviceArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt M, PetscInt N, const PetscInt di[], const PetscInt dj[],
                                                const PetscScalar da[], Mat *mat)
{
  (void)M;
  (void)N;
  if (!mat) return err(PETSC_ERR_ARG_NULL, "null Mat pointer");
  if (n == PETSC_DECIDE) n = m;
  if (!di) return err(PETSC_ERR_ARG_NULL, "null row pointer");
  PB_CHK(dev_init());
  PB_CHK(check_device_array(di, "row pointer"));
  cudaStream_t s   = ctx().stream;
  int          nnz = 0;
  PB_CUDA(cudaMemcpyAsync(&nnz, di + m, sizeof(int), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  if (nnz > 0) {
    if (!dj || !da) return err(PETSC_ERR_ARG_NULL, "null CSR array");
    PB_CHK(check_device_array(dj, "column ids"));
    PB_CHK(check_device_array(da, "values"));
  }
  PhaseTimer pt("MatB200CreateAIJWithDeviceArrays");
  if (comm->size == 1) {
    _p_Mat *A = new _p_Mat;
    A->comm   = comm;
    A->kind   = MK_AIJ;
    A->m = A->M = m;
    A->n = A->N = n;
    int ierr = pb::recode_csr_dev(A->Ad, m, n, di, dj, da);
    if (!ierr) ierr = cudaStreamSynchronize(s) == cudaSuccess ? 0 : err(PETSC_ERR_GPU, "%s", cudaGetErrorString(cudaGetLastError()));
    if (ierr) {
      delete A;
      return ierr;
    }
    *mat = A;
    return 0;
  }
  if (!comm->agi || !comm->agv) return err(PETSC_ERR_ARG_WRONGSTATE, "communicator has no host exchange");
  const int            size = comm->size, rank = comm->rank;
  std::vector<int64_t> rows_all(size), cols_all(size);
  if (comm->agi(comm->agctx, m, rows_all.data()) || comm->agi(comm->agctx, n, cols_all.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  std::vector<int64_t> rs(size + 1, 0), cs(size + 1, 0);
  for (int r = 0; r < size; r++) {
    rs[r + 1] = rs[r] + rows_all[r];
    cs[r + 1] = cs[r] + cols_all[r];
  }
  _p_Mat *A = new _p_Mat;
  A->comm   = comm;
  A->kind   = MK_AIJ;
  A->m      = m;
  A->n      = n;
  A->M      = (PetscInt)rs[size];
  A->N      = (PetscInt)cs[size];
  A->rstart = (PetscInt)rs[rank];
  A->cstart = (PetscInt)cs[rank];
  if (A->M <= PB_MAXEQ_ALL && A->M != A->N) {
    // equality rows (at most PB_MAXEQ_ALL in all): kept on the host like MatCreateMPIAIJWithArrays keeps them
    A->eq_host = new _p_Mat::EqHost;
    A->eq_host->ia.resize((size_t)m + 1);
    A->eq_host->ja.resize((size_t)nnz);
    A->eq_host->a.resize((size_t)nnz);
    PB_CUDA(cudaMemcpyAsync(A->eq_host->ia.data(), di, sizeof(int) * ((size_t)m + 1), cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaMemcpyAsync(A->eq_host->ja.data(), dj, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaMemcpyAsync(A->eq_host->a.data(), da, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaStreamSynchronize(s));
    A->Ad.n     = m;
    A->Ad.ncols = n;
    A->Ad.nnz   = nnz;
    *mat        = A;
    return 0;
  }
  HaloPlan *H = new HaloPlan;
  A->halo     = H;
  auto fail = [&](int ierr) {
    Mat tmp = A;
    MatDestroy(&tmp);
    return ierr;
  };
  // the diagonal block: all-stencil straight from the caller's arrays when the host constructor would try that too (same rule), else
  // a device split into a library-owned CSR with local columns that goes through the general re-coder (and is adopted if it stays CSR)
  bool st_done = false;
  int  ierr    = 0;
  if (windowed_stencil_first(m, n)) ierr = pb::recode_stencil_window_dev(A->Ad, (int)m, di, dj, da, (int)A->cstart, (int)n, &st_done);
  int               *sia = nullptr, *sja = nullptr;
  double            *sa  = nullptr;
  pb::OffDiagEntries off;
  if (!ierr) ierr = pb::split_rows_dev((int)m, di, dj, da, (int)A->cstart, (int)n, !st_done, &sia, &sja, &sa, off);
  if (!ierr && !st_done) ierr = pb::recode_csr_dev(A->Ad, m, n, sia, sja, sa, &sia, &sja, &sa);
  dfree(sia);
  dfree(sja);
  dfree(sa);
  if (ierr) return fail(ierr);
  std::vector<int>           oia, oja, orow;
  std::vector<double>        oa;
  std::vector<unsigned char> skip;
  std::vector<PetscInt>      gh;
  split_from_ghosts(off, m, gh, oia, oja, oa, orow, skip);
  H->garray = gh;
  PB_CHK(halo_plan_finish(A, orow, cs));   // destroys A itself on a non-symmetric pattern
  ierr = upload_csr(A->Ao, (int)orow.size(), (int)H->garray.size(), oia.data(), oja.data(), oa.data(), orow.data());
  if (!ierr) ierr = halo_device_setup(A, orow);
  if (!ierr && comm->p2p) ierr = halo_p2p_setup(A);
  if (!ierr && cudaStreamSynchronize(s) != cudaSuccess) ierr = err(PETSC_ERR_GPU, "%s", cudaGetErrorString(cudaGetLastError()));
  if (ierr) return fail(ierr);
  *mat = A;
  return 0;
}

// ---- dense matrices (MATSEQDENSE / MATSEQDENSECUDA): column-major, entry (i, j) at data[i + j * lda], lda = m until MatDenseSetLDA --------
static int dense_create(MPI_Comm comm, PetscInt m, PetscInt n, const PetscScalar *data, bool dev, Mat *mat)
{
  if (!mat) return err(PETSC_ERR_ARG_NULL, "null Mat pointer");
  if (m < 0 || n < 0) return err(PETSC_ERR_ARG_OUTOFRANGE, "dense matrix: negative size %d x %d", (int)m, (int)n);
  if (!data) return err(PETSC_ERR_ARG_NULL, "dense matrix: null data array");
  if (comm->size > 1) return err(PETSC_ERR_SUP, "dense matrices run on one rank (a %d-rank communicator was given)", comm->size);
  if (dev) {
    PB_CHK(dev_init());
    PB_CHK(check_device_array(data, "dense matrix values"));
  }
  _p_Mat *A     = new _p_Mat;
  A->comm       = comm;
  A->kind       = MK_DENSE;
  A->m = A->M   = m;
  A->n = A->N   = n;
  A->dn_src     = data;
  A->dn_src_lda = m > 0 ? m : 1;
  A->dn_src_dev = dev;
  *mat          = A;
  return 0;
}
PetscErrorCode MatCreateSeqDense(MPI_Comm comm, PetscInt m, PetscInt n, PetscScalar data[], Mat *A) { return dense_create(comm, m, n, data, false, A); }
PetscErrorCode MatCreateSeqDenseCUDA(MPI_Comm comm, PetscInt m, PetscInt n, PetscScalar data[], Mat *A) { return dense_create(comm, m, n, data, true, A); }
PetscErrorCode MatCreateDense(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt M, PetscInt N, PetscScalar data[], Mat *A)
{
  if (comm->size > 1) return err(PETSC_ERR_SUP, "MatCreateDense: dense matrices run on one rank (a %d-rank communicator was given)", comm->size);
  if (m == PETSC_DECIDE) m = M;
  if (n == PETSC_DECIDE) n = N;
  if ((M != PETSC_DECIDE && M != m) || (N != PETSC_DECIDE && N != n))
    return err(PETSC_ERR_ARG_SIZ, "MatCreateDense: local size %d x %d differs from global %d x %d on one rank", (int)m, (int)n, (int)M, (int)N);
  return dense_create(comm, m, n, data, false, A);
}
PetscErrorCode MatDenseSetLDA(Mat A, PetscInt lda)
{
  if (!A || A->kind != MK_DENSE) return err(PETSC_ERR_ARG_WRONG, "MatDenseSetLDA: dense matrix expected");
  if (A->dn_ready) return err(PETSC_ERR_ARG_WRONGSTATE, "MatDenseSetLDA: the matrix has already been used");
  if (lda < A->m || lda < 1) return err(PETSC_ERR_ARG_OUTOFRANGE, "MatDenseSetLDA: lda %d < %d rows", (int)lda, (int)A->m);
  A->dn_src_lda = lda;
  return 0;
}
PetscErrorCode MatDenseGetLDA(Mat A, PetscInt *lda)
{
  if (!A || A->kind != MK_DENSE) return err(PETSC_ERR_ARG_WRONG, "MatDenseGetLDA: dense matrix expected");
  if (!lda) return err(PETSC_ERR_ARG_NULL, "null lda pointer");
  *lda = (PetscInt)A->dn_src_lda;
  return 0;
}
PetscErrorCode MatB200GetDenseInfo(Mat A, int64_t *lda, PetscBool *adopted, PetscInt *rows_per_block, PetscInt *split_columns)
{
  if (!A || A->kind != MK_DENSE) return err(PETSC_ERR_ARG_WRONG, "MatB200GetDenseInfo: dense matrix expected");
  PB_CHK(pb::mat_ensure_device(A));
  if (lda) *lda = A->Ad.dn_lda;
  if (adopted) *adopted = A->dn_adopted ? PETSC_TRUE : PETSC_FALSE;
  if (rows_per_block) *rows_per_block = A->Ad.dn_rpb;
  if (split_columns) *split_columns = A->Ad.dn_split;
  return 0;
}

PetscErrorCode MatB200GetStoredForm(Mat A, PetscInt part, void *buf, size_t *nbytes)
{
  if (!A || A->kind != MK_AIJ) return err(PETSC_ERR_ARG_WRONG, "MatB200GetStoredForm: AIJ matrix expected");
  if (!nbytes) return err(PETSC_ERR_ARG_NULL, "null size pointer");
  const int block = (int)(part / MATB200_FORM_OFFDIAG), field = (int)(part % MATB200_FORM_OFFDIAG);
  if (part < 0 || block > 1) return err(PETSC_ERR_ARG_OUTOFRANGE, "MatB200GetStoredForm: unknown part %d", (int)part);
  if (!A->eq_host) PB_CHK(pb::mat_ensure_device(A));
  static const pb::CsrDev none;
  const pb::CsrDev       &C = block == 0 ? A->Ad : (A->halo ? A->Ao : none);
  const size_t            ntiles = (size_t)(C.n + pb::TR - 1) / pb::TR;
  const void             *src = nullptr;
  bool                    host = false;
  size_t                  sz = 0;
  int64_t                 sc[15];
  switch (field) {
  case MATB200_FORM_SCALARS: {
    const int64_t v[15] = {C.kind, C.n, C.ncols, C.nnz, C.st_npat, C.st_nwin, C.st_lmax, C.st_dlo, C.st_dhi, C.pk_max, C.pk_bytes, C.pk_coded, C.stages, C.tile_cap, C.W};
    memcpy(sc, v, sizeof sc);
    src  = sc;
    host = true;
    sz   = sizeof sc;
    break;
  }
  case MATB200_FORM_ST_MASKS: src = C.st_masks, sz = C.st_masks ? ntiles * pb::TR : 0; break;
  case MATB200_FORM_ST_PID: src = C.st_pid, sz = C.st_pid ? ntiles : 0; break;
  case MATB200_FORM_ST_PATS: src = C.st_pats, sz = C.st_pats ? sizeof(pb::StPattern) * (size_t)C.st_npat : 0; break;
  case MATB200_FORM_PK_BLOB:
    src = C.pk;
    if (C.pk) {
      unsigned last = 0;
      PB_CUDA(cudaMemcpy(&last, C.pk_off + ntiles, sizeof last, cudaMemcpyDeviceToHost));
      sz = (size_t)last * 16 + 16;
    }
    break;
  case MATB200_FORM_PK_OFF: src = C.pk_off, sz = C.pk_off ? sizeof(unsigned) * (ntiles + 1) : 0; break;
  case MATB200_FORM_CSR_IA:
  case MATB200_FORM_CSR_JA:
  case MATB200_FORM_CSR_A:
    if (block == 0 && A->eq_host) {
      host = true;
      if (field == MATB200_FORM_CSR_IA) src = A->eq_host->ia.data(), sz = sizeof(int) * A->eq_host->ia.size();
      if (field == MATB200_FORM_CSR_JA) src = A->eq_host->ja.data(), sz = sizeof(int) * A->eq_host->ja.size();
      if (field == MATB200_FORM_CSR_A) src = A->eq_host->a.data(), sz = sizeof(double) * A->eq_host->a.size();
    } else {
      if (field == MATB200_FORM_CSR_IA) src = C.ia, sz = C.ia ? sizeof(int) * ((size_t)C.n + 1) : 0;
      if (field == MATB200_FORM_CSR_JA) src = C.ja, sz = C.ja ? sizeof(int) * (size_t)C.nnz : 0;
      if (field == MATB200_FORM_CSR_A) src = C.a, sz = C.a ? sizeof(double) * (size_t)C.nnz : 0;
    }
    break;
  case MATB200_FORM_ELL_VAL: src = C.ell_val, sz = C.ell_val ? sizeof(double) * (size_t)C.ell_elems : 0; break;
  case MATB200_FORM_ELL_COL: src = C.ell_col, sz = C.ell_col ? sizeof(int) * (size_t)C.ell_elems : 0; break;
  case MATB200_FORM_ELL_LEN: src = C.ell_len, sz = C.ell_len ? sizeof(int) * (size_t)C.n : 0; break;
  case MATB200_FORM_ELL_LT: src = C.ell_lt, sz = C.ell_lt ? sizeof(int) * ntiles : 0; break;
  case MATB200_FORM_ELL_OFF: src = C.ell_off, sz = C.ell_off ? sizeof(int64_t) * ntiles : 0; break;
  case MATB200_FORM_ROWS: src = C.rows, sz = C.rows ? sizeof(int) * (size_t)C.n : 0; break;
  default: return err(PETSC_ERR_ARG_OUTOFRANGE, "MatB200GetStoredForm: unknown part %d", (int)part);
  }
  if (!buf) {
    *nbytes = sz;
    return 0;
  }
  if (*nbytes < sz) return err(PETSC_ERR_ARG_SIZ, "MatB200GetStoredForm: buffer of %zu bytes, %zu needed", *nbytes, sz);
  if (sz) {
    if (host) memcpy(buf, src, sz);
    else {
      PB_CUDA(cudaStreamSynchronize(ctx().stream));
      PB_CUDA(cudaMemcpy(buf, src, sz, cudaMemcpyDeviceToHost));
    }
  }
  *nbytes = sz;
  return 0;
}

PetscErrorCode PermonB200PackTiles(PetscInt n, const PetscInt ia[], const PetscInt ja[], const PetscScalar a[], unsigned char **blob, unsigned **tile_off,
                                   PetscInt *ntiles, PetscInt *coded_tiles)
{
  if (!ia || !blob || !tile_off) return err(PETSC_ERR_ARG_NULL, "null argument");
  pb::RawBuf            b;
  std::vector<unsigned> off;
  int                        max_tile = 0;
  int64_t                    ncoded = 0;
  bool                       packed = false;
  PB_CHK(pb::pk_build(n, ia, ja, a, b, off, max_tile, ncoded, packed, nullptr, true));
  *blob     = nullptr;
  *tile_off = nullptr;
  if (ntiles) *ntiles = (n + pb::TR - 1) / pb::TR;
  if (coded_tiles) *coded_tiles = (PetscInt)ncoded;
  if (!packed) return 0;
  *blob     = (unsigned char *)malloc(b.size());
  *tile_off = (unsigned *)malloc(sizeof(unsigned) * off.size());
  if (!*blob || !*tile_off) return err(PETSC_ERR_MEM, "out of memory");
  memcpy(*blob, b.data(), b.size());
  memcpy(*tile_off, off.data(), sizeof(unsigned) * off.size());
  return 0;
}

PetscErrorCode PermonB200PackFree(unsigned char *blob, unsigned *tile_off)
{
  free(blob);
  free(tile_off);
  return 0;
}

// MatCreateOneRow: src/mat/impls/onerow/onerow.c:97-113
PetscErrorCode MatCreateOneRow(Vec a, Mat *A_new)
{
  _p_Mat *A = new _p_Mat;
  A->comm = a->comm;
  A->kind = MK_ONEROW;
  A->row  = a;
  pb::ref(a);
  A->m = (a->comm->rank == 0) ? 1 : 0;
  A->M = 1;
  A->n = a->n;
  A->N = a->N;
  *A_new = A;
  return 0;
}

// MatCreateProd: src/mat/impls/composite/matprod.c:42-48 -- product mats[nmat-1]*...*mats[0]
PetscErrorCode MatCreateProd(MPI_Comm comm, PetscInt nmat, const Mat *mats, Mat *mat)
{   // src/mat/impls/prod/matprod.c: the product mats[nmat-1] * ... * mats[0], applied right to left
  if (nmat < 1) return err(PETSC_ERR_ARG_OUTOFRANGE, "MatCreateProd: no factors");
  if (nmat == 1) {
    *mat = mats[0];
    pb::ref(mats[0]);
    return 0;
  }
  if (nmat > 2) {   // (mats[nmat-1] * ... * mats[1]) * mats[0] by nesting two-factor products
    Mat head, pair[2];
    PB_CHK(MatCreateProd(comm, nmat - 1, mats + 1, &head));
    pair[0]  = mats[0];
    pair[1]  = head;
    int ierr = MatCreateProd(comm, 2, pair, mat);
    MatDestroy(&head);
    return ierr;
  }
  Mat M2 = mats[0], M1 = mats[1];
  for (Mat F : {M1, M2})
    if (F->kind != MK_AIJ && F->kind != MK_DENSE && F->kind != MK_PROJ && F->kind != MK_PROD && F->kind != MK_PENALIZED) return err(PETSC_ERR_SUP, "MatCreateProd: unsupported factor kind");
  // several GPUs: the factors are applied one after the other with their own halo exchanges / reductions (the un-fused route; the fused
  // MPGP driver takes product Hessians on one GPU only, qps.cpp: fused_eligible)
  if (M1->n != M2->m) return err(PETSC_ERR_ARG_SIZ, "MatCreateProd: inner dimensions differ (%d vs %d)", (int)M1->n, (int)M2->m);
  _p_Mat *A = new _p_Mat;
  A->comm = comm;
  A->kind = MK_PROD;
  A->M1   = M1;
  A->M2   = M2;
  pb::ref(M1);
  pb::ref(M2);
  A->m = M1->m;
  A->M = M1->M;
  A->n = M2->n;
  A->N = M2->N;
  PB_CHK(vec_create(comm, M2->m, comm->size > 1 ? PETSC_DECIDE : M2->m, &A->twork));
  *mat = A;
  return 0;
}

PetscErrorCode MatDestroy(Mat *A)
{
  if (!A || !*A) return 0;
  pb::unref(*A);
  return 0;
}
PetscErrorCode MatGetSize(Mat A, PetscInt *M, PetscInt *N)
{
  if (M) *M = A->M;
  if (N) *N = A->N;
  return 0;
}
PetscErrorCode MatGetLocalSize(Mat A, PetscInt *m, PetscInt *n)
{
  if (m) *m = A->m;
  if (n) *n = A->n;
  return 0;
}
PetscErrorCode MatGetOwnershipRange(Mat A, PetscInt *low, PetscInt *high)
{
  if (low) *low = A->rstart;
  if (high) *high = A->rstart + A->m;
  return 0;
}
PetscErrorCode MatCreateVecs(Mat A, Vec *right, Vec *left)
{
  if (right) PB_CHK(vec_create(A->comm, A->n, A->comm->size > 1 ? PETSC_DECIDE : A->n, right));
  if (left) PB_CHK(vec_create(A->comm, A->m, A->comm->size > 1 ? PETSC_DECIDE : A->m, left));
  return 0;
}

namespace pb {

int mat_halo_begin(Mat A, const double *x)
{
  HaloPlan *H = A->halo;
  if (!H || A->comm->size == 1) return 0;
  DevCtx &c = ctx();
  if (!H->send_idx.empty()) PB_CHK(k_pack((int)H->send_idx.size(), H->d_send_idx, x, H->d_send));
  PB_CUDA(cudaEventRecord(H->ev_packed, c.stream));
  PB_CUDA(cudaStreamWaitEvent(c.comm_stream, H->ev_packed, 0));
  ncclComm_t nc = (ncclComm_t)A->comm->nccl;
  if (!nc) return err(PETSC_ERR_ARG_WRONGSTATE, "halo exchange needs NCCL");
  c.launches++;
  PB_NCCL(ncclGroupStart());
  for (size_t q = 0; q < H->neigh.size(); q++) {
    PB_NCCL(ncclSend(H->d_send + H->send_off[q], (size_t)(H->send_off[q + 1] - H->send_off[q]), ncclDouble, H->neigh[q], nc, c.comm_stream));
    PB_NCCL(ncclRecv(H->d_ghost + H->recv_off[q], (size_t)(H->recv_off[q + 1] - H->recv_off[q]), ncclDouble, H->neigh[q], nc, c.comm_stream));
  }
  PB_NCCL(ncclGroupEnd());
  PB_CUDA(cudaEventRecord(H->ev_arrived, c.comm_stream));
  return 0;
}
int mat_halo_end(Mat A)
{
  HaloPlan *H = A->halo;
  if (!H || A->comm->size == 1) return 0;
  PB_CUDA(cudaStreamWaitEvent(ctx().stream, H->ev_arrived, 0));
  return 0;
}

int qppf_dense_rows(QPPF pf, const double **Bd, int *m);

int mat_mult_dev(Mat A, const double *x, double *y)
{
  switch (A->kind) {
  case MK_AIJ:
    PB_CHK(mat_ensure_device(A));
    PB_CHK(mat_halo_begin(A, x));
    PB_CHK(k_spmv(A->Ad, x, y, 0));
    if (A->halo && A->comm->size > 1) {
      PB_CHK(mat_halo_end(A));
      PB_CHK(k_spmv(A->Ao, A->halo->d_ghost, y, 1));
    }
    return 0;
  case MK_DENSE:
    PB_CHK(mat_ensure_device(A));
    return k_spmv(A->Ad, x, y, 0);
  case MK_PROD: {
    double *t;
    PB_CHK(vec_dev_write(A->twork, &t));
    PB_CHK(mat_mult_dev(A->M2, x, t));
    return mat_mult_dev(A->M1, t, y);
  }
  case MK_PROJ: return qppf_apply_mode_dev(A->pf, A->proj_mode, x, y);   // QPPFMatMult_P / _Q / _GtG
  case MK_PENALIZED: {
    // MatMult_Penalized (src/qp/utils/matpenalized.c:12-22): y = BtB x; y *= rho; y += A x.  A x goes first here: a projected
    // Hessian (MK_PROD of MK_PROJ) uses the reducer's device scratch for its own coefficients
    const double *Bd;
    int           m;
    PB_CHK(qppf_dense_rows(A->pf, &Bd, &m));
    PB_CHK(mat_mult_dev(A->A, x, y));
    double t[PB_MAXEQ_ALL];
    PB_CHK(dense_rows_mult_host(A->comm, A->n, m, Bd, x, t));                 // t = B x, rank-ordered sums
    if (A->pf->implicit_orth) {   // implicitly orthonormal rows: the penalised term is Q = B^T (B B^T)^{-1} B (qppf.c:586-589)
      double s[PB_MAXEQ_ALL];
      PB_CHK(qppf_coarse_solve(A->pf, t, s));
      memcpy(t, s, sizeof(double) * m);
    }
    return dense_rows_multT_host(A->comm, A->n, m, Bd, t, A->rho, y, 1);      // y += rho B^T t
  }
  case MK_DUMMY: return err(PETSC_ERR_SUP, "MatMult: a dummy matrix (implicit orthonormalisation) has no MatMult");
  default: return err(PETSC_ERR_SUP, "MatMult: unsupported matrix kind for device vectors");
  }
}

int mat_eqrows_dense(Mat A, double **Bd)
{   // every rank publishes its rows as (global row, global column, value) triples; each rank keeps the entries of its own column range
  if (A->rows_d) {
    *Bd = A->rows_d;
    return 0;
  }
  MPI_Comm  c = A->comm;
  const int size = c->size;
  if (!c->agi || !c->agv) return err(PETSC_ERR_ARG_WRONGSTATE, "communicator has no host exchange");
  struct Trip {
    int    r, c;
    double v;
  };
  const _p_Mat::EqHost &E = *A->eq_host;
  std::vector<Trip>     mine;
  for (PetscInt r = 0; r < A->m; r++)
    for (int k = E.ia[r]; k < E.ia[r + 1]; k++) mine.push_back(Trip{(int)(A->rstart + r), E.ja[k], E.a[k]});
  std::vector<int64_t> bytes(size);
  if (c->agi(c->agctx, (int64_t)(mine.size() * sizeof(Trip)), bytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  int64_t tot = 0;
  for (int r = 0; r < size; r++) tot += bytes[r];
  std::vector<Trip> all((size_t)(tot / sizeof(Trip)) + 1);
  if (c->agv(c->agctx, mine.data(), (int64_t)(mine.size() * sizeof(Trip)), all.data(), bytes.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
  const size_t        M = (size_t)A->M, nl = (size_t)A->n;
  std::vector<double> dense(std::max<size_t>(M * nl, 1), 0.0);
  const size_t        cnt = (size_t)(tot / sizeof(Trip));
  for (size_t k = 0; k < cnt; k++) {
    const Trip &t = all[k];
    if (t.c >= A->cstart && t.c < A->cstart + A->n) dense[(size_t)t.r * nl + (size_t)(t.c - A->cstart)] += t.v;   // layout change only
  }
  PB_CHK(dev_init());
  PB_CHK(dmalloc(&A->rows_d, dense.size()));   // stream-ordered allocation: the copy goes on the same stream, and `dense` is a local
  PB_CUDA(cudaMemcpyAsync(A->rows_d, dense.data(), sizeof(double) * dense.size(), cudaMemcpyHostToDevice, ctx().stream));
  PB_CUDA(cudaStreamSynchronize(ctx().stream));
  *Bd = A->rows_d;
  return 0;
}

int mat_mult(Mat A, Vec x, Vec y)
{
  if (A->kind == MK_AIJ && A->eq_host) {   // y = B x for row-partitioned equality rows: every rank computes all M sums, keeps its own rows
    if (x->n != A->n || y->n != A->m) return err(PETSC_ERR_ARG_SIZ, "MatMult: size mismatch (A %dx%d local, x %d, y %d)", (int)A->m, (int)A->n, (int)x->n, (int)y->n);
    double       *Bd;
    const double *dx;
    double        t[PB_MAXEQ_ALL];
    PB_CHK(mat_eqrows_dense(A, &Bd));
    PB_CHK(vec_dev_read(x, &dx));
    PB_CHK(dense_rows_mult_host(A->comm, A->n, A->M, Bd, dx, t));
    if (y->n > 0) {
      double *h;
      PB_CHK(vec_host_write(y, &h));
      for (PetscInt r = 0; r < A->m; r++) h[r] = t[A->rstart + r];
    }
    return 0;
  }
  if (A->kind == MK_ONEROW) {   // MatMult_OneRow onerow.c:5-17: z = a . x
    double d;
    PB_CHK(vec_dot(A->row, x, &d));
    if (y->n > 0) {
      double *h;
      PB_CHK(vec_host_write(y, &h));
      h[0] = d;
    }
    return 0;
  }
  if (x->n != A->n || y->n != A->m) return err(PETSC_ERR_ARG_SIZ, "MatMult: size mismatch (A %dx%d, x %d, y %d)", (int)A->m, (int)A->n, (int)x->n, (int)y->n);
  const double *dx;
  double       *dy;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_write(y, &dy));
  return mat_mult_dev(A, dx, dy);
}

}  // namespace pb

PetscErrorCode MatMult(Mat A, Vec x, Vec y) { return mat_mult(A, x, y); }
PetscErrorCode MatMultAdd(Mat A, Vec x, Vec y, Vec z)
{
  Vec w;
  PB_CHK(VecDuplicate(z, &w));
  int ierr = mat_mult(A, x, w);
  if (!ierr) ierr = VecWAXPY(z, 1.0, w, y);
  VecDestroy(&w);
  return ierr;
}
PetscErrorCode MatMultTranspose(Mat A, Vec x, Vec y)
{
  if (A->kind != MK_ONEROW) return err(PETSC_ERR_SUP, "MatMultTranspose: only MatCreateOneRow matrices");
  // MatMultTranspose_OneRow onerow.c:41-57: z = a * x[0]  (x broadcast from rank 0)
  double xv = 0.0;
  if (A->comm->size == 1) {
    const double *h;
    PB_CHK(vec_host_read(x, &h));
    xv = h[0];
  } else {
    double v = 0.0;
    if (x->n > 0) {
      const double *h;
      PB_CHK(vec_host_read(x, &h));
      v = h[0];
    }
    std::vector<int64_t> all(A->comm->size);
    int64_t              bits;
    memcpy(&bits, &v, 8);
    if (A->comm->agi(A->comm->agctx, bits, all.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
    memcpy(&xv, &all[0], 8);
  }
  PB_CHK(VecCopy(A->row, y));
  return VecScale(y, xv);
}

// PETSCRAND48 (the generator MatGetMaxEigenvalue creates for its null-space restart, permonmatutils.c:496-499): PetscRandomCreate seeds
// it with 0x12345678 + 76543 * rank, VecSetRandom draws one drand48() per local entry, in order.  drand48 is the 48-bit linear
// congruential generator X <- 0x5DEECE66D X + 0xB (mod 2^48) started at (seed << 16) | 0x330E, value X / 2^48.
static void rand48_fill(int rank, PetscInt n, double *out)
{
  uint64_t X = (((uint64_t)(uint32_t)(0x12345678 + 76543 * rank)) << 16) | 0x330Eull;
  for (PetscInt i = 0; i < n; i++) {
    X      = (0x5DEECE66Dull * X + 0xBull) & 0xFFFFFFFFFFFFull;
    out[i] = (double)X * (1.0 / 281474976710656.0);
  }
}

// MatGetMaxEigenvalue: src/mat/interface/permonmatutils.c:442-522 (power method, v0 = 1)
PetscErrorCode MatGetMaxEigenvalue(Mat A, Vec v, PetscReal *lambda_out, PetscReal tol, PetscInt maxits)
{
  Vec    Av = nullptr;
  bool   destroy_v = false;
  double lambda = 0.0, lambda0, err_, relerr, vAv, vv;
  if (tol == PETSC_DECIDE || tol == PETSC_DEFAULT) tol = 1e-4;            /* :473 */
  if (maxits == PETSC_DECIDE || maxits == PETSC_DEFAULT) maxits = 50;     /* :474 */
  // the reference looks for a stashed estimate first (:462-469); nothing in PERMON ever stores one, so there is none to return
  if (!v && (A->kind == MK_AIJ || A->kind == MK_DENSE) && A->comm->size == 1 && !getenv("PERMON_B200_NOFUSEDPOWER")) {
    PB_CHK(mat_ensure_device(A));
    if ((A->Ad.kind == 3 || A->Ad.kind == 4 || A->Ad.kind == 6) && A->m == A->n) {
      // fused form: one kernel per iteration (y = A (s w) with both dot products in its epilogue), the normalised iterate is never stored
      const PetscInt n = A->m;
      double        *w = nullptr, *y = nullptr;
      PB_CHK(dmalloc(&w, (size_t)std::max<PetscInt>(n, 1)));
      PB_CHK(dmalloc(&y, (size_t)std::max<PetscInt>(n, 1)));
      PB_CHK(k_set(n, w, 1.0));                                           /* :477 */
      double   sc = 1.0;
      Reducer &R = reducer(A->comm);
      int      ierr = 0;
      for (PetscInt i = 1; i <= maxits && !ierr; i++) {                   /* :484 */
        lambda0 = lambda;
        ierr = k_power_step(A->Ad, w, sc, y, R.rb);                       /* :487-491 */
        if (!ierr) ierr = R.fetch();
        if (ierr) break;
        vAv    = R.sum(0);
        vv     = R.sum(1);
        lambda = vAv / vv;                                                /* :492 */
        if (lambda < PETSC_MACHINE_EPSILON) {                             /* :493-502: A v fell into the null space */
          std::vector<double> rnd((size_t)std::max<PetscInt>(n, 1));
          rand48_fill(A->comm->rank, n, rnd.data());
          cudaMemcpyAsync(y, rnd.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx().stream);
          cudaStreamSynchronize(ctx().stream);
        }
        err_   = fabs(lambda - lambda0);                                  /* :504 */
        relerr = err_ / fabs(lambda);
        if (relerr < tol) break;                                          /* :506 */
        std::swap(w, y);                                                  /* :509 v = A v ... */
        sc = 1.0 / sqrt(vv);                                              /* :510 ... / ||v|| (applied by the next gather) */
      }
      dfree(w);
      dfree(y);
      if (ierr) return ierr;
      if (lambda_out) *lambda_out = lambda;
      return 0;
    }
  }
  if (!v) {
    PB_CHK(MatCreateVecs(A, &v, NULL));
    PB_CHK(VecSet(v, 1.0));                                               /* :477 */
    destroy_v = true;
  }
  PB_CHK(VecDuplicate(v, &Av));
  for (PetscInt i = 1; i <= maxits; i++) {                                /* :484 */
    lambda0 = lambda;
    PB_CHK(mat_mult(A, v, Av));                                           /* :487 */
    PB_CHK(vec_mdot2(v, Av, v, &vAv, &vv));                               /* :491 */
    lambda = vAv / vv;                                                    /* :492 */
    if (lambda < PETSC_MACHINE_EPSILON) {                                 /* :493-502 */
      double *h;
      PB_CHK(vec_host_write(Av, &h));
      rand48_fill(A->comm->rank, Av->n, h);
    }
    err_   = fabs(lambda - lambda0);                                      /* :504 */
    relerr = err_ / fabs(lambda);
    if (relerr < tol) break;                                              /* :506 */
    {                                                                     /* :509-510 VecCopy + VecScale in one pass */
      const double *dAv;
      double       *dv;
      PB_CHK(vec_dev_read(Av, &dAv));
      PB_CHK(vec_dev_write(v, &dv));
      PB_CHK(k_scale_to(v->n, dv, 1.0 / sqrt(vv), dAv));
    }
  }
  if (lambda_out) *lambda_out = lambda;
  if (destroy_v) VecDestroy(&v);
  VecDestroy(&Av);
  return 0;
}
