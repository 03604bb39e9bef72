// objects.h -- host-side object model behind the opaque handles of include/permon_b200.h.
// The layout follows what the reference keeps in its private headers for the hot path
// (include/permon/private/{qpimpl.h,qpcimpl.h,qppfimpl.h,qpsimpl.h}), minus everything PETSc owns.
#pragma once
#include <stdio.h>

#include <map>
#include <string>
#include <cstdlib>
#include <vector>

#include "../../include/permon_b200.h"
#include "device.h"

struct ncclComm;

// ---- communicator -----------------------------------------------------------------------------------
struct _p_PermonComm {
  int                    rank = 0, size = 1;
  ncclComm              *nccl = nullptr;
  PermonB200AllGatherI64 agi = nullptr;   // host exchange (set-up only)
  PermonB200AllGatherV   agv = nullptr;
  void                  *agctx = nullptr;
  // peer-memory window (CUDA IPC over NVLink): reduction records are pushed, not all-gathered by NCCL
  bool                   p2p = false;
  void                  *win_base = nullptr;
  pb::P2PWin            *d_win = nullptr;
  double                *my_slot = nullptr;
  unsigned long long    *my_flag = nullptr;
  unsigned long long     seq[PB_NKINDS] = {0, 0, 0};
  std::vector<void *>    peer_bases;
};

struct PObj {
  int         refct = 1;
  MPI_Comm    comm  = nullptr;
  std::string prefix, name, type;
  virtual ~PObj() {}
};

struct _p_PetscViewer : PObj {
  FILE *f = nullptr;
  bool  own = false;
  int   tab = 0;
};

struct _p_IS : PObj {
  std::vector<PetscInt> idx;   // global indices (local part)
  int                  *d_local = nullptr;   // device copy of idx - rstart (lazily built by the QPC)
};

struct _p_Vec : PObj {
  PetscInt n = 0, N = 0, rstart = 0;
  double  *h = nullptr;
  bool     h_owned = false;
  double  *d = nullptr;
  bool     d_owned = false;
  bool     h_valid = false, d_valid = false;
  bool     invalidated = false;   // VecInvalidate (permonvecutils.c:266-284); read it through pb::vec_invalid(), set it through pb::vec_mark_invalid()
  int64_t  inval_state = 0;       // object state at the time of the invalidation: a later write makes the vector valid again (:303-326)
  int64_t  state = 0;
  cudaEvent_t up_ev = nullptr;   // a prefetch (H2D on the copy stream) is in flight: settled by the next access
  bool        h2d_inflight = false;   // an asynchronous upload FROM the host buffer was enqueued on the compute stream: a host writer must wait for it
  ~_p_Vec() override;
};

// halo plan of a row-partitioned AIJ matrix (PETSc: Mat_MPIAIJ garray / lvec / Mvctx, mpiaij.h:49-83)
struct HaloPlan {
  std::vector<PetscInt> garray;      // global column of every ghost, ascending
  std::vector<PetscInt> neigh;       // neighbour ranks (ascending)
  std::vector<PetscInt> recv_off;    // [nneigh+1] slices of the ghost buffer per neighbour
  std::vector<PetscInt> send_off;    // [nneigh+1] slices of the send buffer per neighbour
  std::vector<PetscInt> send_idx;    // local indices to pack, grouped by neighbour
  int                  *d_send_idx = nullptr;
  double               *d_send = nullptr, *d_ghost = nullptr;
  int                  *d_row_map = nullptr;   // rows outside [skip_lo, skip_hi): index of the row in the compressed off-diagonal block, -1 = none
  int                   skip_lo = 0, skip_hi = 0;   // widest run of rows without ghost columns
  PetscInt              nboundary = 0;
  cudaEvent_t           ev_packed = nullptr, ev_arrived = nullptr, ev_consumed = nullptr;
  // peer-memory halo: neighbours store their boundary values straight into my ghost window
  bool                  p2p = false;
  void                 *gwin = nullptr;
  double               *d_ghost2[2] = {nullptr, nullptr};      // [0]: ghosts of p, [1]: ghosts of x
  unsigned long long   *my_hflags[2] = {nullptr, nullptr};
  pb::HaloPush          push[2];
  unsigned long long    hseq[2] = {0, 0};
  std::vector<void *>   peer_gwins;
  bool                  contig = false;                       // every pack list is one ascending run of rows
  std::vector<PetscInt> send_lo;                              // first row of each run
  pb::PushRanges       *d_ranges = nullptr;                   // device copies [2] (p, x) for the fused pushes
  // host copy of the split matrix, kept until the first device use (lets the plan be built and inspected
  // without a GPU; the arithmetic still needs one)
  // big arrays of the diagonal block: filled in parallel right after the allocation, never zero-filled first
  template <class T>
  struct UVec {
    T     *p = nullptr;
    size_t n = 0;
    UVec() {}
    UVec(const UVec &) = delete;
    UVec &operator=(const UVec &) = delete;
    ~UVec() { free(p); }
    void resize(size_t k)
    {
      free(p);
      p = (T *)malloc((k ? k : 1) * sizeof(T));
      n = p ? k : 0;
    }
    T       *data() { return p; }
    size_t   size() const { return n; }
    T       &operator[](size_t i) { return p[i]; }
  };
  struct HostSplit {
    std::vector<int>           dia, oia, oja, orow;
    UVec<int>                  dja;
    std::vector<double>        oa;
    UVec<double>               da;
    std::vector<unsigned char> skip;
    // fast path (constant-coefficient stencils): the all-stencil form of the diagonal block, built straight from the caller's arrays;
    // dia / dja / da stay empty unless MatB200GetHostSplit asks for them while those arrays are still alive
    pb::StencilHost    st;
    int64_t            nnz_diag = 0;
    const PetscInt    *ui = nullptr, *uj = nullptr;
    const PetscScalar *ua = nullptr;
    PetscInt           c0 = 0;
  } *host = nullptr;
};

enum MatKind { MK_AIJ = 0, MK_ONEROW, MK_PROD, MK_PENALIZED, MK_PROJ /* P = I - G'(GG')^-1 G of a QPPF */, MK_DENSEROWS /* m x n dense rows on the device */,
               MK_DUMMY /* MatCreateDummy of the implicit orthonormalisation (permonmatorth.c:176-192): no MatMult; `A` = the matrix it stands for */,
               MK_DENSE /* column-major m x n (MATSEQDENSE / MATSEQDENSECUDA), device form in Ad (kind 6) */ };

struct _p_Mat : PObj {
  MatKind  kind = MK_AIJ;
  PetscInt m = 0, n = 0, M = 0, N = 0, rstart = 0, cstart = 0;
  // AIJ: device CSR of the diagonal block (local columns) and of the off-diagonal block (compressed rows)
  pb::CsrDev Ad, Ao;
  bool       d_owned = true;
  HaloPlan  *halo = nullptr;
  // ONEROW
  Vec row = nullptr;
  // PROD: y = M1 (M2 x)
  Mat M1 = nullptr, M2 = nullptr;
  Vec twork = nullptr;
  // DENSEROWS: row-major m x n device array (orthonormalised equality rows)
  double *rows_d = nullptr;
  // AIJ, row-partitioned with at most PB_MAXEQ_ALL GLOBAL rows (an equality matrix B_E created like any PETSc MPIAIJ: rank r owns a few
  // rows with GLOBAL columns): the local rows are kept on the host and turned into dense M x n_local rows (column-partitioned like the
  // vectors) on first use -- no halo plan, the rows are wide and their pattern is not symmetric
  struct EqHost {
    std::vector<int>    ia, ja;
    std::vector<double> a;
  };
  EqHost *eq_host = nullptr;
  // PENALIZED: y = A x + rho G^T G x   (matpenalized.c:4-8); PROJ uses pf only
  Mat    A = nullptr;
  QPPF   pf = nullptr;
  double rho = 0.0;
  int    proj_mode = 0;   // PROJ: 0 P = I - Q (QPPFCreateP), 1 Q (QPPFCreateQ), 2 G^T G (QPPFCreateGtG)
  // DENSE: the caller's array (host, or device when dn_src_dev) and its leading dimension until the first use (mat_ensure_device), which
  // adopts a suitably aligned device array or makes the library's padded device copy (dn_own)
  const double *dn_src = nullptr;
  int64_t       dn_src_lda = 0;
  bool          dn_src_dev = false, dn_ready = false, dn_adopted = false;
  double       *dn_own = nullptr;
  // cached extreme eigenvalue (PetscObjectComposedData in the reference)
  ~_p_Mat() override;
};

struct _p_QPC : PObj {   // qpcimpl.h:27-34 + qpcboximpl.h:5-10
  IS     is = nullptr;
  Vec    lb = nullptr, ub = nullptr, llb = nullptr, lub = nullptr;
  Vec    lb_full = nullptr, ub_full = nullptr;   // IS expanded to full local length (+-PETSC_INFINITY outside)
  Vec    lambdawork = nullptr;
  double astol = 10 * PETSC_MACHINE_EPSILON;
  bool   setupcalled = false;
  ~_p_QPC() override;
};

struct _p_QPPF : PObj {   // qppfimpl.h:6-31
  Mat                 G = nullptr;
  PetscInt            m = 0, n = 0;
  double             *Bd = nullptr;     // dense rows on the device [m][n]
  bool                Bd_owned = false;
  std::vector<double> GGt, L;           // m x m and its Cholesky factor (host, replicated)
  bool                orth = false, setupcalled = false;
  bool                implicit_orth = false;   // G_has_orthonormal_rows_implicitly (qppf.c:123-127): G stands for (G G^T)^{-1/2} G, applied as Q
  Vec                 G_left = nullptr, Gt_right = nullptr;
  // qppfimpl.h: explicitInv (apply inv(G G^T) as an explicit m x m matrix instead of two triangular solves), redundancy (number of
  // redundant coarse solves; the m x m factor is replicated on every rank here, so any value is honoured as "all ranks"), alpha_tilde
  bool                explicitInv = false;
  PetscInt            redundancy = PETSC_DEFAULT, setfromoptionscalled = 0;
  std::vector<double> GGtinv;           // explicit inverse (host, replicated) when explicitInv
  Vec                 alpha_tilde = nullptr;
  Mat                 GGt_mat = nullptr;   // QPPFGetGGt: G G^T as an m x m dense-rows Mat (built on demand)
  ~_p_QPPF() override;
};

typedef PetscErrorCode (*QPPostSolveFn)(QP child, QP parent);

struct _p_QP : PObj {   // qpimpl.h:6-57
  Mat           A = nullptr;
  Vec           b = nullptr, x = nullptr, xwork = nullptr;
  bool          b_plus = false;
  Mat           BE = nullptr;
  Vec           cE = nullptr, lambda_E = nullptr, Bt_lambda = nullptr;
  QPC           qpc = nullptr;
  QPPF          pf = nullptr;
  QP            parent = nullptr, child = nullptr;
  QPPostSolveFn postSolve = nullptr;
  Vec           postSolveCtx = nullptr;   // xtilde of QPTHomogenizeEq
  std::vector<double> postT;              // T (m x m) of QPTOrthonormalizeEq
  int           transform = 0;            // 0 none, 1 penalty, 2 homogenize, 3 projector, 4 orthonormalize
  std::string   transform_name = "";
  int           id = 0;
  bool          setupcalled = false, solved = false, setfromoptionscalled = false;
  PetscErrorCode (*changeListener)(QP) = nullptr;
  void         *changeListenerCtx = nullptr;
  ~_p_QP() override;
};

struct QPSImpl {   // _QPSOps, qpsimpl.h:12-24
  virtual ~QPSImpl() {}
  virtual PetscErrorCode setup(QPS) = 0;
  virtual PetscErrorCode solve(QPS) = 0;
  virtual PetscErrorCode reset(QPS) { return 0; }
  virtual PetscErrorCode resetstatistics(QPS) { return 0; }
  virtual PetscErrorCode setfromoptions(QPS) { return 0; }
  virtual PetscErrorCode isqpcompatible(QPS, QP, PetscBool *flg)
  {
    *flg = PETSC_TRUE;
    return 0;
  }
  virtual PetscErrorCode viewconvergence(QPS, PetscViewer) { return 0; }
  virtual bool           has_monitor() { return false; }
  virtual PetscErrorCode monitor(QPS, PetscInt, PetscViewer) { return 0; }
};

struct QPSConvergedDefaultCtx {   // qpsimpl.h:73-76
  double norm_rhs = NAN, ttol = NAN, norm_rhs_div = NAN;
  bool   setup_called = false;
};

struct _p_QPS : PObj {   // qpsimpl.h:26-71
  QPSImpl *impl = nullptr;
  QP       topQP = nullptr, solQP = nullptr;
  double   rtol = 1e-5, atol = 1e-50, divtol = 1e4, rnorm = 0.0;
  PetscInt max_it = 10000, iteration = 0, iterations_accumulated = 0, nsolves = 0;
  KSPConvergedReason reason = KSP_CONVERGED_ITERATING;
  bool     autoPostSolve = true, setupcalled = false, postsolvecalled = false, user_type = false;
  bool     view_convergence = false, view_kkt = false;
  PetscErrorCode (*convergencetest)(QPS, KSPConvergedReason *) = nullptr;
  PetscErrorCode (*convergencetestdestroy)(void *) = nullptr;
  void    *cnvctx = nullptr;
  struct Mon {
    PetscErrorCode (*f)(QPS, PetscInt, PetscReal, void *);
    void              *ctx;
    PetscCtxDestroyFn *destroy;
  };
  std::vector<Mon> monitors;
  ~_p_QPS() override;
};

namespace pb {

// ---- helpers shared by the translation units -----------------------------------------------------------
int  err(int code, const char *fmt, ...);
bool gpu_required();

// reference counting
template <class T>
inline void ref(T *o)
{
  if (o) o->refct++;
}
template <class T>
inline void unref(T *&o)
{
  if (o && --o->refct == 0) delete o;
  o = nullptr;
}

// Vec access with host/device validity tracking (PETSc: offload mask)
int vec_create(MPI_Comm comm, PetscInt n, PetscInt N, Vec *v);
int vec_dev_read(Vec v, const double **d);
int vec_dev_write(Vec v, double **d);       // contents will be overwritten entirely
int vec_dev_rw(Vec v, double **d);
int vec_host_read(Vec v, const double **h);
int vec_host_write(Vec v, double **h);
int vec_host_rw(Vec v, double **h);
int vec_layout(MPI_Comm comm, PetscInt n, PetscInt *N, PetscInt *rstart);

// reductions: record buffers + cross-rank combination
struct Reducer {
  RedBuf   rb;
  double  *d_local = nullptr;    // PB_NRED doubles: this rank's record
  double  *d_all = nullptr;      // [size][PB_NRED] gathered records (== d_local when size == 1)
  double  *h_all = nullptr;      // pinned host mirror
  MPI_Comm comm = nullptr;
  int      init(MPI_Comm comm);
  void     destroy();
  int      gather();                       // NCCL all-gather of the local record (no-op for 1 rank)
  int      fetch();                        // copy the gathered records to the host and wait
  double   sum(int slot) const;            // rank-ordered sum of h_all
  double   min(int slot) const;
};
Reducer &reducer(MPI_Comm comm);           // shared scratch reducer of the communicator

// VecIsInvalidated semantics of the reference: invalid until the vector is written again (its state counter moves past the recorded one)
inline bool vec_invalid(Vec v)
{
  if (v->invalidated && v->state > v->inval_state) v->invalidated = false;
  return v->invalidated;
}
inline void vec_mark_invalid(Vec v, bool invalid)
{
  v->invalidated = invalid;
  v->inval_state = v->state;
}
int  vec_prefetch(Vec v);                                    // start the H2D copy of a host-valid vector on the copy stream (pinned buffers: truly asynchronous)
// dense equality rows B (m x n, row-major on the device), any m <= PB_MAXEQ_ALL: t = B x (host values, summed over ranks) and
// y (+)= scale * B^T t, in chunks of PB_NRED rows per launch
int  dense_rows_mult_host(MPI_Comm comm, int n, int m, const double *Bd, const double *x, double *t);
int  dense_rows_multT_host(MPI_Comm comm, int n, int m, const double *Bd, const double *t, double scale, double *y, int accumulate);
int  vec_dot(Vec x, Vec y, double *val);
int  vec_norm2(Vec x, double *val);
int  vec_mdot2(Vec x, Vec y0, Vec y1, double *v0, double *v1);
int  mat_mult(Mat A, Vec x, Vec y);
int  mat_mult_dev(Mat A, const double *x, double *y);        // raw device pointers (local lengths)
int  mat_eqrows_dense(Mat A, double **Bd);                  // row-partitioned equality matrix -> dense M x n_local rows on the device (collective)
int  qppf_apply_P_dev(QPPF cp, const double *x, double *y);   // y = x - G^T (G G^T)^{-1} G x on raw device pointers
int  qppf_apply_mode_dev(QPPF cp, int mode, const double *x, double *y);   // 0: P, 1: Q, 2: G^T G
int  qppf_coarse_solve(QPPF cp, const double *r, double *y);               // (G G^T) y = r, m host values
int  mat_ensure_device(Mat A);                               // upload a lazily kept host split (multi-rank AIJ)
int  mat_halo_begin(Mat A, const double *x);                 // pack + post send/recv on the comm stream
int  mat_halo_end(Mat A);                                    // make the compute stream wait for the ghosts
int  box_dev(QPC qpc, BoxDev *bx);
int  qpc_box_for_vec(QPC qpc, Vec x, BoxDev *bx);   // sets the QPC up for the layout of x (IS expansion) first
int  qppf_dense_rows(QPPF pf, const double **Bd, int *m);
int  comm_allgather_records(MPI_Comm comm, const double *d_local, double *d_all);
int  options_get(const std::string &prefix, const char *name, std::string *val);
bool options_real(const std::string &prefix, const char *name, double *v);
bool options_int(const std::string &prefix, const char *name, PetscInt *v);
bool options_bool(const std::string &prefix, const char *name, bool *v);
bool options_string(const std::string &prefix, const char *name, std::string *v);
void vprintf_viewer(PetscViewer v, const char *fmt, ...);

}  // namespace pb
