// device.h -- internal C++ interface between the host-side PERMON objects and the CUDA kernels.
// Nothing here is exported; the C ABI lives in include/permon_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <vector>

#include "mpgp_ctl.h"

namespace pb {

// ---- device context -----------------------------------------------------------------------------
struct DevCtx {
  int          device      = -1;
  int          sm_count    = 0;
  bool         ready       = false;
  cudaStream_t stream      = nullptr;   // compute stream (library-owned or caller-provided)
  cudaStream_t own_stream  = nullptr;
  cudaStream_t comm_stream = nullptr;   // NCCL halo traffic, overlapped with interior rows
  cudaStream_t copy_stream = nullptr;   // vector prefetches (H2D) that overlap the power method of the set-up
  int64_t      launches    = 0;         // kernels launched by this library (bench.py: gpu_launches)
};
DevCtx &ctx();
extern int g_p2p_size;
int     dev_init();                      // 0 on success, PETSC_ERR_GPU otherwise
void    set_error(const char *fmt, ...);
const char *last_error();
int     cuda_fail(cudaError_t e, const char *what, const char *file, int line);
#define PB_CUDA(call)                                                  \
  do {                                                                 \
    cudaError_t e_ = (call);                                           \
    if (e_ != cudaSuccess) return pb::cuda_fail(e_, #call, __FILE__, __LINE__); \
  } while (0)
#define PB_CHK(call)            \
  do {                          \
    int ierr_ = (call);         \
    if (ierr_) return ierr_;    \
  } while (0)

// ---- device / pinned memory -----------------------------------------------------------------------------------------------
// Device buffers come from the stream-ordered CUDA memory pool of the device with the release threshold lifted: memory freed by a
// destroyed Vec / Mat / solver stays cached in the pool and the next object of the same size gets it back without a trip to the
// driver (cudaMalloc / cudaFree of 100 MB-1 GB buffers cost milliseconds each and cudaFree synchronises the device).  Buffers that
// peers map through CUDA IPC are NOT allocated here.  Small pinned host blocks are cached by size for the same reason.
int   dmalloc_bytes(void **p, size_t bytes);
void  dfree(const void *p);
template <class T>
int dmalloc(T **p, size_t count)
{
  return dmalloc_bytes((void **)p, count * sizeof(T));
}
void *pinned_get(size_t bytes);             // nullptr when out of memory
void  pinned_put(void *p, size_t bytes);

// ---- wall-clock phase timer (PERMON_B200_TIMING=1): synchronises the device on both sides and prints one line to stderr ----
struct PhaseTimer {
  const char *name;
  double      t0;
  bool        on;
  explicit PhaseTimer(const char *name);
  ~PhaseTimer();
};

// ---- profiling (bench.py roofline) -----------------------------------------------------------------
enum KFamily { KF_SPMV_A = 0, KF_UPDATE_B, KF_SPMV_A2, KF_DIR_C, KF_CTRL, KF_SPMV_PLAIN, KF_VEC, KF_QPC, KF_HALO, KF_COUNT };
const char *family_name(int f);
void        prof_begin();
int         prof_end();
int         prof_get(int family, int64_t *launches, double *ms, double *bytes_per_launch);
int         prof_get_working(int family, int64_t *launches, double *ms);   // launches that did work (not early exits) and their time
int         prof_dump(const char *path);
void        prof_pre(int family, double bytes);
void        prof_post(int family);

// ---- device CSR ------------------------------------------------------------------------------------
static constexpr int TR = 256;   // rows per SpMV tile

// one tile of the packed (dictionary-coded) matrix format, see pack.cpp
struct PkHeader {
  uint16_t kind;    // 1: coded (dictionary of (col - row, value) pairs + one byte per non-zero), 0: raw
  uint16_t ndict;
  uint32_t nnz;
  uint16_t ulen;    // common row length, 0xFFFF when the rows differ (then rowoff[] is present)
  uint16_t nrows;
  uint32_t pad;
};
static_assert(sizeof(PkHeader) == 16, "tile header is one 16-byte line");

// All-stencil matrices (kind 4): every 256-row tile is a stencil tile (pack.cpp) and the matrix has at most PB_ST_MAXPAT distinct
// patterns.  The device form is one presence byte per row, one pattern id per tile and the pattern table; the SpMV kernel stages the
// x WINDOWS a tile gathers from -- x[r0 + d .. r0 + d + 256) for every pattern delta d, deltas closer than PB_ST_SPAN share a window --
// with bulk copies, so that the gathers of the consumer threads are shared-memory loads.
#define PB_ST_MAXPAT 32
#define PB_ST_SPAN 64
#define PB_ST_WCAP ((256 + PB_ST_SPAN + 2) * 8)   // bytes reserved per window in a shared-memory stage (multiple of 16)
struct StPattern {
  int    L, nwin;
  int    d[8];       // col - row of the pattern entries, ascending (storage order)
  int    wlo[8];     // window w holds x[r0 + wlo[w] .. r0 + wlo[w] + wlen[w]); wlo and wlen are even (16-byte granules)
  int    wlen[8];
  int    erel[8];    // byte offset of x[r0 + d[j]] from the start of the stage's window area
  double v[8];
};
static_assert(sizeof(StPattern) % 8 == 0, "pattern table entries are 8-byte aligned");

// uninitialised host byte buffer (std::vector would zero-fill ~100 MB on one thread before the parallel fill)
struct RawBuf {
  unsigned char *p = nullptr;
  size_t         n = 0;
  RawBuf() {}
  RawBuf(const RawBuf &) = delete;
  RawBuf &operator=(const RawBuf &) = delete;
  ~RawBuf() { free(p); }
  bool alloc(size_t bytes)
  {
    free(p);
    p = (unsigned char *)malloc(bytes ? bytes : 1);
    n = p ? bytes : 0;
    return p != nullptr;
  }
  unsigned char *data() { return p; }
  size_t         size() const { return n; }
};

// blob bytes of one tile of each kind (pack.cpp); shared by the host builder and the device re-coder (recode.cu)
__host__ __device__ inline size_t pk_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
__host__ __device__ inline size_t pk_coded_bytes(int ndict, int nrows, int nnz, bool uniform)
{
  size_t b = sizeof(PkHeader) + pk_up(ndict, 2) * 8 + pk_up(ndict, 4) * 4;
  if (!uniform) b += pk_up((size_t)nrows + 1, 8) * 2;
  b += pk_up(nnz, 16);
  return pk_up(b, 16);
}
__host__ __device__ inline size_t pk_stencil_bytes(int L, int nrows) { return pk_up(sizeof(PkHeader) + pk_up(L, 2) * 8 + pk_up(L, 4) * 4 + pk_up((size_t)nrows, 16), 16); }
__host__ __device__ inline size_t pk_raw_bytes(int nrows, int nnz)
{
  return pk_up(sizeof(PkHeader) + pk_up(nnz, 2) * 8 + pk_up(nnz, 4) * 4 + pk_up((size_t)nrows + 1, 8) * 2, 16);
}
int pattern_windows(StPattern &P);   // lays out the x windows of a pattern; returns the last window index

struct StencilHost {   // host side of the all-stencil form, filled by pk_build
  bool                       valid = false;
  std::vector<StPattern>     pats;
  std::vector<unsigned char> pid;
  RawBuf                     masks;   // ntiles * 256 bytes (zero beyond n)
  int                        nwin = 0;
};

struct OffDiagEntries {   // ghost-column entries of a row block, in row order (storage order within a row)
  std::vector<int>    row, gcol;
  std::vector<double> val;
};

struct CsrDev {
  int           n      = 0;        // rows
  int           ncols  = 0;
  int64_t       nnz    = 0;
  const int    *ia     = nullptr;  // [n+1]
  const int    *ja     = nullptr;  // [nnz] local column ids
  const double *a      = nullptr;  // [nnz]
  const int    *rows   = nullptr;  // optional compressed row list (off-diagonal block): row id of each stored row
  int64_t       nnz_alloc = 0;     // elements of ja / a that may be read (allocation incl. padding)
  int           ia_alloc = 0;      // entries of ia that may be read
  int           stages = 2;        // shared-memory stages of the TMA kernel
  int           kind   = 0;        // 0: tile-streamed plain loads, 1: vector (W lanes per row), 2: TMA-staged CSR tiles, 3: TMA-staged packed tiles, 4: stencil windows,
                                   // 5: tile-ELL, 6: dense column-major
  // packed tiles (kind 3): blob + tile directory (offsets in 16-byte units); the raw CSR arrays are then absent
  const unsigned char *pk     = nullptr;
  const unsigned      *pk_off = nullptr;
  int                  pk_max = 0;      // largest tile blob in bytes
  int64_t              pk_bytes = 0;    // blob + directory bytes (what one SpMV streams for the matrix)
  int64_t              pk_coded = 0;    // tiles that are dictionary-coded
  // all-stencil form (kind 4)
  const unsigned char *st_masks = nullptr;   // [n] presence byte per row
  const unsigned char *st_pid = nullptr;     // [ntiles] pattern of each tile
  const StPattern     *st_pats = nullptr;
  int                  st_npat = 0, st_nwin = 0, st_lmax = 0;   // patterns; largest number of windows of a pattern; longest pattern
  int                  st_dlo = 0, st_dhi = 0;                  // smallest / largest col - row over all patterns
  // long-row matrices in tile-ELL form (kind 5): 256-row tiles stored COLUMN-major (entry t of all rows of the tile is contiguous), one
  // thread per row -- unit-stride matrix stream, products added in storage order
  const double *ell_val = nullptr;
  const int    *ell_col = nullptr;
  const int    *ell_len = nullptr;     // [n] row lengths
  const int    *ell_lt  = nullptr;     // [ntiles] longest row of each tile
  const int64_t *ell_off = nullptr;    // [ntiles] first element of each tile in ell_val / ell_col
  int64_t       ell_elems = 0;         // elements stored (padding included)
  // dense matrices (kind 6): column-major, entry (i, j) at dn_a[i + j * dn_lda]; dn_a is 16-byte aligned and dn_lda even, so every
  // column segment can be staged with bulk copies.  dn_rpb rows per CTA (one consumer thread per row); dn_split > 0: split-column
  // variant with column chunks of dn_split columns, partial sums in dn_part [nchunks][n]
  const double *dn_a     = nullptr;
  int64_t       dn_lda   = 0;
  int           dn_rpb   = 0;
  int           dn_split = 0;
  double       *dn_part  = nullptr;
  int           W      = 32;
  int           tile_cap = 0;      // max nnz of a 256-row tile (stream kind)
  int           grid   = 0;        // persistent grid size (fixed => reproducible reductions)
};

struct BoxDev {
  const double *lb = nullptr, *ub = nullptr;   // full local length; NULL = absent
  double        astol = 0.0;
};

// Peer-memory window of the communicator (multi-GPU): every rank owns a small buffer that all peers map through
// CUDA IPC.  Reduction records are PUSHED by the last CTA of the producing kernel straight into every peer's window
// over NVLink, followed by a sequence-number flag; the ctrl kernels spin on their local flags.  No NCCL call, no
// host round trip, no extra kernel for the scalar "all-gathers" of the iteration.
#define PB_NKINDS 3      // 0: after K_A, 1: after K_B / projection, 2: after K_A'
#define PB_MAXNEIGH 16
#define PB_FLAG_STRIDE 16   // unsigned long long per flag slot (128 bytes: one line per flag)
struct P2PWin {
  int                 rank = 0, size = 1;
  double             *slot[PB_MAXRANKS];   // peer q: [PB_NKINDS][2 parities][PB_MAXRANKS][PB_NRED]
  unsigned long long *flag[PB_MAXRANKS];   // peer q: [PB_NKINDS][PB_MAXRANKS] * PB_FLAG_STRIDE
};
__host__ __device__ inline size_t p2p_slot_index(int kind, unsigned long long seq, int rank) { return (((size_t)kind * 2 + (seq & 1)) * PB_MAXRANKS + rank) * PB_NRED; }
__host__ __device__ inline size_t p2p_flag_index(int kind, int rank) { return ((size_t)kind * PB_MAXRANKS + rank) * PB_FLAG_STRIDE; }

struct RedBuf {
  double   *partials = nullptr;   // [maxblocks][PB_NRED]
  unsigned *counter  = nullptr;
  double   *out      = nullptr;   // where the last block stores the record (PB_NRED doubles)
  const double *add_part = nullptr;   // optional per-CTA partial sums of an earlier kernel (stride PB_NRED), added into slot add_slot
  int           add_n = 0, add_slot = 0;
  const P2PWin      *win = nullptr;   // when set: also publish the record to every peer (kind, seq)
  int                kind = 0;
  unsigned long long seq = 0;
};

// halo exchange by direct peer stores ("pack + send" in one kernel) and the matching wait of the ghost pass
struct HaloPush {
  int                 nneigh = 0, total = 0;
  int                 send_off[PB_MAXNEIGH + 1];
  double             *dst[PB_MAXNEIGH];    // neighbour q's ghost buffer at the offset reserved for this rank
  unsigned long long *flag[PB_MAXNEIGH];   // neighbour q's flag slot for this rank
  const int          *send_idx = nullptr;
  unsigned           *counter = nullptr;
};
// control step folded into the prologue of K_B (ctrl_A) / K_C (ctrl_B): every CTA recomputes the (tiny, deterministic)
// scalar logic from the reduction records into shared memory; CTA 0 stores the new state for the following kernels.
struct CtrlFold {
  int                       fold = 0;
  const MpgpCtl            *Sin = nullptr;    // fold: state before the control step; else: state after it
  MpgpCtl                  *Sout = nullptr;   // fold: where CTA 0 stores the updated state
  const double             *rec0 = nullptr, *rec1 = nullptr;       // rank-0 record (K_B: rec0 = after K_A; K_C: rec0 = after K_B, rec1 = after K_A')
  const unsigned long long *flags0 = nullptr, *flags1 = nullptr;   // peer-memory mode: local flags to wait on (one per rank)
  unsigned long long        seq0 = 0, seq1 = 0;
  int                       size = 1;
};
// halo push fused into the kernel that produces the vector (contiguous boundary ranges, e.g. slab partitions)
struct PushRanges {
  int                 n = 0;
  int                 lo[PB_MAXNEIGH], hi[PB_MAXNEIGH];
  double             *dst[PB_MAXNEIGH];
  unsigned long long *flag[PB_MAXNEIGH];
  unsigned           *counter = nullptr;
  int                 gap_lo = 0, gap_hi = 0;   // largest run of rows outside every range
};
// Off-diagonal (ghost column) part of a row-partitioned matrix, merged into K_A / K_A' (multi-GPU): rows outside [lo, hi) -- the
// widest run of rows without ghost columns, i.e. the interior of a slab -- look up their compressed off-diagonal row, wait (once per
// thread) until every neighbour's halo push of this sequence number has landed, and add the ghost products to the row sum before
// the fused epilogue (the order of PETSc's MatMult_MPIAIJ: diagonal block first, then MatMultAdd of the off-diagonal block).
// The tiles that hold such rows are processed LAST (TileOrder), so the wait is over by the time it is reached.
struct GhostMerge {
  const int                *row_map = nullptr;   // [lo + (n - hi)] index into the compressed off-diagonal rows, -1: no ghost column
  int                       lo = 0, hi = 0;
  const int                *oia = nullptr, *oja = nullptr;
  const double             *oa = nullptr;
  const double             *ghost = nullptr;     // ghost values (written by the neighbours over NVLink, or by ncclRecv)
  const unsigned long long *flags = nullptr;     // peer-memory mode: local flag slots (PB_FLAG_STRIDE apart), one per neighbour
  int                       nflags = 0;
  unsigned long long        seq = 0;
};
// order in which the persistent SpMV grid walks the 256-row tiles: tiles [ta, tb) first (ascending, or descending when the
// sweep direction of the iteration says so), then the tiles outside that range
struct TileOrder {
  int ta = 0, tb = 0;
  int pf = 0;        // direct stencil kernels: L2 prefetch distance in grid sweeps (0: off)
  int dlo = 0, dhi = 0;   // smallest / largest col - row of the stencil patterns (the gather that touches a line first, per sweep direction)
};

// ---- kernels: generic vector ops (deterministic) -----------------------------------------------------
int k_set(int n, double *x, double a);
int k_copy(int n, const double *x, double *y);
int k_scale(int n, double *x, double a);
int k_filter(int n, double *x, double tol);                            // x_i = 0 where |x_i| < tol (VecFilter)
int k_scale_to(int n, double *y, double a, const double *x);           // y = a x
int k_axpy(int n, double *y, double a, const double *x);
int k_aypx(int n, double *y, double a, const double *x);
int k_waxpy(int n, double *w, double a, const double *x, const double *y);
int k_pmax(int n, double *w, const double *x, const double *y);
int k_pmin(int n, double *w, const double *x, const double *y);
int k_dot(int n, const double *x, const double *y, RedBuf rb);          // rb.out[0] = local x.y
int k_mdot2(int n, const double *x, const double *y0, const double *y1, RedBuf rb);   // out[0]=x.y0, out[1]=x.y1
int k_cg_update(int n, double a, const double *p, const double *w, double *x, double *r, RedBuf rb);   // x += a p; r -= a w; out[0] = r.r
int k_dense_rows_mult(int n, int m, const double *B, const double *x, RedBuf rb);     // out[j] = B_j . x
int k_dense_rows_multT_add(int n, int m, const double *B, const double *t /*device, m*/, double scale, double *y, int accumulate);
int k_rows_forward_solve(int n, int m, const double *L /*host, m x m lower*/, const double *G, double *TB);   // L TB = G, column by column
int k_scatter_is(int nis, const int *is, const double *sub, double fill, int n, double *full);  // full = fill; full[is]=sub

// QPC box (generic path and the public QPC* API)
int k_qpc_project(int n, const double *x, BoxDev bx, double *Px);
int k_qpc_grads(int n, const double *x, const double *g, BoxDev bx, double *gf, double *gc);
int k_qpc_gradreduced(int n, const double *x, const double *gf, double alpha, BoxDev bx, double *gr);
int k_qpc_feas(int n, const double *x, const double *d, BoxDev bx, RedBuf rb);        // out[RA_FEAS] = local min
int k_box_mult(int n, const double *r, int has_lb, int has_ub, double *llb, double *lub);
int k_kkt_box(int n, const double *x, const double *bound, const double *lam, int upper, RedBuf rb);

// SpMV
int k_power_step(const CsrDev &A, const double *w, double s, double *y, RedBuf rb);   // y = A (s w); rb.out[0] = (s w).y, rb.out[1] = (s w).(s w); packed matrices
int k_spmv(const CsrDev &A, const double *x, double *y, int accumulate);   // y (+)= A x ; honours A.rows

// ---- fused MPGP kernels -------------------------------------------------------------------------------
struct MpgpVecs {
  int     n = 0;
  double *x = nullptr, *g = nullptr, *p = nullptr, *Ap = nullptr, *gf = nullptr;
  const double *b = nullptr;
  BoxDev  bx;
  const double *B = nullptr;     // [m][n] dense equality rows (local columns), or NULL
  int     m = 0;
  double *t = nullptr;           // inner-dimension work vector for product operators
};
// K_A  : Ap = A xin (xin = p, or t for product operators) + [p.Ap, g.p, B p, alpha_f]
int k_fused_A(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm);
// K_A' : g = A xin - b (+rho B^T Bu), split, p = gf, [|gP|^2, |gc|^2, |gf|^2]; runs when step=='e' or init
int k_fused_A2(const CsrDev &A, const double *xin, const MpgpVecs &v, const MpgpCtl *S, RedBuf rb, const GhostMerge &gm);
// peer-memory halo push (which: 0 = p before K_A, 1 = x before K_A' [gated on step 'e' / init])
int k_halo_push(const HaloPush &hp, const double *vec, int gated, unsigned long long seq, const MpgpCtl *S);
// ctrl kernels that first wait for every rank's pushed record (peer-memory all-gather)
int k_ctrl_A_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq);
int k_ctrl_E_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq);
int k_ctrl_B_p2p(MpgpCtl *S, const P2PWin *win, const double *my_slot, const unsigned long long *my_flag, unsigned long long seq1, unsigned long long seq2);
// K_B  : the c / p / e update of x, g (+ split, reductions)
int k_fused_B(const MpgpVecs &v, const CtrlFold &cf, RedBuf rb, const PushRanges *d_push_x, unsigned long long push_seq);   // d_push_x: device memory or NULL
// K_C  : direction update p = gf - bcg p | p = gc | nothing
int k_fused_C(const MpgpVecs &v, const CtrlFold &cf, RedBuf rc, const PushRanges *d_push_p, unsigned long long push_seq);   // rc.out[RA_GP] = local g.p of the new direction (CG steps)
// initial projection x = P(x) (+ B u)
int k_fused_project(const MpgpVecs &v, const MpgpCtl *S, RedBuf rb);
// plain product-operator first factor, device-driven: t = M2 xin when the phase is active
int k_spmv_gated(const CsrDev &A, const double *x, double *y, const MpgpCtl *S, int phase /*0: K_A, 1: K_A'*/);
// one-thread control kernels
int k_ctrl_A(MpgpCtl *S, const double *ra);
int k_ctrl_E(MpgpCtl *S, const double *rb);
int k_ctrl_B(MpgpCtl *S, const double *rb);
// halo pack: buf[k] = x[idx[k]]
int k_pack(int n, const int *idx, const double *x, double *buf);

double csr_stream_bytes(const CsrDev &A);   // bytes one SpMV must read for the matrix itself (CSR: 12 nnz + 4(n+1); packed: blob + directory)
int  spmv_config(CsrDev &A, const int *h_ia);   // picks kind / W / grid from the host row pointer (spmv_stats + spmv_decide)
void spmv_stats(int n, const int *h_ia, int *maxrow, int *tile_cap);   // longest row, most non-zeros of a 256-row tile
void spmv_decide(CsrDev &A, int maxrow, int tile_cap);                  // the kernel flavour from those statistics and A.nnz
int  csr_to_tile_ell(CsrDev &A, const int *h_ia);   // long-row matrices: re-lay the uploaded CSR out as tile-ELL (kind 5) on the device
int  csr_to_tile_ell_widths(CsrDev &A, const std::vector<int> &tile_maxrow);   // same, from the longest row of every tile
// all-stencil form (kind 4) on the device: sets the scalar fields of A from the pattern table (upload_stencil, recode.cu)
void stencil_set_fields(CsrDev &A, const std::vector<StPattern> &pats, int nwin, size_t masks_bytes, size_t npid);
// device re-coder (recode.cu): the stored form upload_csr builds from a host CSR, built on the device from a device CSR (int32
// row pointer, column ids in [0, ncols), fp64 values).  The caller's arrays are only read, unless own_ia / own_ja / own_a are given:
// library-owned arrays padded like upload_csr's (8 zero elements behind each) that a matrix staying CSR adopts (the pointers are then
// set to NULL; whatever is left non-NULL still belongs to the caller)
int  recode_csr_dev(CsrDev &A, int nrows, int ncols, const int *d_ia, const int *d_ja, const double *d_a, int **own_ia = nullptr, int **own_ja = nullptr,
                    double **own_a = nullptr);
// all-stencil form of the diagonal block [c0, c0 + ncols) of a row-partitioned device CSR with GLOBAL columns, straight from the caller's
// arrays (pk_stencil_windowed); *done = false when some tile is not a stencil tile or there are too many patterns
int  recode_stencil_window_dev(CsrDev &A, int m, const int *d_ia, const int *d_ja, const double *d_a, int c0, int ncols, bool *done);
// row-partitioned device CSR with GLOBAL columns: the ghost entries (row, global column, value) in storage order on the host and, with
// want_diag, the diagonal block [c0, c0 + ncols) as a padded device CSR with local columns (library-owned, released with dfree)
int  split_rows_dev(int m, const int *d_ia, const int *d_ja, const double *d_a, int c0, int ncols, bool want_diag, int **dia, int **dja, double **da,
                    OffDiagEntries &off);
// dense form (kind 6): rows per CTA and split-column chunk from (m, n, SM count) only, so that grids and reductions are reproducible
void dense_config(CsrDev &A);
int  elementwise_grid();
int  fused_C_grid(int n);   // CTAs of K_C for n local rows (K_A adds that many partial sums of g.p)
int  max_red_blocks();

}  // namespace pb
