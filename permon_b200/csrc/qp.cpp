// qp.cpp -- QPC (box), QPPF (projector factory on G = B_E), QP (problem container), the QP chain and the
// two QP transforms on the SMALXE path.  Host logic mirrors the reference; all arithmetic runs in CUDA
// kernels through the Vec/Mat layer (shim.cpp) -- there is no CPU path.
//
//   QPC   src/qpc/interface/qpc.c, src/qpc/impls/box/qpcbox.c
//   QPPF  src/qppf/interface/qppf.c            (+ MatMult_Inv  src/mat/impls/inv/matinv.c:734-743)
//   QP    src/qp/interface/qp.c, qpchain.c, qptransform.c:329-527, src/qp/utils/matpenalized.c
#include <math.h>
#include <string.h>

#include <algorithm>

#include "objects.h"

using namespace pb;

static int g_qp_ids = 0;

// =====================================================================================================
// QPC
// =====================================================================================================
_p_QPC::~_p_QPC()
{
  if (is && --is->refct == 0) {
    if (is->d_local) cudaFree(is->d_local);
    delete is;
  }
  pb::unref(lb);
  pb::unref(ub);
  pb::unref(llb);
  pb::unref(lub);
  pb::unref(lb_full);
  pb::unref(ub_full);
  pb::unref(lambdawork);
}

PetscErrorCode QPCCreate(MPI_Comm comm, QPC *qpc)
{
  _p_QPC *q = new _p_QPC;
  q->comm   = comm;
  q->astol  = 10 * PETSC_MACHINE_EPSILON;   // qpc.c:28
  *qpc      = q;
  return 0;
}
PetscErrorCode QPCDestroy(QPC *qpc)
{
  if (!qpc || !*qpc) return 0;
  pb::unref(*qpc);
  return 0;
}
PetscErrorCode QPCSetType(QPC qpc, const QPCType type)
{
  if (strcmp(type, QPCBOX)) return err(PETSC_ERR_ARG_UNKNOWN_TYPE, "unknown QPC type %s (only \"box\" is on the path)", type);
  qpc->type = type;
  return 0;
}
PetscErrorCode QPCGetType(QPC qpc, const QPCType *type)
{
  *(const char **)type = qpc->type.c_str();
  return 0;
}
PetscErrorCode QPCSetIS(QPC qpc, IS is)
{
  if (is) is->refct++;
  if (qpc->is && --qpc->is->refct == 0) delete qpc->is;
  qpc->is          = is;
  qpc->setupcalled = false;
  return 0;
}
PetscErrorCode QPCGetIS(QPC qpc, IS *is)
{
  *is = qpc->is;
  return 0;
}
PetscErrorCode QPCGetBlockSize(QPC, PetscInt *bs)
{
  *bs = 1;   // qpcbox.c:216
  return 0;
}
PetscErrorCode QPCGetNumberOfConstraints(QPC qpc, PetscInt *num)
{
  if (qpc->is) *num = (PetscInt)qpc->is->idx.size();
  else *num = qpc->lb ? qpc->lb->N : (qpc->ub ? qpc->ub->N : 0);
  return 0;
}
PetscErrorCode QPCBoxSet(QPC qpc, Vec lb, Vec ub)
{   // QPCBoxSet_Box qpcbox.c:150-172
  pb::ref(lb);
  pb::ref(ub);
  pb::unref(qpc->lb);
  pb::unref(qpc->ub);
  pb::unref(qpc->llb);
  pb::unref(qpc->lub);
  pb::unref(qpc->lb_full);
  pb::unref(qpc->ub_full);
  qpc->lb = lb;
  qpc->ub = ub;
  if (lb) {
    PB_CHK(VecDuplicate(lb, &qpc->llb));
    PB_CHK(VecInvalidate(qpc->llb));
  }
  if (ub) {
    PB_CHK(VecDuplicate(ub, &qpc->lub));
    PB_CHK(VecInvalidate(qpc->lub));
  }
  qpc->setupcalled = false;
  return 0;
}
PetscErrorCode QPCBoxGet(QPC qpc, Vec *lb, Vec *ub)
{
  if (lb) *lb = qpc->lb;
  if (ub) *ub = qpc->ub;
  return 0;
}
PetscErrorCode QPCBoxGetMultipliers(QPC qpc, Vec *llb, Vec *lub)
{
  if (llb) *llb = qpc->llb;
  if (lub) *lub = qpc->lub;
  return 0;
}
PetscErrorCode QPCCreateBox(MPI_Comm comm, IS is, Vec lb, Vec ub, QPC *qpc_new)
{   // qpcbox.c:554-571
  if (lb && ub && lb->n != ub->n) return err(PETSC_ERR_ARG_INCOMP, "lb and ub have different layouts");
  QPC qpc;
  PB_CHK(QPCCreate(comm, &qpc));
  PB_CHK(QPCSetIS(qpc, is));
  PB_CHK(QPCSetType(qpc, (char *)QPCBOX));
  PB_CHK(QPCBoxSet(qpc, lb, ub));
  *qpc_new = qpc;
  return 0;
}

// With an index set the bounds live on a sub-vector (QPCGetSubvector qpc.c:416-437).  On the device the
// same semantics are obtained by expanding them to the full local length with -inf / +inf outside the
// IS: those entries are never active (qpcbox.c:41,48), never reduce gf (:86-92), never limit the step
// (:126,132) and project to themselves (:298-303).
static int qpc_expand(QPC qpc, Vec sub, double fill, PetscInt nfull, PetscInt rstart, Vec *full)
{
  if (!sub) return 0;
  IS is = qpc->is;
  if (!is->d_local) {
    std::vector<int> loc(is->idx.size());
    for (size_t k = 0; k < loc.size(); k++) {
      loc[k] = is->idx[k] - rstart;
      if (loc[k] < 0 || loc[k] >= nfull) return err(PETSC_ERR_ARG_OUTOFRANGE, "IS index %d is not owned by this rank", (int)is->idx[k]);
    }
    PB_CHK(dev_init());
    PB_CUDA(cudaMalloc(&is->d_local, sizeof(int) * std::max<size_t>(loc.size(), 1)));
    PB_CUDA(cudaMemcpy(is->d_local, loc.data(), sizeof(int) * loc.size(), cudaMemcpyHostToDevice));
  }
  if ((size_t)sub->n != is->idx.size()) return err(PETSC_ERR_ARG_SIZ, "bound vector length %d differs from IS length %d", (int)sub->n, (int)is->idx.size());
  if (!*full) PB_CHK(vec_create(qpc->comm, nfull, PETSC_DECIDE, full));
  const double *ds;
  double       *df;
  PB_CHK(vec_dev_read(sub, &ds));
  PB_CHK(vec_dev_write(*full, &df));
  return k_scatter_is((int)is->idx.size(), is->d_local, ds, fill, nfull, df);
}

static int qpc_setup_for(QPC qpc, Vec x)
{
  if (!qpc->lb && !qpc->ub) return err(PETSC_ERR_ORDER, "QPC box has no bounds");
  if (qpc->is) {
    PB_CHK(qpc_expand(qpc, qpc->lb, PETSC_NINFINITY, x->n, x->rstart, &qpc->lb_full));
    PB_CHK(qpc_expand(qpc, qpc->ub, PETSC_INFINITY, x->n, x->rstart, &qpc->ub_full));
  }
  if (!qpc->lambdawork) {   // QPCSetUp_Box qpcbox.c:5-17
    PB_CHK(VecDuplicate(qpc->lb ? qpc->lb : qpc->ub, &qpc->lambdawork));
    PB_CHK(VecSet(qpc->lambdawork, 0.0));
  }
  qpc->setupcalled = true;
  return 0;
}
PetscErrorCode QPCSetUp(QPC qpc)
{
  if (qpc->setupcalled) return 0;
  if (qpc->is) return 0;   // needs the layout of x: done lazily by the first operation
  Vec ref = qpc->lb ? qpc->lb : qpc->ub;
  if (!ref) return err(PETSC_ERR_ORDER, "QPC box has no bounds");
  return qpc_setup_for(qpc, ref);
}

namespace pb {
int box_dev(QPC qpc, BoxDev *bx)
{
  bx->astol = qpc->astol;
  bx->lb = bx->ub = nullptr;
  Vec l = qpc->is ? qpc->lb_full : qpc->lb, u = qpc->is ? qpc->ub_full : qpc->ub;
  if (l) PB_CHK(vec_dev_read(l, &bx->lb));
  if (u) PB_CHK(vec_dev_read(u, &bx->ub));
  return 0;
}
}  // namespace pb

static int qpc_box_for(QPC qpc, Vec x, BoxDev *bx)
{
  if (!qpc->setupcalled || (qpc->is && !qpc->lb_full && !qpc->ub_full)) PB_CHK(qpc_setup_for(qpc, x));
  PB_CHK(box_dev(qpc, bx));
  Vec ref = qpc->is ? (qpc->lb_full ? qpc->lb_full : qpc->ub_full) : (qpc->lb ? qpc->lb : qpc->ub);
  if (ref->n != x->n) return err(PETSC_ERR_ARG_INCOMP, "bound vectors (%d) and x (%d) have different local sizes", (int)ref->n, (int)x->n);
  return 0;
}

namespace pb {
int qpc_box_for_vec(QPC qpc, Vec x, BoxDev *bx) { return qpc_box_for(qpc, x, bx); }
}  // namespace pb

PetscErrorCode QPCProject(QPC qpc, Vec x, Vec Px)
{   // qpc.c:466-491
  BoxDev bx;
  PB_CHK(qpc_box_for(qpc, x, &bx));
  const double *dx;
  double       *dp;
  if (x == Px) {
    PB_CHK(vec_dev_rw(Px, &dp));
    dx = dp;
  } else {
    PB_CHK(vec_dev_read(x, &dx));
    PB_CHK(vec_dev_write(Px, &dp));
  }
  return k_qpc_project(x->n, dx, bx, dp);
}
PetscErrorCode QPCGrads(QPC qpc, Vec x, Vec g, Vec gf, Vec gc)
{   // qpc.c:540-569
  BoxDev bx;
  PB_CHK(qpc_box_for(qpc, x, &bx));
  const double *dx, *dg;
  double       *df, *dc;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(g, &dg));
  PB_CHK(vec_dev_write(gf, &df));
  PB_CHK(vec_dev_write(gc, &dc));
  return k_qpc_grads(x->n, dx, dg, bx, df, dc);
}
PetscErrorCode QPCGradReduced(QPC qpc, Vec x, Vec gf, PetscReal alpha, Vec gr)
{   // qpc.c:589-615
  BoxDev bx;
  PB_CHK(qpc_box_for(qpc, x, &bx));
  const double *dx, *df;
  double       *dr;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(gf, &df));
  PB_CHK(vec_dev_write(gr, &dr));
  return k_qpc_gradreduced(x->n, dx, df, alpha, bx, dr);
}
PetscErrorCode QPCFeas(QPC qpc, Vec x, Vec d, PetscReal *alpha)
{   // qpc.c:503-527 (the MPI_Allreduce(MIN) of :521 is the rank-ordered min of the gathered records)
  BoxDev bx;
  PB_CHK(qpc_box_for(qpc, x, &bx));
  const double *dx, *dd;
  PB_CHK(vec_dev_read(x, &dx));
  PB_CHK(vec_dev_read(d, &dd));
  Reducer &R = reducer(x->comm);
  PB_CHK(k_qpc_feas(x->n, dx, dd, bx, R.rb));
  PB_CHK(R.gather());
  PB_CHK(R.fetch());
  double a = R.min(RA_FEAS);
  *alpha   = (a > PETSC_INFINITY) ? PETSC_INFINITY : a;   // alpha_temp starts at PETSC_INFINITY (qpcbox.c:117)
  return 0;
}

// QPCViewKKT_Box: qpcbox.c:333-427
PetscErrorCode QPCViewKKT(QPC qpc, Vec x, PetscReal normb, PetscViewer v)
{
  BoxDev bx;
  PB_CHK(qpc_box_for(qpc, x, &bx));
  const double *dx;
  PB_CHK(vec_dev_read(x, &dx));
  Reducer &R = reducer(x->comm);
  for (int upper = 0; upper < 2; upper++) {
    Vec bound = upper ? qpc->ub : qpc->lb, lam = upper ? qpc->lub : qpc->llb;
    if (!bound) continue;
    const double *dbound = upper ? bx.ub : bx.lb, *dl;
    Vec           lamfull = lam, tmp = nullptr;
    if (qpc->is) {   // multipliers live on the IS: expand with zeros
      PB_CHK(qpc_expand(qpc, lam, 0.0, x->n, x->rstart, &tmp));
      lamfull = tmp;
    }
    PB_CHK(vec_dev_read(lamfull, &dl));
    PB_CHK(k_kkt_box(x->n, dx, dbound, dl, upper, R.rb));
    PB_CHK(R.gather());
    PB_CHK(R.fetch());
    double r0 = sqrt(R.sum(0)), r1 = sqrt(R.sum(1)), r2 = fabs(R.sum(2));
    pb::unref(tmp);
    if (!upper) {
      vprintf_viewer(v, "r = ||min(x-lb,0)||      = %.2e    r/||b|| = %.2e\n", r0, r0 / normb);
      vprintf_viewer(v, "r = ||min(lambda_lb,0)|| = %.2e    r/||b|| = %.2e\n", r1, r1 / normb);
      vprintf_viewer(v, "r = |lambda_lb'*(lb-x)|  = %.2e    r/||b|| = %.2e\n", r2, r2 / normb);
    } else {
      vprintf_viewer(v, "r = ||max(x-ub,0)||      = %.2e    r/||b|| = %.2e\n", r0, r0 / normb);
      vprintf_viewer(v, "r = ||min(lambda_ub,0)|| = %.2e    r/||b|| = %.2e\n", r1, r1 / normb);
      vprintf_viewer(v, "r = |lambda_ub'*(x-ub)|  = %.2e    r/||b|| = %.2e\n", r2, r2 / normb);
    }
  }
  return 0;
}

// =====================================================================================================
// QPPF
// =====================================================================================================
_p_QPPF::~_p_QPPF()
{
  pb::unref(G);
  if (Bd_owned && Bd) cudaFree(Bd);
  pb::unref(G_left);
  pb::unref(Gt_right);
  pb::unref(alpha_tilde);
  pb::unref(GGt_mat);
}
PetscErrorCode QPPFCreate(MPI_Comm comm, QPPF *cp)
{
  _p_QPPF *p = new _p_QPPF;
  p->comm = comm;
  *cp     = p;
  return 0;
}
PetscErrorCode QPPFDestroy(QPPF *cp)
{
  if (!cp || !*cp) return 0;
  pb::unref(*cp);
  return 0;
}
PetscErrorCode QPPFReset(QPPF cp)
{
  if (cp->Bd_owned && cp->Bd) cudaFree(cp->Bd);
  cp->Bd          = nullptr;
  cp->Bd_owned    = false;
  cp->setupcalled = false;
  cp->GGt.clear();
  cp->L.clear();
  cp->GGtinv.clear();
  pb::unref(cp->GGt_mat);
  cp->GGt_mat = nullptr;
  return 0;
}
PetscErrorCode QPPFSetExplicitInv(QPPF cp, PetscBool explicitInv)
{   // qppf.c:143-154
  if (cp->explicitInv != (explicitInv != PETSC_FALSE)) {
    cp->explicitInv = explicitInv != PETSC_FALSE;
    cp->setupcalled = false;
  }
  return 0;
}
PetscErrorCode QPPFSetRedundancy(QPPF cp, PetscInt nred)
{   // qppf.c:158-166.  The coarse problem (G G^T, m x m) is factored redundantly on EVERY rank here (the PCREDUNDANT end of the
    // reference's range, matinv.c:565-569): the value is recorded and reported back, it does not change the arithmetic.
  cp->redundancy = nred;
  return 0;
}
PetscErrorCode QPPFSetFromOptions(QPPF cp)
{   // qppf.c:170-188 (-qppf_explicit, -qppf_redundancy); -qppf_explicit_GGt (:237) is read as well: G G^T is always formed explicitly here
  bool     flg = cp->explicitInv;
  PetscInt nred = cp->redundancy;
  if (pb::options_bool(cp->prefix, "-qppf_explicit", &flg)) PB_CHK(QPPFSetExplicitInv(cp, flg ? PETSC_TRUE : PETSC_FALSE));
  if (pb::options_int(cp->prefix, "-qppf_redundancy", &nred)) PB_CHK(QPPFSetRedundancy(cp, nred));
  bool ggt = true;
  pb::options_bool(cp->prefix, "-qppf_explicit_GGt", &ggt);
  cp->setfromoptionscalled++;
  return 0;
}
PetscErrorCode QPPFSetG(QPPF cp, Mat G)
{   // qppf.c:116-138: a dummy left behind by the implicit orthonormalisation stands for its original matrix
  bool implicit = false;
  if (G && G->kind == MK_DUMMY && G->A) {
    G        = G->A;
    implicit = true;
  }
  if (G == cp->G && implicit == cp->implicit_orth) return 0;
  cp->implicit_orth = implicit;
  pb::ref(G);
  pb::unref(cp->G);
  cp->G = G;
  PB_CHK(QPPFReset(cp));
  return 0;
}
PetscErrorCode QPPFGetG(QPPF cp, Mat *G)
{
  *G = cp->G;
  return 0;
}

static int qppf_solve(QPPF cp, const double *r, double *y)
{   // (G G^T) y = r through the Cholesky factor (MatMult_Inv: KSPPREONLY + PCCHOLESKY, matinv.c:487-488,734-743)
  const int     m = cp->m;
  if (cp->explicitInv && !cp->GGtinv.empty()) {   // qppf.c:314-330: the explicit inverse applied as a matrix
    for (int i = 0; i < m; i++) {
      double v = 0.0;
      for (int k = 0; k < m; k++) v += cp->GGtinv[(size_t)i * m + k] * r[k];
      y[i] = v;
    }
    return 0;
  }
  const double *L = cp->L.data();
  for (int i = 0; i < m; i++) {
    double v = r[i];
    for (int k = 0; k < i; k++) v -= L[i * m + k] * y[k];
    y[i] = v / L[i * m + i];
  }
  for (int i = m - 1; i >= 0; i--) {
    double v = y[i];
    for (int k = i + 1; k < m; k++) v -= L[k * m + i] * y[k];
    y[i] = v / L[i * m + i];
  }
  return 0;
}

PetscErrorCode QPPFSetUp(QPPF cp)
{   // qppf.c:371-437
  if (cp->setupcalled) return 0;
  Mat G = cp->G;
  if (!G) return err(PETSC_ERR_ORDER, "QPPFSetG must be called first");
  PB_CHK(dev_init());
  cp->m = G->M;
  cp->n = G->n;
  if (cp->m > PB_MAXEQ_ALL) return err(PETSC_ERR_SUP, "at most %d equality rows are handled (got %d)", PB_MAXEQ_ALL, (int)cp->m);
  if (G->kind == MK_ONEROW) {
    const double *d;
    PB_CHK(vec_dev_read(G->row, &d));
    cp->Bd       = const_cast<double *>(d);
    cp->Bd_owned = false;
  } else if (G->kind == MK_DENSEROWS) {
    cp->Bd       = G->rows_d;
    cp->Bd_owned = false;
  } else if (G->kind == MK_AIJ && G->eq_host) {
    // row-partitioned AIJ equality matrix (several GPUs): re-distributed by columns into dense rows (shim.cpp: mat_eqrows_dense)
    PB_CHK(mat_eqrows_dense(G, &cp->Bd));
    cp->Bd_owned = false;
  } else if (G->kind == MK_DENSE) {
    // column-major m x n (m <= PB_MAXEQ_ALL, checked above) -> the row-major [m][n] rows: one strided device-to-device copy per row
    PB_CHK(mat_ensure_device(G));
    const int     m = G->m, n = G->n;
    const int64_t lda = G->Ad.dn_lda;
    PB_CUDA(cudaMalloc(&cp->Bd, sizeof(double) * std::max<size_t>((size_t)m * n, 1)));
    for (int r = 0; r < m && n > 0; r++)
      PB_CUDA(cudaMemcpy2DAsync(cp->Bd + (size_t)r * n, sizeof(double), G->Ad.dn_a + r, sizeof(double) * (size_t)lda, sizeof(double), (size_t)n,
                                cudaMemcpyDeviceToDevice, ctx().stream));
    PB_CUDA(cudaStreamSynchronize(ctx().stream));
    cp->Bd_owned = true;
  } else if (G->kind == MK_AIJ) {
    if (G->comm->size > 1) return err(PETSC_ERR_SUP, "a row-partitioned AIJ equality matrix may have at most %d rows", PB_MAXEQ_ALL);
    const int        m = G->m, n = G->n;
    std::vector<int> ia(m + 1), ja((size_t)G->Ad.nnz);
    std::vector<double> a((size_t)G->Ad.nnz), dense((size_t)m * n, 0.0);
    PB_CUDA(cudaMemcpy(ia.data(), G->Ad.ia, sizeof(int) * (m + 1), cudaMemcpyDeviceToHost));
    PB_CUDA(cudaMemcpy(ja.data(), G->Ad.ja, sizeof(int) * ja.size(), cudaMemcpyDeviceToHost));
    PB_CUDA(cudaMemcpy(a.data(), G->Ad.a, sizeof(double) * a.size(), cudaMemcpyDeviceToHost));
    for (int r = 0; r < m; r++)
      for (int k = ia[r]; k < ia[r + 1]; k++) dense[(size_t)r * n + ja[k]] += a[k];   // layout change only
    PB_CUDA(cudaMalloc(&cp->Bd, sizeof(double) * std::max<size_t>(dense.size(), 1)));
    PB_CUDA(cudaMemcpy(cp->Bd, dense.data(), sizeof(double) * dense.size(), cudaMemcpyHostToDevice));
    cp->Bd_owned = true;
  } else {
    return err(PETSC_ERR_SUP, "unsupported equality matrix kind");
  }
  // G G^T (m x m) on the device, factor on the host (replicated on every rank: PCREDUNDANT, matinv.c:565-569)
  const int m = cp->m;
  cp->GGt.assign((size_t)m * m, 0.0);
  for (int i = 0; i < m; i++) PB_CHK(dense_rows_mult_host(cp->comm, cp->n, m, cp->Bd, cp->Bd + (size_t)i * cp->n, &cp->GGt[(size_t)i * m]));
  // MatHasOrthonormalRows(G, PETSC_SMALL, 3) (qppf.c:394, permonmatorth.c:551): the reference tests
  // G G^T v = v on 3 random vectors; m is tiny here so G G^T is compared with I entry by entry.
  cp->orth = true;
  for (int i = 0; i < m; i++)
    for (int j = 0; j < m; j++)
      if (fabs(cp->GGt[(size_t)i * m + j] - (i == j ? 1.0 : 0.0)) > PETSC_SMALL) cp->orth = false;
  cp->L = cp->GGt;
  for (int j = 0; j < m; j++) {
    double d = cp->L[j * m + j];
    for (int k = 0; k < j; k++) d -= cp->L[j * m + k] * cp->L[j * m + k];
    if (!(d > 0.0)) return err(PETSC_ERR_ARG_WRONG, "G G^T is not positive definite (dependent equality rows)");
    d = sqrt(d);
    cp->L[j * m + j] = d;
    for (int i = j + 1; i < m; i++) {
      double v = cp->L[i * m + j];
      for (int k = 0; k < j; k++) v -= cp->L[i * m + k] * cp->L[j * m + k];
      cp->L[i * m + j] = v / d;
    }
  }
  cp->GGtinv.clear();
  if (cp->explicitInv) {   // MatInvExplicitly (qppf.c:319): column j of the inverse = solve with the j-th unit vector
    std::vector<double> inv((size_t)m * m), e(m), y(m);
    for (int j = 0; j < m; j++) {
      std::fill(e.begin(), e.end(), 0.0);
      e[j] = 1.0;
      PB_CHK(qppf_solve(cp, e.data(), y.data()));
      for (int i = 0; i < m; i++) inv[(size_t)i * m + j] = y[i];
    }
    cp->GGtinv = inv;
  }
  cp->setupcalled = true;
  return 0;
}
PetscErrorCode QPPFGetGHasOrthonormalRows(QPPF cp, PetscBool *flg)
{   // qppf.c:732-740: explicitly or implicitly
  PB_CHK(QPPFSetUp(cp));
  *flg = (cp->orth || cp->implicit_orth) ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}

namespace pb {
int qppf_dense_rows(QPPF pf, const double **Bd, int *m)
{
  PB_CHK(QPPFSetUp(pf));
  if (pf->G->kind == MK_ONEROW) {   // the row Vec may have been edited on the host
    const double *d;
    PB_CHK(vec_dev_read(pf->G->row, &d));
    pf->Bd = const_cast<double *>(d);
  }
  *Bd = pf->Bd;
  *m  = pf->m;
  return 0;
}
}  // namespace pb

static int qppf_G_mult(QPPF cp, Vec v, double *t)
{   // t = G v  (m host values, identical on every rank)
  const double *dv;
  PB_CHK(vec_dev_read(v, &dv));
  if (v->n != cp->n) return err(PETSC_ERR_ARG_SIZ, "QPPF: vector has local size %d, G has %d columns", (int)v->n, (int)cp->n);
  return dense_rows_mult_host(cp->comm, cp->n, cp->m, cp->Bd, dv, t);
}
static int qppf_Gt_mult(QPPF cp, const double *t, Vec y)
{   // y = G^T t
  double *dy;
  PB_CHK(vec_dev_write(y, &dy));
  return dense_rows_multT_host(cp->comm, cp->n, cp->m, cp->Bd, t, 1.0, dy, 0);
}
static int mvec_get(Vec x, int m, double *t)
{   // m-vector on the host.  In the reference's layout rank 0 owns the m entries (MatCreateOneRow, onerow.c:97-113);
    // the values are replicated here with the set-up-time host exchange (MPI_Bcast in onerow.c:52).
  MPI_Comm c = x->comm;
  if (c->size == 1) {
    const double *h;
    PB_CHK(vec_host_read(x, &h));
    if (x->n != m) return err(PETSC_ERR_ARG_SIZ, "expected a vector of length %d", m);
    memcpy(t, h, sizeof(double) * m);
    return 0;
  }
  if (x->N != m) return err(PETSC_ERR_ARG_SIZ, "expected a vector of global length %d (got %d)", m, (int)x->N);
  if (!c->agi) return err(PETSC_ERR_ARG_WRONGSTATE, "communicator has no host exchange");
  const double *h = nullptr;
  if (x->n > 0) PB_CHK(vec_host_read(x, &h));
  std::vector<int64_t> all(c->size);
  for (int j = 0; j < m; j++) {
    // entry j lives on the rank whose ownership range contains it
    const bool mine = (j >= x->rstart && j < x->rstart + x->n);
    int64_t    bits = 0;
    if (mine) memcpy(&bits, &h[j - x->rstart], 8);
    if (c->agi(c->agctx, mine ? bits : 0, all.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
    std::vector<int64_t> own(c->size);
    if (c->agi(c->agctx, mine ? 1 : 0, own.data())) return err(PETSC_ERR_LIB, "host all-gather failed");
    for (int r = 0; r < c->size; r++)
      if (own[r]) memcpy(&t[j], &all[r], 8);
  }
  return 0;
}
static int mvec_put(Vec y, int m, const double *t)
{   // every rank holds all m values; each stores the entries of its ownership range (rank 0 owns everything in the MatCreateOneRow layout,
    // a row-partitioned B_E spreads them like its rows)
  if (y->n == 0) return 0;
  const bool whole = (y->comm->size == 1) || (y->N == m);
  if ((y->comm->size == 1 && y->n != m) || !whole || y->rstart + y->n > m) return err(PETSC_ERR_ARG_SIZ, "expected a vector of (global) length %d", m);
  double *h;
  PB_CHK(vec_host_write(y, &h));
  memcpy(h, t + (y->comm->size == 1 ? 0 : y->rstart), sizeof(double) * y->n);
  return 0;
}

PetscErrorCode QPPFApplyCP(QPPF cp, Vec x, Vec y)
{   // qppf.c:610-645
  PB_CHK(QPPFSetUp(cp));
  double r[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(mvec_get(x, cp->m, r));
  PB_CHK(qppf_solve(cp, r, s));
  return mvec_put(y, cp->m, s);
}
PetscErrorCode QPPFApplyGtG(QPPF cp, Vec v, Vec GtGv)
{   // qppf.c:580-605 (with explicitly orthonormal rows the reference routes through ApplyQ = G^T (G v) as well; with IMPLICITLY
    // orthonormal rows ApplyQ = G^T (G G^T)^{-1} G v is the product with the orthonormalised matrix, :586-589)
  PB_CHK(QPPFSetUp(cp));
  if (cp->implicit_orth) return QPPFApplyQ(cp, v, GtGv);
  double t[PB_MAXEQ_ALL];
  PB_CHK(qppf_G_mult(cp, v, t));
  return qppf_Gt_mult(cp, t, GtGv);
}
static int qppf_store_alpha_tilde(QPPF cp, const double *s)
{   // qppf.c:486-487: alpha_tilde = (G G^T)^{-1} G v of the last Q / P application (an m-vector: rank 0 owns the entries, onerow.c:97-113)
  if (!cp->alpha_tilde) {
    const int nloc = (cp->comm->rank == 0) ? (int)cp->m : 0;
    PB_CHK(VecCreateMPI(cp->comm, nloc, cp->m, &cp->alpha_tilde));
  }
  return mvec_put(cp->alpha_tilde, cp->m, s);
}
PetscErrorCode QPPFGetAlphaTilde(QPPF cp, Vec *alpha_tilde)
{   // qppf.c:441-449 (borrowed pointer; NULL before the first application, like the reference before QPPFSetUp)
  *alpha_tilde = cp->alpha_tilde;
  return 0;
}
PetscErrorCode QPPFApplyQ(QPPF cp, Vec v, Vec Qv)
{   // qppf.c:454-502
  PB_CHK(QPPFSetUp(cp));
  double t[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(qppf_G_mult(cp, v, t));
  if (!cp->orth) PB_CHK(qppf_solve(cp, t, s));
  else memcpy(s, t, sizeof(double) * cp->m);
  PB_CHK(qppf_store_alpha_tilde(cp, s));
  return qppf_Gt_mult(cp, s, Qv);
}
PetscErrorCode QPPFApplyP(QPPF cp, Vec v, Vec Pv)
{   // qppf.c:572: Pv = v - Q v
  PB_CHK(QPPFApplyQ(cp, v, Pv));
  return VecAYPX(Pv, -1.0, v);
}
namespace pb {
int qppf_apply_P_dev(QPPF cp, const double *x, double *y)
{   // QPPFMatMult_P -> QPPFApplyP (qppf.c:560-575): y = x - G^T (G G^T)^{-1} G x
  PB_CHK(QPPFSetUp(cp));
  double t[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(dense_rows_mult_host(cp->comm, cp->n, cp->m, cp->Bd, x, t));
  if (!cp->orth) PB_CHK(qppf_solve(cp, t, s));
  else memcpy(s, t, sizeof(double) * cp->m);
  PB_CHK(dense_rows_multT_host(cp->comm, cp->n, cp->m, cp->Bd, s, 1.0, y, 0));   // y = Q x
  return k_aypx(cp->n, y, -1.0, x);                                            // VecAYPX(Pv, -1, v)
}
int qppf_coarse_solve(QPPF cp, const double *r, double *y)
{
  PB_CHK(QPPFSetUp(cp));
  return qppf_solve(cp, r, y);
}
int qppf_apply_mode_dev(QPPF cp, int mode, const double *x, double *y)
{   // the shell operators of qppf.c:648-718: 0 P, 1 Q = G^T (G G^T)^{-1} G, 2 G^T G
  if (mode == 0) return qppf_apply_P_dev(cp, x, y);
  PB_CHK(QPPFSetUp(cp));
  double t[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(dense_rows_mult_host(cp->comm, cp->n, cp->m, cp->Bd, x, t));
  if ((mode == 1 || cp->implicit_orth) && !cp->orth) PB_CHK(qppf_solve(cp, t, s));
  else memcpy(s, t, sizeof(double) * cp->m);
  return dense_rows_multT_host(cp->comm, cp->n, cp->m, cp->Bd, s, 1.0, y, 0);
}
}   // namespace pb

static int qppf_create_shell(QPPF cp, int mode, Mat *out)
{
  if (!cp->G) return err(PETSC_ERR_ORDER, "QPPFSetG must be called first");
  _p_Mat *P = new _p_Mat;
  P->comm      = cp->comm;
  P->kind      = MK_PROJ;
  P->proj_mode = mode;
  P->pf        = cp;
  cp->refct++;
  P->m = P->n = cp->G->n;
  P->M = P->N = cp->G->N;
  *out        = P;
  return 0;
}
PetscErrorCode QPPFCreateQ(QPPF cp, Mat *newQ) { return qppf_create_shell(cp, 1, newQ); }         // qppf.c:650-663
PetscErrorCode QPPFCreateGtG(QPPF cp, Mat *newGtG) { return qppf_create_shell(cp, 2, newGtG); }   // qppf.c:705-718
PetscErrorCode QPPFGetGGt(QPPF cp, Mat *GGt)
{   // qppf.c:744-755: the coarse-problem matrix (NULL when the explicit inverse replaced it or G has orthonormal rows, :225-229)
  *GGt = nullptr;
  PB_CHK(QPPFSetUp(cp));
  if (cp->explicitInv || cp->orth) return 0;
  if (!cp->GGt_mat) {
    const int m = cp->m;
    _p_Mat   *T = new _p_Mat;
    T->comm = cp->comm;
    T->kind = MK_DENSEROWS;
    T->m = T->n = T->M = T->N = m;
    // rows_d of a dense-rows Mat comes from the pool (its destructor returns it there): stream-ordered allocation and copy
    PB_CHK(pb::dmalloc(&T->rows_d, std::max<size_t>((size_t)m * m, 1)));
    PB_CUDA(cudaMemcpyAsync(T->rows_d, cp->GGt.data(), sizeof(double) * (size_t)m * m, cudaMemcpyHostToDevice, pb::ctx().stream));
    PB_CUDA(cudaStreamSynchronize(pb::ctx().stream));
    cp->GGt_mat = T;
  }
  *GGt = cp->GGt_mat;
  return 0;
}

PetscErrorCode QPPFCreateP(QPPF cp, Mat *newP)
{   // qppf.c:685-700: P = I - G' inv(G G') G in implicit form
  if (!cp->G) return err(PETSC_ERR_ORDER, "QPPFSetG must be called first");
  _p_Mat *P = new _p_Mat;
  P->comm   = cp->comm;
  P->kind   = MK_PROJ;
  P->pf     = cp;
  cp->refct++;
  P->m = P->n = cp->G->n;
  P->M = P->N = cp->G->N;
  *newP       = P;
  return 0;
}

PetscErrorCode QPPFApplyHalfQ(QPPF cp, Vec x, Vec y)
{   // qppf.c:507-530: y = (G G^T)^{-1} G x
  PB_CHK(QPPFSetUp(cp));
  double t[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(qppf_G_mult(cp, x, t));
  PB_CHK(qppf_solve(cp, t, s));
  return mvec_put(y, cp->m, s);
}
PetscErrorCode QPPFApplyHalfQTranspose(QPPF cp, Vec x, Vec y)
{   // qppf.c:535-568: y = G^T (G G^T)^{-1} x
  PB_CHK(QPPFSetUp(cp));
  double r[PB_MAXEQ_ALL], s[PB_MAXEQ_ALL];
  PB_CHK(mvec_get(x, cp->m, r));
  if (!cp->orth) PB_CHK(qppf_solve(cp, r, s));
  else memcpy(s, r, sizeof(double) * cp->m);
  return qppf_Gt_mult(cp, s, y);
}

// =====================================================================================================
// QP
// =====================================================================================================
_p_QP::~_p_QP()
{
  pb::unref(A);
  pb::unref(b);
  pb::unref(x);
  pb::unref(xwork);
  pb::unref(BE);
  pb::unref(cE);
  pb::unref(lambda_E);
  pb::unref(Bt_lambda);
  pb::unref(qpc);
  pb::unref(pf);
  pb::unref(postSolveCtx);
}

static int qp_changed(QP qp)
{
  qp->setupcalled = false;
  if (qp->changeListener) return qp->changeListener(qp);
  return 0;
}

PetscErrorCode QPCreate(MPI_Comm comm, QP *qp_new)
{
  _p_QP *qp = new _p_QP;
  qp->comm  = comm;
  qp->id    = g_qp_ids++;
  *qp_new   = qp;
  return 0;
}
PetscErrorCode QPRemoveChild(QP qp)
{
  if (!qp->child) return 0;
  QP c = qp->child;
  QPRemoveChild(c);
  c->parent = nullptr;
  qp->child = nullptr;
  pb::unref(c);
  return 0;
}
PetscErrorCode QPDestroy(QP *qp)
{
  if (!qp || !*qp) return 0;
  if ((*qp)->refct == 1) QPRemoveChild(*qp);
  pb::unref(*qp);
  return 0;
}
PetscErrorCode QPSetOperator(QP qp, Mat A)
{   // qp.c:1086-1100
  if (A == qp->A) return 0;
  if (A->M != A->N) return err(PETSC_ERR_ARG_SIZ, "the Hessian must be square (%d x %d)", (int)A->M, (int)A->N);
  pb::ref(A);
  pb::unref(qp->A);
  qp->A = A;
  return qp_changed(qp);
}
PetscErrorCode QPSetRhs(QP qp, Vec b)
{   // qp.c:1259-1280
  if (b == qp->b && !qp->b_plus) return 0;
  pb::ref(b);
  pb::unref(qp->b);
  qp->b      = b;
  qp->b_plus = false;
  return qp_changed(qp);
}
PetscErrorCode QPSetRhsPlus(QP qp, Vec b)
{   // qp.c:1296-1316: objective 1/2 x'Ax + x'b  =>  store -b
  Vec nb;
  PB_CHK(VecDuplicate(b, &nb));
  PB_CHK(VecCopy(b, nb));
  PB_CHK(VecScale(nb, -1.0));
  pb::unref(qp->b);
  qp->b      = nb;
  qp->b_plus = true;
  return qp_changed(qp);
}
PetscErrorCode QPSetInitialVector(QP qp, Vec x)
{   // qp.c:1978-1995: the user's Vec is the solution storage
  if (x == qp->x) return 0;
  pb::ref(x);
  pb::unref(qp->x);
  qp->x = x;
  return qp_changed(qp);
}
PetscErrorCode QPSetQPC(QP qp, QPC qpc)
{
  if (qpc == qp->qpc) return 0;
  pb::ref(qpc);
  pb::unref(qp->qpc);
  qp->qpc = qpc;
  return qp_changed(qp);
}
PetscErrorCode QPGetQPC(QP qp, QPC *qpc)
{
  *qpc = qp->qpc;
  return 0;
}
PetscErrorCode QPSetBox(QP qp, IS is, Vec lb, Vec ub)
{   // qp.c:1858-1882
  if (lb || ub) {
    QPC qpc;
    PB_CHK(QPCCreateBox(qp->comm, is, lb, ub, &qpc));
    PB_CHK(QPSetQPC(qp, qpc));
    PB_CHK(QPCDestroy(&qpc));
  }
  return qp_changed(qp);
}
PetscErrorCode QPGetBox(QP qp, IS *is, Vec *lb, Vec *ub)
{
  if (qp->qpc) {
    PB_CHK(QPCBoxGet(qp->qpc, lb, ub));
    if (is) *is = qp->qpc->is;
  } else {
    if (is) *is = nullptr;
    if (lb) *lb = nullptr;
    if (ub) *ub = nullptr;
  }
  return 0;
}
PetscErrorCode QPGetQPPF(QP qp, QPPF *pf)
{
  if (!qp->pf) PB_CHK(QPPFCreate(qp->comm, &qp->pf));
  *pf = qp->pf;
  return 0;
}
static int qp_set_qppf(QP qp, QPPF pf)
{
  pb::ref(pf);
  pb::unref(qp->pf);
  qp->pf = pf;
  return 0;
}
PetscErrorCode QPSetEq(QP qp, Mat Beq, Vec ceq)
{   // qp.c:1467-1528
  bool change = false;
  if (Beq != qp->BE) {
    if (Beq) {
      QPPF pf;
      PB_CHK(QPGetQPPF(qp, &pf));
      PB_CHK(QPPFSetG(pf, Beq));
      pb::ref(Beq);
    }
    pb::unref(qp->BE);
    pb::unref(qp->lambda_E);
    pb::unref(qp->Bt_lambda);
    qp->BE = Beq;
    change = true;
  }
  if (ceq) {
    if (!Beq) {
      ceq = nullptr;
    } else {
      double norm;
      PB_CHK(vec_norm2(ceq, &norm));
      if (norm < PETSC_MACHINE_EPSILON) ceq = nullptr;   // zero equality RHS detected (:1501-1504)
    }
  }
  if (ceq != qp->cE) {
    pb::ref(ceq);
    pb::unref(qp->cE);
    qp->cE = ceq;
    change = true;
  }
  if (!Beq) pb::unref(qp->lambda_E);
  return change ? qp_changed(qp) : 0;
}
PetscErrorCode QPSetOptionsPrefix(QP qp, const char prefix[])
{
  qp->prefix = prefix ? prefix : "";
  return 0;
}
PetscErrorCode QPSetFromOptions(QP qp)
{   // qp.c:2480-2490: only records the request; the objects that exist at QPSetUp time read their options there (QPSetFromOptions_Private,
    // qp.c:2448-2465: the QPPF inherits the QP's prefix and reads -qppf_*); -qp_chain_view_kkt is read at post-solve
  qp->setfromoptionscalled = true;
  qp->setupcalled          = false;
  return 0;
}
PetscErrorCode QPGetSolutionVector(QP qp, Vec *x)
{
  *x = qp->x;
  return 0;
}
PetscErrorCode QPGetOperator(QP qp, Mat *A)
{
  *A = qp->A;
  return 0;
}
PetscErrorCode QPGetRhs(QP qp, Vec *b)
{
  *b = qp->b;
  return 0;
}
PetscErrorCode QPGetEq(QP qp, Mat *Beq, Vec *ceq)
{
  if (Beq) *Beq = qp->BE;
  if (ceq) *ceq = qp->cE;
  return 0;
}
PetscErrorCode QPGetChild(QP qp, QP *child)
{
  *child = qp->child;
  return 0;
}
PetscErrorCode QPGetParent(QP qp, QP *parent)
{
  *parent = qp->parent;
  return 0;
}
PetscErrorCode QPIsSolved(QP qp, PetscBool *flg)
{
  *flg = qp->solved ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode QPGetEqMultiplier(QP qp, Vec *lambda_E, Vec *Bt_lambda)
{
  if (lambda_E) *lambda_E = qp->lambda_E;
  if (Bt_lambda) *Bt_lambda = qp->Bt_lambda;
  return 0;
}

// QPSetUpInnerObjects qp.c:492-598 (the parts that exist without PC / inequality constraints)
static int qp_setup_inner_objects(QP qp)
{
  if (!qp->A) return err(PETSC_ERR_ORDER, "Hessian must be set before QPSetUpInnerObjects");
  if (!qp->b) return err(PETSC_ERR_ORDER, "linear term must be set before QPSetUpInnerObjects");
  if (!qp->x) {   // QPInitializeInitialVector_Private qp.c:23-43
    if (!qp->parent || !qp->parent->x) {
      PB_CHK(MatCreateVecs(qp->A, &qp->x, NULL));
      PB_CHK(VecZeroEntries(qp->x));
    } else {
      PB_CHK(VecDuplicate(qp->parent->x, &qp->x));
      PB_CHK(VecCopy(qp->parent->x, qp->x));
    }
  }
  if (qp->x->n != qp->A->n || qp->b->n != qp->A->m) return err(PETSC_ERR_ARG_SIZ, "A (%d x %d local), b (%d) and x (%d) do not conform", (int)qp->A->m, (int)qp->A->n, (int)qp->b->n, (int)qp->x->n);
  if (!qp->xwork) PB_CHK(VecDuplicate(qp->x, &qp->xwork));
  if (qp->BE && !qp->lambda_E) {
    PB_CHK(vec_create(qp->comm, qp->BE->m, PETSC_DECIDE, &qp->lambda_E));
    PB_CHK(VecInvalidate(qp->lambda_E));
  }
  if (!qp->BE) pb::unref(qp->lambda_E);
  if (qp->BE && !qp->Bt_lambda) {
    PB_CHK(VecDuplicate(qp->x, &qp->Bt_lambda));
    PB_CHK(VecInvalidate(qp->Bt_lambda));
  }
  if (!qp->BE) pb::unref(qp->Bt_lambda);
  return 0;
}
PetscErrorCode QPSetUp(QP qp)
{   // qp.c:614-635
  if (qp->setupcalled) return 0;
  if (qp->setfromoptionscalled && qp->pf) {   // QPSetFromOptions_Private qp.c:2448-2465
    if (qp->pf->prefix.empty()) qp->pf->prefix = qp->prefix;
    PB_CHK(QPPFSetFromOptions(qp->pf));
  }
  PB_CHK(qp_setup_inner_objects(qp));
  qp->setupcalled = true;
  return 0;
}
PetscErrorCode QPChainGetLast(QP qp, QP *last)
{
  while (qp->child) qp = qp->child;
  *last = qp;
  return 0;
}
PetscErrorCode QPChainSetUp(QP qp)
{
  for (; qp; qp = qp->child) PB_CHK(QPSetUp(qp));
  return 0;
}

// QPComputeObjective qp.c:913-927: f = -x'(b - 1/2 A x)
PetscErrorCode QPComputeObjective(QP qp, Vec x, PetscReal *f)
{
  if (!qp->setupcalled) return err(PETSC_ERR_ORDER, "QPSetUp must be called first.");
  double dot;
  PB_CHK(mat_mult(qp->A, x, qp->xwork));
  PB_CHK(VecAYPX(qp->xwork, -0.5, qp->b));
  PB_CHK(vec_dot(x, qp->xwork, &dot));
  *f = -dot;
  return 0;
}
// QPComputeObjectiveFromGradient qp.c:981-996: f = x'(g - b)/2
PetscErrorCode QPComputeObjectiveFromGradient(QP qp, Vec x, Vec g, PetscReal *f)
{
  if (!qp->setupcalled) return err(PETSC_ERR_ORDER, "QPSetUp must be called first.");
  double dot;
  PB_CHK(VecWAXPY(qp->xwork, -1.0, qp->b, g));
  PB_CHK(vec_dot(x, qp->xwork, &dot));
  *f = .5 * dot;
  return 0;
}

// r = A x - b [- lambda_lb + lambda_ub] [+ B^T lambda]   (QPComputeLagrangianGradient qp.c:668-775)
static int lagrangian_gradient(QP qp, Vec x, Vec r, bool with_box, bool with_eq, bool *avail, std::string *name)
{
  *avail = true;
  *name  = "A*x - b";
  PB_CHK(QPSetUp(qp));
  PB_CHK(mat_mult(qp->A, x, r));
  PB_CHK(VecAXPY(r, -1.0, qp->b));
  QPC qpc = qp->qpc;
  if (with_box && qpc) {
    for (int upper = 0; upper < 2; upper++) {
      Vec bound = upper ? qpc->ub : qpc->lb, lam = upper ? qpc->lub : qpc->llb;
      if (!bound) continue;
      if (qpc->is) {
        Vec full = nullptr;
        PB_CHK(qpc_expand(qpc, lam, 0.0, x->n, x->rstart, &full));
        PB_CHK(VecAXPY(r, upper ? 1.0 : -1.0, full));
        pb::unref(full);
      } else {
        PB_CHK(VecAXPY(r, upper ? 1.0 : -1.0, lam));
      }
    }
  }
  if (with_eq && qp->BE) {
    if (qp->Bt_lambda && !pb::vec_invalid(qp->Bt_lambda)) {
      PB_CHK(VecAXPY(r, 1.0, qp->Bt_lambda));
      *name += " + (B'*lambda)";
    } else if (qp->lambda_E && !pb::vec_invalid(qp->lambda_E) && qp->pf) {
      Vec t;
      PB_CHK(VecDuplicate(r, &t));
      double lam[PB_MAXEQ_ALL];
      PB_CHK(mvec_get(qp->lambda_E, qp->pf->m, lam));
      PB_CHK(QPPFSetUp(qp->pf));
      PB_CHK(qppf_Gt_mult(qp->pf, lam, t));
      PB_CHK(VecAXPY(r, 1.0, t));
      pb::unref(t);
      *name += " + B'*lambda";
    } else {
      *name += " + BE'*lambda_E";
      *avail = false;
    }
  }
  if (with_box && qpc) {
    if (qpc->lb) *name += " - lambda_lb";
    if (qpc->ub) *name += " + lambda_ub";
  }
  return 0;
}
PetscErrorCode QPComputeLagrangianGradient(QP qp, Vec x, Vec r, char *kkt_name[])
{
  bool        avail;
  std::string name;
  PB_CHK(lagrangian_gradient(qp, x, r, true, true, &avail, &name));
  if (!avail) PB_CHK(VecInvalidate(r));
  if (kkt_name) *kkt_name = strdup(name.c_str());
  return 0;
}

// QPComputeMissingBoxMultipliers qp.c:829-890
PetscErrorCode QPComputeMissingBoxMultipliers(QP qp)
{
  PB_CHK(QPSetUp(qp));
  QPC qpc = qp->qpc;
  if (!qpc || (!qpc->lb && !qpc->ub)) return 0;
  bool flg = qpc->lb && pb::vec_invalid(qpc->llb), flg2 = qpc->ub && pb::vec_invalid(qpc->lub);
  if (!flg && !flg2) return 0;
  bool        avail;
  std::string name;
  Vec         r = qp->xwork;
  PB_CHK(lagrangian_gradient(qp, qp->x, r, false, true, &avail, &name));   // QP duplicate without the QPC (:853-856)
  if (!avail) return 0;
  const double *dr;
  PB_CHK(vec_dev_read(r, &dr));
  Vec rs = r;
  Vec sub = nullptr;
  if (qpc->is) {   // VecISCopy(r, is, SCATTER_REVERSE, llb)
    PB_CHK(VecDuplicate(qpc->lb ? qpc->lb : qpc->ub, &sub));
    double *ds;
    PB_CHK(vec_dev_write(sub, &ds));
    PB_CHK(k_pack((int)qpc->is->idx.size(), qpc->is->d_local, dr, ds));
    rs = sub;
    PB_CHK(vec_dev_read(rs, &dr));
  }
  double *dl = nullptr, *du = nullptr;
  if (qpc->lb) PB_CHK(vec_dev_write(qpc->llb, &dl));
  if (qpc->ub) PB_CHK(vec_dev_write(qpc->lub, &du));
  PB_CHK(k_box_mult(rs->n, dr, qpc->lb != nullptr, qpc->ub != nullptr, dl, du));
  if (qpc->llb) qpc->llb->invalidated = false;
  if (qpc->lub) qpc->lub->invalidated = false;
  pb::unref(sub);
  return 0;
}

// QPComputeMissingEqMultiplier qp.c:778-825
PetscErrorCode QPComputeMissingEqMultiplier(QP qp)
{
  PB_CHK(QPSetUp(qp));
  if (!qp->BE) return 0;
  if (!pb::vec_invalid(qp->lambda_E)) return 0;
  if (qp->Bt_lambda && !pb::vec_invalid(qp->Bt_lambda)) return 0;
  bool        avail;
  std::string name;
  Vec         r = qp->xwork;
  PB_CHK(lagrangian_gradient(qp, qp->x, r, true, false, &avail, &name));   // QP duplicate without the equality (:796-799)
  // BE == B (no inequality constraints on this path): Bt_lambda = -r  (:802-804)
  PB_CHK(VecCopy(r, qp->Bt_lambda));
  PB_CHK(VecScale(qp->Bt_lambda, -1.0));
  qp->Bt_lambda->invalidated = false;
  return 0;
}

// QPViewKKT qp.c:245-370 (the lines the golden outputs grep for)
PetscErrorCode QPViewKKT(QP qp, PetscViewer v)
{
  double normb, norm;
  PB_CHK(vec_norm2(qp->b, &normb));
  vprintf_viewer(v, "QP Object: %s#%d in chain, derived by %s\n", qp->prefix.c_str(), qp->id, qp->transform_name.c_str());
  if (!qp->solved) vprintf_viewer(v, "*** WARNING: QP is not solved. ***\n");
  Vec r;
  PB_CHK(VecDuplicate(qp->b, &r));
  bool        avail;
  std::string name;
  PB_CHK(lagrangian_gradient(qp, qp->x, r, true, true, &avail, &name));
  if (avail) {
    PB_CHK(vec_norm2(r, &norm));
    vprintf_viewer(v, "r = ||%s|| = %.2e    rO/||b|| = %.2e\n", name.c_str(), norm, norm / normb);
  } else {
    vprintf_viewer(v, "r = ||%s|| not available\n", name.c_str());
  }
  pb::unref(r);
  if (qp->BE && qp->pf) {
    double t[PB_MAXEQ_ALL], s = 0.0;
    PB_CHK(QPPFSetUp(qp->pf));
    PB_CHK(qppf_G_mult(qp->pf, qp->x, t));
    if (qp->cE) {
      double c[PB_MAXEQ_ALL];
      PB_CHK(mvec_get(qp->cE, qp->pf->m, c));
      for (int j = 0; j < qp->pf->m; j++) t[j] -= c[j];
    }
    for (int j = 0; j < qp->pf->m; j++) s += t[j] * t[j];
    norm = sqrt(s);
    if (qp->cE) vprintf_viewer(v, "r = ||BE*x-cE||          = %.2e    r/||b|| = %.2e\n", norm, norm / normb);
    else vprintf_viewer(v, "r = ||BE*x||             = %.2e    r/||b|| = %.2e\n", norm, norm / normb);
  }
  if (qp->qpc) PB_CHK(QPCViewKKT(qp->qpc, qp->x, normb, v));
  return 0;
}
PetscErrorCode QPChainViewKKT(QP qp, PetscViewer v)
{
  vprintf_viewer(v, "=====================\n");
  QP   cqp;
  bool first = true;
  PB_CHK(QPChainGetLast(qp, &cqp));
  while (1) {
    if (!first) vprintf_viewer(v, "-------------------\n");
    first = false;
    PB_CHK(QPViewKKT(cqp, v));
    if (!cqp->parent || cqp == qp) break;
    cqp = cqp->parent;
  }
  vprintf_viewer(v, "=====================\n");
  return 0;
}

// QPChainPostSolve qpchain.c:200-275
PetscErrorCode QPChainPostSolve(QP qp)
{
  QP cqp;
  PB_CHK(QPChainGetLast(qp, &cqp));
  const bool solved = cqp->solved;
  bool       view = options_get(qp->prefix, "-qp_chain_view_kkt", nullptr) != 0;
  bool       first = true;
  if (view) vprintf_viewer(nullptr, "=====================\n");
  while (1) {
    PB_CHK(QPComputeMissingBoxMultipliers(cqp));
    PB_CHK(QPComputeMissingEqMultiplier(cqp));
    QP parent = cqp->parent;
    if (cqp->postSolve && parent) PB_CHK(cqp->postSolve(cqp, parent));
    if (view) {
      if (!first) vprintf_viewer(nullptr, "-------------------\n");
      first = false;
      PB_CHK(QPViewKKT(cqp, nullptr));
    }
    if (!parent) break;
    parent->solved = solved;
    if (cqp == qp) break;
    cqp = parent;
  }
  if (view) vprintf_viewer(nullptr, "=====================\n");
  return 0;
}

// ---- transforms ------------------------------------------------------------------------------------------
static int qp_chain_add(QP qp, QP *child_new, int transform, const char *name, QPPostSolveFn post)
{   // QPTransformBegin_Private qptransform.c:15-43
  PB_CHK(QPChainGetLast(qp, &qp));
  PB_CHK(qp_setup_inner_objects(qp));
  QP child;
  PB_CHK(QPCreate(qp->comm, &child));
  child->parent         = qp;
  qp->child             = child;
  child->transform      = transform;
  child->transform_name = name;
  child->postSolve      = post;
  child->prefix         = qp->prefix;
  if (qp->changeListener) PB_CHK(qp->changeListener(qp));
  *child_new = child;
  return 0;
}
static PetscErrorCode post_default(QP child, QP parent)
{   // QPDefaultPostSolve qptransform.c:47-55
  if (child->x == parent->x) return 0;
  return VecCopy(child->x, parent->x);
}
static PetscErrorCode post_penalty(QP, QP) { return 0; }   // qptransform.c:320-325
static PetscErrorCode post_homogenize(QP child, QP parent)
{   // qptransform.c:414-422: x_parent = x_child + xtilde
  return VecWAXPY(parent->x, 1.0, child->x, child->postSolveCtx);
}

static PetscErrorCode post_projector(QP child, QP parent)
{   // QPTEnforceEqByProjectorPostSolve_Private qptransform.c:57-93
  PB_CHK(post_default(child, parent));
  bool skip_lambda_E = true, skip_Bt_lambda = true;
  if (child->BE) {   // -qpt_project_inherit_eq_multipliers defaults to true
    skip_lambda_E  = !child->lambda_E || pb::vec_invalid(child->lambda_E);
    skip_Bt_lambda = !child->Bt_lambda || pb::vec_invalid(child->Bt_lambda);
  }
  if (skip_lambda_E && skip_Bt_lambda) return 0;
  Vec r = parent->xwork;
  PB_CHK(mat_mult(parent->A, parent->x, r));
  PB_CHK(VecAYPX(r, -1.0, parent->b));   // r = b - A x
  if (!skip_lambda_E) {                    // lambda_E1 = lambda_E2 + (B B')\B (b - A x)
    PB_CHK(QPPFApplyHalfQ(parent->pf, r, parent->lambda_E));
    PB_CHK(VecAXPY(parent->lambda_E, 1.0, child->lambda_E));
  }
  if (!skip_Bt_lambda) {                   // (B' lambda)_1 = (B' lambda)_2 + B' (B B')\B (b - A x)
    PB_CHK(QPPFApplyQ(parent->pf, r, parent->Bt_lambda));
    PB_CHK(VecAXPY(parent->Bt_lambda, 1.0, child->Bt_lambda));
  }
  return 0;
}

// QPTEnforceEqByProjector qptransform.c:215-316: child = (P A P, P b, box, eq kept) or, with equality constraints only,
// (P A, P b, unconstrained); P = I - B'(B B')^{-1} B through the QPPF.
PetscErrorCode QPTEnforceEqByProjector(QP qp)
{
  PB_CHK(QPChainGetLast(qp, &qp));
  if (!qp->BE) {
    pb::unref(qp->cE);
    return 0;
  }
  if (qp->cE) {   // non-zero right-hand side: homogenise first (:236-240)
    PB_CHK(QPTHomogenizeEq(qp));
    PB_CHK(QPChainGetLast(qp, &qp));
  }
  QP child;
  PB_CHK(qp_chain_add(qp, &child, 3, "QPTEnforceEqByProjector", post_projector));
  child->prefix += "proj_";
  const bool eqonly = !qp->qpc;
  QPPF       pf;
  PB_CHK(QPGetQPPF(qp, &pf));
  if (eqonly) {
    PB_CHK(QPSetEq(child, NULL, NULL));
  } else {
    PB_CHK(qp_set_qppf(child, pf));
    PB_CHK(QPSetEq(child, qp->BE, qp->cE));
  }
  if (qp->qpc) PB_CHK(QPSetBox(child, qp->qpc->is, qp->qpc->lb, qp->qpc->ub));
  Mat P, newA, arr[3];
  PB_CHK(QPPFCreateP(pf, &P));
  if (eqonly) {   // newA = P*A
    arr[0] = qp->A;
    arr[1] = P;
    PB_CHK(MatCreateProd(qp->comm, 2, arr, &newA));
  } else {        // newA = P*A*P
    arr[0] = P;
    arr[1] = qp->A;
    arr[2] = P;
    PB_CHK(MatCreateProd(qp->comm, 3, arr, &newA));
  }
  PB_CHK(QPSetOperator(child, newA));
  PB_CHK(MatDestroy(&newA));
  Vec newb;
  PB_CHK(VecDuplicate(qp->b, &newb));
  PB_CHK(mat_mult(P, qp->b, newb));   // newb = P*b
  PB_CHK(QPSetRhs(child, newb));
  PB_CHK(VecDestroy(&newb));
  PB_CHK(MatDestroy(&P));
  return 0;
}

static PetscErrorCode post_orthonormalize(QP, QP) { return 0; }   // QPTPostSolve_QPTOrthonormalizeEq :528-550: both branches are disabled upstream

// QPTOrthonormalizeEq qptransform.c:566-636 with MatOrthRows (permonmatorth.c:494-520) for the small dense G of this path:
// MAT_ORTH_GS = MatOrthColumns_GS_Default (:196-234), MAT_ORTH_CHOLESKY = MatOrthColumns_Cholesky_Default (:33-150).
// The orthonormalised rows are always formed explicitly (m <= 4 rows): `form` only selects how the reference stores T*BE.
PetscErrorCode QPTOrthonormalizeEq(QP qp, MatOrthType type, MatOrthForm form)
{
  (void)form;
  PB_CHK(QPChainGetLast(qp, &qp));
  if (!qp->BE) return 0;
  if (type == MAT_ORTH_NONE) return 0;
  if (type != MAT_ORTH_GS && type != MAT_ORTH_CHOLESKY && type != MAT_ORTH_IMPLICIT)
    return err(PETSC_ERR_SUP, "QPTOrthonormalizeEq: the B200 path provides MAT_ORTH_GS, MAT_ORTH_CHOLESKY and MAT_ORTH_IMPLICIT");
  if (type != MAT_ORTH_IMPLICIT) {
    if (qp->BE && qp->BE->M > PB_MAXEQ) return err(PETSC_ERR_SUP, "explicit QPTOrthonormalizeEq handles at most %d equality rows (got %d)", PB_MAXEQ, (int)qp->BE->M);
  }
  QPPF pf;
  PB_CHK(QPGetQPPF(qp, &pf));
  PB_CHK(QPPFSetUp(pf));
  const int m = pf->m, n = pf->n;
  QP        child;
  PB_CHK(qp_chain_add(qp, &child, 4, "QPTOrthonormalizeEq", post_orthonormalize));
  // QP_DUPLICATE_COPY_POINTERS: the child shares A, b, x, the box and the multipliers' layout with its parent
  PB_CHK(QPSetOperator(child, qp->A));
  PB_CHK(QPSetRhs(child, qp->b));
  if (qp->x) PB_CHK(QPSetInitialVector(child, qp->x));
  if (qp->qpc) PB_CHK(QPSetQPC(child, qp->qpc));
  if (type == MAT_ORTH_IMPLICIT) {
    // MatOrthRows_Implicit_Default (permonmatorth.c:176-192): nothing is computed -- T*BE is a dummy that remembers BE, the child's QPPF
    // works on the ORIGINAL rows and applies G^T G as Q = G^T (G G^T)^{-1} G (qppf.c:123-127,586-589); c_E stays as it is (:609-611)
    _p_Mat *D = new _p_Mat;
    D->comm   = qp->comm;
    D->kind   = MK_DUMMY;
    D->m      = qp->BE->m;
    D->M      = qp->BE->M;
    D->n      = qp->BE->n;
    D->N      = qp->BE->N;
    D->rstart = qp->BE->rstart;
    D->cstart = qp->BE->cstart;
    D->A      = qp->BE;
    pb::ref(qp->BE);
    PB_CHK(qp_set_qppf(child, nullptr));
    PB_CHK(QPSetEq(child, D, qp->cE));
    Mat dm = D;
    PB_CHK(MatDestroy(&dm));
    child->postT.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; i++) child->postT[(size_t)i * m + i] = 1.0;
    return 0;
  }
  // TBE
  _p_Mat *TB = new _p_Mat;
  TB->comm   = qp->comm;
  TB->kind   = MK_DENSEROWS;
  TB->m = TB->M = m;
  TB->n      = n;
  TB->N      = qp->BE->N;
  PB_CHK(dmalloc(&TB->rows_d, (size_t)m * std::max(n, 1)));
  std::vector<double> T((size_t)m * m, 0.0);
  for (int i = 0; i < m; i++) T[i * m + i] = 1.0;
  if (type == MAT_ORTH_CHOLESKY) {
    PB_CHK(k_rows_forward_solve(n, m, pf->L.data(), pf->Bd, TB->rows_d));
    // T = L^{-1}: forward solve of the identity, column by column (permonmatorth.c:111-117)
    const double *L = pf->L.data();
    for (int col = 0; col < m; col++)
      for (int i = 0; i < m; i++) {
        double v = (i == col) ? 1.0 : 0.0;
        for (int k = 0; k < i; k++) v -= L[i * m + k] * T[k * m + col];
        T[i * m + col] = v / L[i * m + i];
      }
  } else {
    PB_CHK(k_copy(m * n, pf->Bd, TB->rows_d));
    Reducer &R = reducer(qp->comm);
    auto     dot = [&](const double *x, const double *y, double *val) -> int {
      PB_CHK(k_dot(n, x, y, R.rb));
      PB_CHK(R.gather());
      PB_CHK(R.fetch());
      *val = R.sum(0);
      return 0;
    };
    for (int i = 0; i < m; i++) {
      double *q = TB->rows_d + (size_t)i * n;
      double  d, norm, norm_last, dots[PB_MAXEQ_ALL];
      PB_CHK(dot(q, q, &d));
      norm = sqrt(d);
      do {
        norm_last = norm;
        for (int j = 0; j < i; j++) {
          PB_CHK(dot(q, TB->rows_d + (size_t)j * n, &dots[j]));
          dots[j] = -dots[j];
        }
        for (int j = 0; j < i; j++) PB_CHK(k_axpy(n, q, dots[j], TB->rows_d + (size_t)j * n));
        for (int j = 0; j < i; j++)
          for (int k = 0; k < m; k++) T[i * m + k] += dots[j] * T[j * m + k];
        PB_CHK(dot(q, q, &d));
        norm = sqrt(d);
        if (norm < 1e2 * PETSC_MACHINE_EPSILON) {
          {
            Mat tbm = TB;
            MatDestroy(&tbm);
          }
          return err(PETSC_ERR_NOT_CONVERGED, "MatOrthColumns has not converged due to zero norm of the current column %d (i.e. columns 0 - %d are linearly dependent)", i, i);
        }
      } while (norm <= 0.5 * norm_last);
      PB_CHK(k_scale(n, q, 1.0 / norm));
      for (int k = 0; k < m; k++) T[i * m + k] *= 1.0 / norm;
    }
  }
  Vec TcE = nullptr;
  if (qp->cE) {   // TcE = T*cE (:610-613)
    double c[PB_MAXEQ_ALL], tc[PB_MAXEQ_ALL];
    PB_CHK(mvec_get(qp->cE, m, c));
    for (int i = 0; i < m; i++) {
      double s2 = 0.0;
      for (int k = 0; k < m; k++) s2 += T[i * m + k] * c[k];
      tc[i] = s2;
    }
    PB_CHK(VecDuplicate(qp->cE, &TcE));
    PB_CHK(mvec_put(TcE, m, tc));
  }
  PB_CHK(qp_set_qppf(child, nullptr));
  PB_CHK(QPSetEq(child, TB, TcE));   // QPPF re-created in QPSetEq
  {
    Mat tbm = TB;
    PB_CHK(MatDestroy(&tbm));
  }
  if (TcE) PB_CHK(VecDestroy(&TcE));
  child->postT = T;
  return 0;
}

PetscErrorCode MatCreatePenalized(QP qp, PetscReal rho, Mat *Arho_new)
{   // matpenalized.c:212-243
  if (!qp->A) return err(PETSC_ERR_ORDER, "A specified");
  QPPF pf;
  PB_CHK(QPGetQPPF(qp, &pf));
  _p_Mat *M = new _p_Mat;
  M->comm   = qp->comm;
  M->kind   = MK_PENALIZED;
  M->A      = qp->A;
  pb::ref(qp->A);
  M->pf = pf;
  pf->refct++;
  M->rho    = rho;
  M->m      = qp->A->m;
  M->n      = qp->A->n;
  M->M      = qp->A->M;
  M->N      = qp->A->N;
  M->rstart = qp->A->rstart;
  M->cstart = qp->A->cstart;
  *Arho_new = M;
  return 0;
}
PetscErrorCode MatPenalizedSetPenalty(Mat Arho, PetscReal rho)
{
  if (Arho->kind != MK_PENALIZED) return err(PETSC_ERR_ARG_WRONG, "not a penalized matrix");
  Arho->rho = rho;
  return 0;
}
PetscErrorCode MatPenalizedUpdatePenalty(Mat Arho, PetscReal rho_update)
{
  if (Arho->kind != MK_PENALIZED) return err(PETSC_ERR_ARG_WRONG, "not a penalized matrix");
  Arho->rho *= rho_update;
  return 0;
}
PetscErrorCode MatPenalizedGetPenalty(Mat Arho, PetscReal *rho)
{
  if (Arho->kind != MK_PENALIZED) return err(PETSC_ERR_ARG_WRONG, "not a penalized matrix");
  *rho = Arho->rho;
  return 0;
}

// QPTEnforceEqByPenalty qptransform.c:329-410
PetscErrorCode QPTEnforceEqByPenalty(QP qp, PetscReal rho_user, PetscBool rho_direct)
{
  if (!rho_user) return 0;
  PB_CHK(QPChainGetLast(qp, &qp));
  if (!qp->BE) {
    pb::unref(qp->cE);
    return 0;
  }
  if (qp->cE) {   // qptransform.c:352-360
    bool flg = false;
    options_bool("", "-qpt_homogenize_eq_always", &flg);
    if (flg) {
      PB_CHK(QPTHomogenizeEq(qp));
      PB_CHK(QPChainGetLast(qp, &qp));
    }
  }
  double   rho, maxeig_tol = PETSC_DECIDE;
  PetscInt maxeig_iter = PETSC_DECIDE;
  options_real("", "-qpt_penalize_maxeig_tol", &maxeig_tol);    // :362-363
  options_int("", "-qpt_penalize_maxeig_iter", &maxeig_iter);
  if (!rho_direct) {
    double maxeig;
    PB_CHK(MatGetMaxEigenvalue(qp->A, NULL, &maxeig, maxeig_tol, maxeig_iter));
    rho = rho_user * maxeig;
  } else {
    rho = rho_user;
  }
  if (!(rho >= 0)) return err(PETSC_ERR_ARG_WRONG, "rho must be nonnegative");
  QP child;
  PB_CHK(qp_chain_add(qp, &child, 1, "QPTEnforceEqByPenalty", post_penalty));
  child->prefix = qp->prefix + "pnlt_";
  PB_CHK(QPSetQPC(child, qp->qpc));
  PB_CHK(QPSetRhs(child, qp->b));
  PB_CHK(QPSetInitialVector(child, qp->x));   // shares x with the parent (:389)
  Mat newA;
  PB_CHK(MatCreatePenalized(qp, rho, &newA));
  PB_CHK(QPSetOperator(child, newA));
  PB_CHK(MatDestroy(&newA));
  if (qp->cE) {   // newb = b + rho BE' c  (:396-401)
    Vec newb;
    PB_CHK(VecDuplicate(qp->b, &newb));
    double c[PB_MAXEQ_ALL];
    PB_CHK(QPPFSetUp(qp->pf));
    PB_CHK(mvec_get(qp->cE, qp->pf->m, c));
    PB_CHK(qppf_Gt_mult(qp->pf, c, newb));
    PB_CHK(VecAYPX(newb, rho, qp->b));
    PB_CHK(QPSetRhs(child, newb));
    PB_CHK(VecDestroy(&newb));
  }
  pb::ref(qp->xwork);
  pb::unref(child->xwork);
  child->xwork = qp->xwork;   // QPSetWorkVector (:404)
  return 0;
}

// QPTHomogenizeEq qptransform.c:437-527
PetscErrorCode QPTHomogenizeEq(QP qp)
{
  PB_CHK(QPChainGetLast(qp, &qp));
  if (!qp->cE) return 0;
  QP child;
  PB_CHK(qp_chain_add(qp, &child, 2, "QPTHomogenizeEq", post_homogenize));
  // QP_DUPLICATE_COPY_POINTERS: the child starts as a copy of the parent's pointers
  PB_CHK(QPSetOperator(child, qp->A));
  Vec xtilde, b_bar;
  PB_CHK(VecDuplicate(qp->x, &xtilde));
  PB_CHK(QPPFApplyHalfQTranspose(qp->pf, qp->cE, xtilde));   // xtilde = BE' inv(BE BE') cE  (:465)
  PB_CHK(VecDuplicate(qp->b, &b_bar));
  PB_CHK(mat_mult(qp->A, xtilde, b_bar));
  PB_CHK(VecAYPX(b_bar, -1.0, qp->b));                        // b_bar = b - A xtilde       (:469)
  PB_CHK(QPSetRhs(child, b_bar));
  PB_CHK(VecDestroy(&b_bar));
  PB_CHK(qp_set_qppf(child, qp->pf));                         // :487
  PB_CHK(QPSetEq(child, qp->BE, NULL));                       // cE is eliminated           (:488)
  QPC qpc = qp->qpc;
  if (qpc) {
    Vec lbnew = nullptr, ubnew = nullptr, xs = xtilde, sub = nullptr;
    if (qpc->is) {   // VecGetSubVector(xtilde, is)
      PB_CHK(qpc_setup_for(qpc, qp->x));
      PB_CHK(VecDuplicate(qpc->lb ? qpc->lb : qpc->ub, &sub));
      const double *dx;
      double       *ds;
      PB_CHK(vec_dev_read(xtilde, &dx));
      PB_CHK(vec_dev_write(sub, &ds));
      PB_CHK(k_pack((int)qpc->is->idx.size(), qpc->is->d_local, dx, ds));
      xs = sub;
    }
    if (qpc->lb) {
      PB_CHK(VecDuplicate(qpc->lb, &lbnew));
      PB_CHK(VecWAXPY(lbnew, -1.0, xs, qpc->lb));   // lb - xtilde  (:499-500)
    }
    if (qpc->ub) {
      PB_CHK(VecDuplicate(qpc->ub, &ubnew));
      PB_CHK(VecWAXPY(ubnew, -1.0, xs, qpc->ub));   // ub - xtilde  (:504-505)
    }
    PB_CHK(QPSetBox(child, qpc->is, lbnew, ubnew));
    PB_CHK(VecDestroy(&lbnew));
    PB_CHK(VecDestroy(&ubnew));
    pb::unref(sub);
  }
  // child->x is destroyed (:515); QPSetUpInnerObjects then copies the parent's x as the initial guess
  pb::unref(child->x);
  child->postSolveCtx = xtilde;
  (void)post_default;
  return 0;
}
