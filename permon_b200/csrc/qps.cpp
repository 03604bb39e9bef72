// qps.cpp -- QPS base class, QPSMPGP and QPSSMALXE.
//
// MPGP has two drivers over the same kernels:
//   * fused / device-driven (default; expansion std + fixed length, no fallback): per iteration the host only
//     ENQUEUES  K_A -> ctrl_A -> K_B -> [ctrl_E] -> K_A' -> ctrl_B -> K_C ; step selection, the stopping test
//     (QPSConvergedDefault or the SMALXE inner test) and the counters live in device memory (mpgp_ctl.h).
//     The host looks at the `reason` word once per batch of iterations; kernels enqueued past the stopping
//     iteration see reason != 0 and exit, so iteration counts are exact.
//   * generic / host-driven: one kernel per reference Vec/Mat call, in the reference's order.  Used for the
//     option variants off the headline path (expansion types gf/g/gfgr/ggr/projcg, length types opt/
//     optapprox/bb, fallback) and selectable with -qps_mpgp_b200_driver generic for cross-checks.
//   A user monitor or a user convergence test switches the fused driver to one host sync per iteration.
//
// Reference: src/qps/interface/qps.c, src/qps/impls/mpgp/mpgp.c, src/qps/impls/smalxe/smalxe.c
#include <math.h>
#include <stddef.h>
#include <string.h>

#include <algorithm>
#include <memory>

#include "objects.h"

using namespace pb;

static std::map<std::string, PetscErrorCode (*)(QPS)> g_qps_registry;
static PetscErrorCode                                QPSCreate_MPGP(QPS qps);
static PetscErrorCode                                QPSCreate_SMALXE(QPS qps);
PetscErrorCode                                       QPSCreate_KSP(QPS qps);    // qps_lin.cpp
PetscErrorCode                                       QPSCreate_PCPG(QPS qps);
extern "C" PetscErrorCode                            QPSConverged_Inner_SMALXE(QPS qps_inner, KSPConvergedReason *reason);
int                                                  smalxe_fill_ctl(QPS inner, MpgpCtl *S, bool *host_needed);
int                                                  smalxe_read_ctl(QPS inner, const MpgpCtl *S);

static const char *reason_name(int r)
{
  switch (r) {
  case KSP_CONVERGED_RTOL: return "CONVERGED_RTOL";
  case KSP_CONVERGED_ATOL: return "CONVERGED_ATOL";
  case KSP_CONVERGED_ITS: return "CONVERGED_ITS";
  case KSP_CONVERGED_HAPPY_BREAKDOWN: return "CONVERGED_HAPPY_BREAKDOWN";
  case KSP_DIVERGED_NULL: return "DIVERGED_NULL";
  case KSP_DIVERGED_ITS: return "DIVERGED_ITS";
  case KSP_DIVERGED_DTOL: return "DIVERGED_DTOL";
  case KSP_DIVERGED_BREAKDOWN: return "DIVERGED_BREAKDOWN";
  case KSP_DIVERGED_NANORINF: return "DIVERGED_NANORINF";
  case KSP_DIVERGED_INDEFINITE_MAT: return "DIVERGED_INDEFINITE_MAT";
  case KSP_CONVERGED_ITERATING: return "CONVERGED_ITERATING";
  }
  return "UNKNOWN";
}

// =====================================================================================================
// QPS base
// =====================================================================================================
_p_QPS::~_p_QPS()
{
  if (impl) {
    impl->reset(this);
    delete impl;
  }
  if (convergencetestdestroy && cnvctx) convergencetestdestroy(cnvctx);
  for (auto &m : monitors)
    if (m.destroy) m.destroy(&m.ctx);
  if (topQP) {
    if (topQP->changeListenerCtx == this) {
      topQP->changeListener    = nullptr;
      topQP->changeListenerCtx = nullptr;
    }
    QPDestroy(&topQP);
  }
  QPDestroy(&solQP);
}

PetscErrorCode QPSRegister(const char sname[], PetscErrorCode (*create)(QPS))
{
  g_qps_registry[sname] = create;
  return 0;
}
static void qps_register_all()
{   // QPSRegisterAll qpsregis.c:17-27 (only the types on the path)
  if (!g_qps_registry.empty()) return;
  QPSRegister(QPSMPGP, QPSCreate_MPGP);
  QPSRegister(QPSSMALXE, QPSCreate_SMALXE);
  QPSRegister(QPSKSP, QPSCreate_KSP);
  QPSRegister(QPSPCPG, QPSCreate_PCPG);
}

PetscErrorCode QPSConvergedDefaultCreate(void **ctx)
{
  *ctx = new QPSConvergedDefaultCtx;
  return 0;
}
PetscErrorCode QPSConvergedDefaultDestroy(void *ctx)
{
  delete (QPSConvergedDefaultCtx *)ctx;
  return 0;
}
static PetscErrorCode QPSConvergedDefaultSetUp(QPS qps)
{   // qps.c:718-731
  QPSConvergedDefaultCtx *c = (QPSConvergedDefaultCtx *)qps->cnvctx;
  if (c->setup_called) return 0;
  if (!qps->setupcalled) return err(PETSC_ERR_ARG_WRONGSTATE, "QPSSetUp() not yet called");
  PB_CHK(vec_norm2(qps->solQP->b, &c->norm_rhs));
  c->ttol         = std::max(qps->rtol * c->norm_rhs, qps->atol);
  c->norm_rhs_div = c->norm_rhs;
  c->setup_called = true;
  return 0;
}
PetscErrorCode QPSConvergedDefault(QPS qps, KSPConvergedReason *reason)
{   // qps.c:675-714
  QPSConvergedDefaultCtx *c = (QPSConvergedDefaultCtx *)qps->cnvctx;
  *reason = KSP_CONVERGED_ITERATING;
  if (!c) return err(PETSC_ERR_ARG_NULL, "Convergence context must have been created with QPSConvergedDefaultCreate()");
  if (!c->setup_called) PB_CHK(QPSConvergedDefaultSetUp(qps));
  *reason = (KSPConvergedReason)pb_converged_default(qps->iteration, qps->rnorm, qps->max_it, c->ttol, qps->atol, qps->divtol, c->norm_rhs_div);
  return 0;
}
PetscErrorCode QPSConvergedSkip(QPS qps, KSPConvergedReason *reason)
{   // qps.c:775-783
  *reason = KSP_CONVERGED_ITERATING;
  if (qps->iteration >= qps->max_it) *reason = KSP_CONVERGED_ITS;
  return 0;
}

PetscErrorCode QPSCreate(MPI_Comm comm, QPS *qps_new)
{   // qps.c:61-100
  qps_register_all();
  _p_QPS *qps = new _p_QPS;
  qps->comm   = comm;
  void *ctx;
  QPSConvergedDefaultCreate(&ctx);
  QPSSetConvergenceTest(qps, QPSConvergedDefault, ctx, QPSConvergedDefaultDestroy);
  *qps_new = qps;
  return 0;
}
PetscErrorCode QPSDestroy(QPS *qps)
{
  if (!qps || !*qps) return 0;
  pb::unref(*qps);
  return 0;
}
PetscErrorCode QPSSetConvergenceTest(QPS qps, PetscErrorCode (*converge)(QPS, KSPConvergedReason *), void *cctx, PetscErrorCode (*destroy)(void *))
{   // qps.c:617-628
  if (qps->convergencetestdestroy && qps->cnvctx) qps->convergencetestdestroy(qps->cnvctx);
  qps->convergencetest        = converge;
  qps->convergencetestdestroy = destroy;
  qps->cnvctx                 = cctx;
  return 0;
}
PetscErrorCode QPSGetConvergenceContext(QPS qps, void **ctx)
{
  *ctx = qps->cnvctx;
  return 0;
}
PetscErrorCode QPSSetType(QPS qps, const QPSType type)
{   // qps.c:379-406
  if (qps->impl && qps->type == type) return 0;
  auto it = g_qps_registry.find(type);
  if (it == g_qps_registry.end()) return err(PETSC_ERR_ARG_UNKNOWN_TYPE, "Unable to find requested QPS type %s (the B200 build provides \"mpgp\", \"smalxe\", \"ksp\" and \"pcpg\")", type);
  if (qps->impl) {
    qps->impl->reset(qps);
    delete qps->impl;
    qps->impl = nullptr;
  }
  qps->setupcalled = false;
  qps->type        = type;
  PB_CHK(it->second(qps));
  qps->user_type = true;
  return 0;
}
PetscErrorCode QPSGetType(QPS qps, const QPSType *type)
{
  *(const char **)type = qps->type.c_str();
  return 0;
}
PetscErrorCode QPSSetDefaultType(QPS qps)
{   // qps.c:420-455
  if (!qps->topQP) return err(PETSC_ERR_ORDER, "QPS needs QP to be set in order to find a default type");
  QP qp;
  PB_CHK(QPChainGetLast(qps->topQP, &qp));
  if (qp->BE) PB_CHK(QPSSetType(qps, (char *)QPSSMALXE));
  else if (qp->qpc) PB_CHK(QPSSetType(qps, (char *)QPSMPGP));
  else PB_CHK(QPSSetType(qps, (char *)QPSKSP));
  qps->user_type = false;
  return 0;
}
static PetscErrorCode qps_changed(QP qp)
{
  QPS qps = (QPS)qp->changeListenerCtx;
  if (qps) qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSSetQP(QPS qps, QP qp)
{   // qps.c:171-183
  if (qps->topQP == qp) return 0;
  if (qps->topQP) {
    qps->topQP->changeListener    = nullptr;
    qps->topQP->changeListenerCtx = nullptr;
    QPDestroy(&qps->topQP);
  }
  QPDestroy(&qps->solQP);
  qps->topQP = qp;
  pb::ref(qp);
  qp->changeListener    = qps_changed;
  qp->changeListenerCtx = qps;
  qps->setupcalled      = false;
  return 0;
}
PetscErrorCode QPSGetQP(QPS qps, QP *qp)
{
  if (!qps->topQP) {
    QP q;
    PB_CHK(QPCreate(qps->comm, &q));
    PB_CHK(QPSSetQP(qps, q));
    PB_CHK(QPDestroy(&q));
  }
  *qp = qps->topQP;
  return 0;
}
PetscErrorCode QPSGetSolvedQP(QPS qps, QP *qp)
{
  *qp = qps->solQP;
  return 0;
}
PetscErrorCode QPSSetTolerances(QPS qps, PetscReal rtol, PetscReal atol, PetscReal dtol, PetscInt maxits)
{   // qps.c:793-830
  if (rtol != PETSC_DEFAULT) {
    if (rtol < 0.0 || 1.0 <= rtol) return err(PETSC_ERR_ARG_OUTOFRANGE, "Relative tolerance %g must be non-negative and less than 1.0", rtol);
    qps->rtol = rtol;
  }
  if (atol != PETSC_DEFAULT) {
    if (atol < 0.0) return err(PETSC_ERR_ARG_OUTOFRANGE, "Absolute tolerance %g must be non-negative", atol);
    qps->atol = atol;
  }
  if (dtol != PETSC_DEFAULT) {
    if (dtol <= 0.0) return err(PETSC_ERR_ARG_OUTOFRANGE, "Divergence tolerance %g must be larger than 1.0", dtol);
    qps->divtol = dtol;
  }
  if (maxits != PETSC_DEFAULT) {
    if (maxits < 0) return err(PETSC_ERR_ARG_OUTOFRANGE, "Maximum number of iterations %d must be non-negative", (int)maxits);
    qps->max_it = maxits;
  }
  // as in the reference (qps.c:793-830) the cached ttol / norm_rhs_div of QPSConvergedDefaultCtx are NOT invalidated here: they are
  // computed once, at the first convergence test after QPSConvergedDefaultCreate (qps.c:686,723-728)
  return 0;
}
PetscErrorCode QPSGetTolerances(QPS qps, PetscReal *rtol, PetscReal *atol, PetscReal *dtol, PetscInt *maxits)
{
  if (rtol) *rtol = qps->rtol;
  if (atol) *atol = qps->atol;
  if (dtol) *dtol = qps->divtol;
  if (maxits) *maxits = qps->max_it;
  return 0;
}
PetscErrorCode QPSSetOptionsPrefix(QPS qps, const char prefix[])
{
  qps->prefix = prefix ? prefix : "";
  return 0;
}
PetscErrorCode QPSAppendOptionsPrefix(QPS qps, const char prefix[])
{
  qps->prefix += prefix ? prefix : "";
  return 0;
}
PetscErrorCode QPSGetOptionsPrefix(QPS qps, const char *prefix[])
{
  *prefix = qps->prefix.c_str();
  return 0;
}
PetscErrorCode QPSSetAutoPostSolve(QPS qps, PetscBool flg)
{
  qps->autoPostSolve = flg;
  return 0;
}
PetscErrorCode QPSGetAutoPostSolve(QPS qps, PetscBool *flg)
{
  *flg = qps->autoPostSolve ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode QPSGetConvergedReason(QPS qps, KSPConvergedReason *reason)
{
  *reason = qps->reason;
  return 0;
}
PetscErrorCode QPSGetResidualNorm(QPS qps, PetscReal *rnorm)
{
  *rnorm = qps->rnorm;
  return 0;
}
PetscErrorCode QPSGetIterationNumber(QPS qps, PetscInt *its)
{
  *its = qps->iteration;
  return 0;
}
PetscErrorCode QPSGetAccumulatedIterationNumber(QPS qps, PetscInt *its)
{
  *its = qps->iterations_accumulated;
  return 0;
}
PetscErrorCode QPSMonitorSet(QPS qps, PetscErrorCode (*monitor)(QPS, PetscInt, PetscReal, void *), void *mctx, PetscCtxDestroyFn *destroy)
{
  if (qps->monitors.size() >= 5) return err(PETSC_ERR_ARG_OUTOFRANGE, "Too many QPS monitors set");   // qpsimpl.h:8
  qps->monitors.push_back({monitor, mctx, destroy});
  return 0;
}
PetscErrorCode QPSMonitorCancel(QPS qps)
{
  for (auto &m : qps->monitors)
    if (m.destroy) m.destroy(&m.ctx);
  qps->monitors.clear();
  return 0;
}
PetscErrorCode QPSMonitorDefault(QPS qps, PetscInt n, PetscReal rnorm, void *ctx)
{   // qps.c:1364-1384
  PetscViewer v = (PetscViewer)ctx;
  if (qps->impl && qps->impl->has_monitor()) return qps->impl->monitor(qps, n, v);
  if (n == 0 && !qps->prefix.empty()) vprintf_viewer(v, "  Projected gradient norms for %s solve.\n", qps->prefix.c_str());
  vprintf_viewer(v, "%3d QPS Projected gradient norm %14.12e \n", (int)n, rnorm);
  return 0;
}
static PetscErrorCode qps_monitor(QPS qps, PetscInt it, PetscReal rnorm)
{   // QPSMonitor qps.c:1135-1142
  for (auto &m : qps->monitors) PB_CHK(m.f(qps, it, rnorm, m.ctx));
  return 0;
}

PetscErrorCode QPSSetFromOptions(QPS qps)
{   // qps.c:859-905
  qps_register_all();
  std::string type;
  if (options_string(qps->prefix, "-qps_type", &type)) PB_CHK(QPSSetType(qps, (char *)type.c_str()));
  else if (!qps->impl && qps->topQP) PB_CHK(QPSSetDefaultType(qps));
  PetscInt maxit;
  double   rtol, atol, dtol;
  if (options_int(qps->prefix, "-qps_max_it", &maxit)) PB_CHK(QPSSetTolerances(qps, PETSC_DEFAULT, PETSC_DEFAULT, PETSC_DEFAULT, maxit));
  if (options_real(qps->prefix, "-qps_rtol", &rtol)) PB_CHK(QPSSetTolerances(qps, rtol, PETSC_DEFAULT, PETSC_DEFAULT, PETSC_DEFAULT));
  if (options_real(qps->prefix, "-qps_atol", &atol)) PB_CHK(QPSSetTolerances(qps, PETSC_DEFAULT, atol, PETSC_DEFAULT, PETSC_DEFAULT));
  if (options_real(qps->prefix, "-qps_divtol", &dtol)) PB_CHK(QPSSetTolerances(qps, PETSC_DEFAULT, PETSC_DEFAULT, dtol, PETSC_DEFAULT));
  bool flg;
  if (options_bool(qps->prefix, "-qps_auto_post_solve", &flg)) qps->autoPostSolve = flg;
  if (options_bool(qps->prefix, "-qps_monitor_cancel", &flg) && flg) PB_CHK(QPSMonitorCancel(qps));
  if (options_bool(qps->prefix, "-qps_monitor", &flg) && flg) PB_CHK(QPSMonitorSet(qps, QPSMonitorDefault, NULL, NULL));
  if (options_bool(qps->prefix, "-qps_view_convergence", &flg)) qps->view_convergence = flg;
  if (qps->impl) PB_CHK(qps->impl->setfromoptions(qps));
  return 0;
}

PetscErrorCode QPSIsQPCompatible(QPS qps, QP qp, PetscBool *flg)
{
  *flg = PETSC_FALSE;
  if (!qps->impl) return 0;
  return qps->impl->isqpcompatible(qps, qp, flg);
}

PetscErrorCode QPSSetUp(QPS qps)
{   // qps.c:198-221
  if (qps->setupcalled) return 0;
  if (!qps->topQP) return err(PETSC_ERR_ORDER, "QPSSetQP must be called first");
  PB_CHK(dev_init());   // fail loudly: no CPU execution path
  PhaseTimer pt_all("QPSSetUp");
  {
    PhaseTimer pt("QPSSetUp: QPChainSetUp");
    PB_CHK(QPChainSetUp(qps->topQP));
  }
  if (!qps->solQP) {
    PB_CHK(QPChainGetLast(qps->topQP, &qps->solQP));
    pb::ref(qps->solQP);
  }
  if (!qps->impl) PB_CHK(QPSSetDefaultType(qps));
  PetscBool flg;
  PB_CHK(QPSIsQPCompatible(qps, qps->solQP, &flg));
  if (!flg) return err(PETSC_ERR_ARG_INCOMP, "QPS solver %s is not compatible with its attached QP", qps->type.c_str());
  {
    PhaseTimer pt("QPSSetUp: solver set-up (work vectors, maxeig)");
    PB_CHK(qps->impl->setup(qps));
  }
  PB_CHK(QPChainSetUp(qps->solQP));
  qps->setupcalled = true;
  return 0;
}
PetscErrorCode QPSResetStatistics(QPS qps)
{   // qps.c:265-275
  qps->iteration              = 0;
  qps->iterations_accumulated = 0;
  qps->nsolves                = 0;
  if (qps->impl) PB_CHK(qps->impl->resetstatistics(qps));
  return 0;
}
PetscErrorCode QPSReset(QPS qps)
{   // qps.c:236-249
  if (qps->impl) PB_CHK(qps->impl->reset(qps));
  if (qps->topQP) {
    qps->topQP->changeListener    = nullptr;
    qps->topQP->changeListenerCtx = nullptr;
    PB_CHK(QPDestroy(&qps->topQP));
  }
  PB_CHK(QPDestroy(&qps->solQP));
  qps->setupcalled = false;
  return QPSResetStatistics(qps);
}
PetscErrorCode QPSSolve(QPS qps)
{   // qps.c:537-555
  PB_CHK(QPSSetUp(qps));
  {
    PhaseTimer pt("QPSSolve: solve");
    PB_CHK(qps->impl->solve(qps));
  }
  qps->iterations_accumulated += qps->iteration;
  qps->nsolves++;
  qps->postsolvecalled = false;
  qps->solQP->solved   = (qps->reason > 0);
  if (qps->autoPostSolve) PB_CHK(QPSPostSolve(qps));
  return 0;
}
PetscErrorCode QPSViewConvergence(QPS qps, PetscViewer v)
{   // qps.c:968-1000
  _p_PetscViewer tmp;
  if (!v) v = &tmp;
  const int r = qps->reason;
  vprintf_viewer(v, "QPS Object: %s%d MPI process%s\n", qps->prefix.empty() ? "" : ("(" + qps->prefix + ") ").c_str(), qps->comm->size, qps->comm->size > 1 ? "es" : "");
  vprintf_viewer(v, "  type: %s\n", qps->type.c_str());
  v->tab++;
  vprintf_viewer(v, "last QPSSolve %s due to %s, KSPReason=%d, required %d iterations\n", (r > 0) ? "CONVERGED" : "DIVERGED", reason_name(r), r, (int)qps->iteration);
  vprintf_viewer(v, "all %d QPSSolves from last QPSReset/QPSResetStatistics have required %d iterations\n", (int)qps->nsolves, (int)qps->iterations_accumulated);
  vprintf_viewer(v, "tolerances: rtol=%.1e, abstol=%.1e, dtol=%.1e, maxits=%d\n", qps->rtol, qps->atol, qps->divtol, (int)qps->max_it);
  if (qps->impl) {
    vprintf_viewer(v, "%s specific:\n", qps->type.c_str());
    v->tab++;
    PB_CHK(qps->impl->viewconvergence(qps, v));
    v->tab--;
  }
  v->tab--;
  return 0;
}
PetscErrorCode QPSPostSolve(QPS qps)
{   // qps.c:579-613
  if (qps->postsolvecalled) return 0;
  bool flg = qps->view_convergence;
  if (options_get(qps->prefix, "-qps_view_convergence", nullptr)) {
    bool b = true;
    options_bool(qps->prefix, "-qps_view_convergence", &b);
    flg = b;
  }
  if (flg) PB_CHK(QPSViewConvergence(qps, nullptr));
  QP qp;
  PB_CHK(QPSGetQP(qps, &qp));
  PB_CHK(QPChainPostSolve(qp));
  qps->postsolvecalled = true;
  return 0;
}

// =====================================================================================================
// MPGP
// =====================================================================================================
struct SmalxeImpl;
struct SmalxeInnerCtx {   // QPSConvergedCtx_Inner_SMALXE smalxeimpl.h:5-11
  double      gtol = NAN, norm_rhs_outer = NAN, ttol_outer = NAN, MNormBu = NAN;
  QPS         qps_outer = nullptr;
  SmalxeImpl *smalxe = nullptr;
};

struct MpgpImpl : QPSImpl {   // QPS_MPGP mpgpimpl.h:5-38
  double           alpha = 0, alpha_user = PETSC_DECIDE, gamma = 1.0, maxeig = PETSC_DECIDE, maxeig_tol = PETSC_DECIDE;
  QPSScalarArgType alpha_type = QPS_ARG_MULTIPLE;
  PetscInt         maxeig_iter = PETSC_DECIDE;
  double           btol = 10 * PETSC_MACHINE_EPSILON, bchop_tol = 0.0;
  int              exptype = QPS_MPGP_EXPANSION_STD, explengthtype = QPS_MPGP_EXPANSION_LENGTH_FIXED;
  bool             expproject = true, resetalpha = false, fallback = false, fallback2 = false;
  PetscInt         nmv = 0, ncg = 0, nexp = 0, nprop = 0, nfinc = 0, nfall = 0;
  char             currentStepType = ' ';
  double           gfnorm = 0, gcnorm = 0;
  std::string      driver = "auto";
  int              batch = 16;
  // work vectors (mpgp.c:6-17): gP gf gc g p Ap gr [7 8 9]
  std::vector<Vec> work;
  Vec              expdirection = nullptr, explengthvec = nullptr, explengthvecold = nullptr, xold = nullptr;
  // device-driven engine
  MpgpCtl *dS = nullptr, *hS = nullptr;
  Reducer  RA, RB, RC;   // records after K_A, after K_B / K_A', and K_C's local g.p
  bool     engine_ready = false;

  ~MpgpImpl() override { free_all(); }
  void free_all()
  {
    for (auto &w : work) pb::unref(w);
    work.clear();
    if (engine_ready) {
      dfree(dS);
      pinned_put(hS, sizeof(MpgpCtl));
      RA.destroy();
      RB.destroy();
      RC.destroy();
      engine_ready = false;
    }
  }
  int set_work(QPS qps, int nw)
  {
    for (auto &w : work) pb::unref(w);
    work.assign(nw, nullptr);
    for (int i = 0; i < nw; i++) PB_CHK(VecDuplicate(qps->solQP->x, &work[i]));
    return 0;
  }
  PetscErrorCode setup(QPS qps) override;
  PetscErrorCode solve(QPS qps) override;
  PetscErrorCode reset(QPS) override
  {
    free_all();
    return 0;
  }
  PetscErrorCode resetstatistics(QPS) override
  {   // mpgp.c:654-664
    ncg = nexp = nmv = nprop = 0;
    return 0;
  }
  PetscErrorCode setfromoptions(QPS qps) override;
  PetscErrorCode isqpcompatible(QPS, QP qp, PetscBool *flg) override
  {   // mpgp.c:695-711
    *flg = (!qp->BE && !qp->cE && qp->qpc && qp->qpc->type == QPCBOX) ? PETSC_TRUE : PETSC_FALSE;
    return 0;
  }
  PetscErrorCode viewconvergence(QPS, PetscViewer v) override
  {   // mpgp.c:751-770
    vprintf_viewer(v, "from the last QPSReset:\n");
    vprintf_viewer(v, "number of Hessian multiplications %d\n", (int)nmv);
    vprintf_viewer(v, "number of CG steps %d\n", (int)ncg);
    vprintf_viewer(v, "number of expansion steps %d\n", (int)nexp);
    vprintf_viewer(v, "number of proportioning steps %d\n", (int)nprop);
    if (fallback || fallback2) {
      vprintf_viewer(v, "number of cost function value increases: %d\n", (int)nfinc);
      vprintf_viewer(v, "number of fallbacks: %d\n", (int)nfall);
    }
    return 0;
  }
  bool           has_monitor() override { return true; }
  PetscErrorCode monitor(QPS qps, PetscInt n, PetscViewer v) override
  {   // QPSMonitorDefault_MPGP mpgp.c:21-34
    if (n == 0 && !qps->prefix.empty()) vprintf_viewer(v, "  Projected gradient norms for %s solve.\n", qps->prefix.c_str());
    vprintf_viewer(v, "%3d MPGP [%c] ||gp||=%.10e,\t||gf||=%.10e,\t||gc||=%.10e,\talpha=%.10e\n", (int)n, currentStepType, qps->rnorm, gfnorm, gcnorm, alpha);
    return 0;
  }
  bool fused_eligible(QPS qps) const
  {
    if (driver == "generic") return false;
    if (exptype != QPS_MPGP_EXPANSION_STD || explengthtype != QPS_MPGP_EXPANSION_LENGTH_FIXED) return false;
    if (fallback || fallback2) return false;
    Mat A = qps->solQP->A;
    if (A->kind == MK_PENALIZED) {
      if (A->pf && A->pf->G && A->pf->G->M > PB_MAXEQ) return false;   // the rank-m fusion keeps PB_MAXEQ accumulators; more rows: un-fused route
      if (A->pf && A->pf->implicit_orth) return false;                 // penalised term Q = B'(BB')^-1 B: the coarse solve sits between the two rank-m halves
      A = A->A;
    }
    auto one_gpu = [](Mat F) { return F->kind == MK_AIJ || F->kind == MK_DENSE; };   // dense matrices live on one rank only
    if (A->kind == MK_PROD) return one_gpu(A->M1) && one_gpu(A->M2) && A->comm->size == 1;
    return A->kind == MK_AIJ || A->kind == MK_DENSE;
  }
  int engine_init(QPS qps);
  int solve_fused(QPS qps);
  int solve_generic(QPS qps);
  int grads(QPS qps, Vec x, Vec g);
  int expansion_length(QPS qps);
  int expansion_std(QPS qps, double afeas, double acg);
};

static MpgpImpl *mpgp_of(QPS qps) { return (qps->impl && qps->type == QPSMPGP) ? static_cast<MpgpImpl *>(qps->impl) : nullptr; }

static const char *const kExpTypes[] = {"std", "projcg", "gf", "g", "gfgr", "ggr"};
static const char *const kLenTypes[] = {"fixed", "opt", "optapprox", "bb"};

PetscErrorCode MpgpImpl::setfromoptions(QPS qps)
{   // mpgp.c:715-747
  const std::string &p = qps->prefix;
  bool               alpha_direct = false, flg1, flg2;
  double             a = alpha_user, v;
  PetscInt           iv;
  flg1 = options_bool(p, "-qps_mpgp_alpha_direct", &alpha_direct);
  flg2 = options_real(p, "-qps_mpgp_alpha", &a);
  if (flg1 || flg2) PB_CHK(QPSMPGPSetAlpha(qps, a, alpha_direct ? QPS_ARG_DIRECT : QPS_ARG_MULTIPLE));
  if (options_real(p, "-qps_mpgp_gamma", &v)) gamma = v;
  if (options_real(p, "-qps_mpgp_maxeig", &v)) PB_CHK(QPSMPGPSetOperatorMaxEigenvalue(qps, v));
  if (options_real(p, "-qps_mpgp_maxeig_tol", &v)) maxeig_tol = v;
  if (options_int(p, "-qps_mpgp_maxeig_iter", &iv)) maxeig_iter = iv;
  options_real(p, "-qps_mpgp_btol", &btol);
  options_real(p, "-qps_mpgp_bound_chop_tol", &bchop_tol);
  std::string s;
  if (options_string(p, "-qps_mpgp_expansion_type", &s)) {
    int k;
    for (k = 0; k < 6 && s != kExpTypes[k]; k++) {}
    if (k == 6) return err(PETSC_ERR_ARG_UNKNOWN_TYPE, "Unknown MPGP expansion type %s", s.c_str());
    exptype = k;
  }
  if (options_string(p, "-qps_mpgp_expansion_length_type", &s)) {
    int k;
    for (k = 0; k < 4 && s != kLenTypes[k]; k++) {}
    if (k == 4) return err(PETSC_ERR_ARG_UNKNOWN_TYPE, "Unknown MPGP expansion length type %s", s.c_str());
    explengthtype = k;
  }
  options_bool(p, "-qps_mpgp_alpha_reset", &resetalpha);
  options_bool(p, "-qps_mpgp_fallback", &fallback);
  options_bool(p, "-qps_mpgp_fallback2", &fallback2);
  if (fallback2) fallback = false;
  options_string(p, "-qps_mpgp_b200_driver", &driver);   // auto | fused | generic
  if (options_int(p, "-qps_mpgp_b200_batch", &iv)) batch = std::max<PetscInt>(1, iv);
  qps->setupcalled = false;
  return 0;
}

PetscErrorCode MpgpImpl::setup(QPS qps)
{   // QPSSetup_MPGP mpgp.c:359-428
  int nw = 7;
  if (fallback || fallback2) nw = (explengthtype != QPS_MPGP_EXPANSION_LENGTH_BB) ? 9 : 10;
  else if (explengthtype == QPS_MPGP_EXPANSION_LENGTH_BB) nw = 9;
  const bool fused = fused_eligible(qps);
  if (driver == "fused" && !fused) return err(PETSC_ERR_SUP, "-qps_mpgp_b200_driver fused needs expansion std/fixed, no fallback and an AIJ or dense Hessian (or a product of such)");
  {
    PhaseTimer pt("MPGP set-up: work vectors");
    PB_CHK(set_work(qps, nw));
  }
  if (bchop_tol) {   // mpgp.c:379-382: VecFilter(lb / ub, bchop_tol) -- bounds closer to 0 than the tolerance become 0 (in the user's Vecs)
    QPC qpc = qps->solQP->qpc;
    for (Vec bnd : {qpc ? qpc->lb : (Vec) nullptr, qpc ? qpc->ub : (Vec) nullptr}) {
      if (!bnd) continue;
      double *d;
      PB_CHK(vec_dev_rw(bnd, &d));
      PB_CHK(k_filter(bnd->n, d, bchop_tol));
    }
    if (qpc) qpc->setupcalled = false;   // expanded (IS) copies of the bounds are rebuilt from the filtered vectors
  }
  expproject = true;   // QPSCreate_MPGP :839 (re-evaluated at every set-up here)
  switch (exptype) {
  case QPS_MPGP_EXPANSION_STD:
    expdirection = work[6];
    explengthvec = work[6];
    if (explengthtype == QPS_MPGP_EXPANSION_LENGTH_FIXED) expproject = false;   // :388
    break;
  case QPS_MPGP_EXPANSION_GF: expdirection = work[1]; explengthvec = work[1]; break;
  case QPS_MPGP_EXPANSION_G: expdirection = work[3]; explengthvec = work[3]; break;
  case QPS_MPGP_EXPANSION_GFGR: expdirection = work[1]; explengthvec = work[6]; break;
  case QPS_MPGP_EXPANSION_GGR: expdirection = work[3]; explengthvec = work[6]; break;
  case QPS_MPGP_EXPANSION_PROJCG: expdirection = work[1]; explengthvec = work[1]; break;
  default: return err(PETSC_ERR_PLIB, "Unknown MPGP expansion type");
  }
  {   // the uploads of b, x and the bounds travel on the copy stream while the power method below runs
    QP qp = qps->solQP;
    PB_CHK(vec_prefetch(qp->b));
    PB_CHK(vec_prefetch(qp->x));
    if (qp->qpc && !qp->qpc->is) {
      PB_CHK(vec_prefetch(qp->qpc->lb));
      PB_CHK(vec_prefetch(qp->qpc->ub));
    }
  }
  if (alpha_type == QPS_ARG_MULTIPLE) {   // :417-425
    if (maxeig == PETSC_DECIDE) {
      PhaseTimer pt("MPGP set-up: MatGetMaxEigenvalue");
      PB_CHK(MatGetMaxEigenvalue(qps->solQP->A, NULL, &maxeig, maxeig_tol, maxeig_iter));
    }
    if (alpha_user == PETSC_DECIDE) alpha_user = 2.0;
    alpha = alpha_user / maxeig;
  } else {
    alpha = alpha_user;
  }
  return 0;
}

int MpgpImpl::engine_init(QPS qps)
{
  if (engine_ready) return 0;
  PB_CHK(dev_init());
  PB_CHK(dmalloc(&dS, 2));
  hS = (MpgpCtl *)pinned_get(sizeof(MpgpCtl));
  if (!hS) return err(PETSC_ERR_MEM, "out of pinned host memory");
  PB_CHK(RA.init(qps->comm));
  PB_CHK(RB.init(qps->comm));
  PB_CHK(RC.init(qps->comm));
  engine_ready = true;
  return 0;
}

// ---- the fused, device-driven driver --------------------------------------------------------------------
int MpgpImpl::solve_fused(QPS qps)
{
  QP  qp = qps->solQP;
  Mat A = qp->A, base = A;
  std::unique_ptr<PhaseTimer> pt_pre(new PhaseTimer("MPGP fused: engine init + vector uploads"));
  PB_CHK(engine_init(qps));
  PB_CHK(mat_ensure_device(A));
  cudaStream_t s = ctx().stream;

  MpgpVecs v;
  MpgpCtl  S;
  memset(&S, 0, sizeof S);
  if (A->kind == MK_PENALIZED) {
    base = A->A;
    PB_CHK(qppf_dense_rows(A->pf, &v.B, &v.m));
    S.rho = A->rho;
  }
  const bool prod = base->kind == MK_PROD;
  Mat        M1 = prod ? base->M1 : base, M2 = prod ? base->M2 : nullptr;
  const bool multi = (qps->comm->size > 1);
  HaloPlan  *H = multi ? M1->halo : nullptr;
  v.n = qp->x->n;
  PB_CHK(vec_dev_rw(qp->x, &v.x));
  PB_CHK(vec_dev_read(qp->b, &v.b));
  PB_CHK(vec_dev_write(work[3], &v.g));
  PB_CHK(vec_dev_write(work[4], &v.p));
  PB_CHK(vec_dev_write(work[5], &v.Ap));
  PB_CHK(vec_dev_write(work[1], &v.gf));
  PB_CHK(qpc_box_for_vec(qp->qpc, qp->x, &v.bx));
  if (prod) PB_CHK(vec_dev_write(base->twork, &v.t));

  // ---- control block
  const bool inner_smalxe = (qps->convergencetest == QPSConverged_Inner_SMALXE);
  const bool default_test = (qps->convergencetest == QPSConvergedDefault);
  S.max_it = qps->max_it;
  S.nranks = qps->comm->size;
  S.m      = v.m;
  S.gamma2 = gamma * gamma;   // mpgp.c:489
  S.alpha  = alpha;
  S.rtol = qps->rtol; S.atol = qps->atol; S.divtol = qps->divtol;
  bool host_conv = !qps->monitors.empty() || !(inner_smalxe || default_test);
  if (inner_smalxe) {
    bool need_host = false;
    PB_CHK(smalxe_fill_ctl(qps, &S, &need_host));
    if (need_host) host_conv = true;
    S.inner_mode = 1;
  } else if (default_test) {
    QPSConvergedDefaultCtx *c = (QPSConvergedDefaultCtx *)qps->cnvctx;
    if (!c->setup_called) PB_CHK(QPSConvergedDefaultSetUp(qps));
    S.ttol = c->ttol;
    S.norm_rhs_div = c->norm_rhs_div;
  }
  S.host_conv = host_conv ? 1 : 0;
  S.iteration = 0; S.reason = 0; S.step = ' '; S.do_prop = 0; S.pmode = 0; S.init = 1;
  {
    const char *e = getenv("PERMON_B200_SERPENTINE");
    S.serp = (e && !strcmp(e, "0")) ? 0 : 1;
  }
  *hS = S;
  PB_CUDA(cudaMemcpyAsync(dS, hS, sizeof(MpgpCtl), cudaMemcpyHostToDevice, s));

  // Two copies of the control block: S0 = state at the top of the iteration (after ctrl_B), S1 = state after
  // ctrl_A.  In the device-driven mode ctrl_A / ctrl_B run in the prologues of K_B / K_C (every CTA recomputes the
  // scalar step from the records into shared memory, CTA 0 stores the other copy).  With host callbacks
  // (fold == false) the stand-alone ctrl kernels update S0 in place and S1 aliases S0.
  const bool fold = !host_conv && !getenv("PERMON_B200_NOFOLD");
  MpgpCtl   *S0 = dS, *S1 = fold ? dS + 1 : dS;
  if (fold) PB_CUDA(cudaMemcpyAsync(dS + 1, hS, sizeof(MpgpCtl), cudaMemcpyHostToDevice, s));

  // multi-GPU plumbing: peer-memory pushes (CUDA IPC over NVLink) when available, NCCL otherwise
  MPI_Comm   comm = qps->comm;
  const bool p2p = multi && comm->p2p && H && H->p2p;
  const bool fused_push = p2p && H->contig && !getenv("PERMON_B200_NOFUSEDPUSH");
  auto red = [&](Reducer &R, int kind, bool publish) -> RedBuf {
    RedBuf rb = R.rb;
    if (kind == 0) {   // K_A: slot RA_GP of its record is the local g.p that K_C summed while it wrote p
      rb.add_part = RC.rb.partials;
      rb.add_n    = fused_C_grid(v.n);
      rb.add_slot = RA_GP;
    }
    if (p2p && publish) {
      rb.win  = comm->d_win;
      rb.kind = kind;
      rb.seq  = ++comm->seq[kind];
    }
    return rb;
  };
  auto rec_ptr = [&](Reducer &R, int kind) -> const double * {   // rank-0 record of the current sequence number
    return p2p ? comm->my_slot + p2p_slot_index(kind, comm->seq[kind], 0) : R.d_all;
  };
  auto flag_ptr = [&](int kind) -> const unsigned long long * { return p2p ? comm->my_flag + p2p_flag_index(kind, 0) : nullptr; };
  auto gather_ctrl_E = [&]() -> int {   // B u of the new iterate for the second SpMV (SMALXE only)
    if (p2p) return k_ctrl_E_p2p(S1, comm->d_win, comm->my_slot, comm->my_flag, comm->seq[1]);
    PB_CHK(RB.gather());
    return k_ctrl_E(S1, RB.d_all);
  };
  auto ghost_merge = [&](int which) -> GhostMerge {   // which: 0 = ghosts of p (K_A), 1 = ghosts of x (K_A')
    GhostMerge gm;
    if (!H) return gm;
    gm.row_map = H->d_row_map;
    gm.lo      = H->skip_lo;
    gm.hi      = H->skip_hi;
    gm.oia     = M1->Ao.ia;
    gm.oja     = M1->Ao.ja;
    gm.oa      = M1->Ao.a;
    if (p2p) {
      gm.ghost  = H->d_ghost2[which];
      gm.flags  = H->my_hflags[which];
      gm.nflags = (int)H->neigh.size();
      gm.seq    = H->hseq[which];
    } else {
      gm.ghost = H->d_ghost;   // ncclRecv target; the stream already waits for the transfer (mat_halo_end)
    }
    return gm;
  };
  auto second_spmv = [&](bool x_already_pushed) -> int {   // K_A' with its halo / product plumbing
    const double *xin = v.x;
    if (prod) {
      PB_CHK(k_spmv_gated(M2->Ad, v.x, v.t, S1, 1));
      xin = v.t;
    }
    if (H) {
      if (p2p) {
        if (!x_already_pushed) PB_CHK(k_halo_push(H->push[1], v.x, 1, ++H->hseq[1], S1));
      } else {
        PB_CHK(mat_halo_begin(M1, v.x));
      }
    }
    if (H && !p2p) PB_CHK(mat_halo_end(M1));
    PB_CHK(k_fused_A2(M1->Ad, xin, v, S1, red(RB, 2, true), ghost_merge(1)));
    return 0;
  };
  auto step_B = [&]() -> int {   // [all-gather] -> ctrl_A -> K_B (+ x halo push in expansion steps)
    if (!p2p) PB_CHK(RA.gather());
    CtrlFold cf;
    cf.fold = fold ? 1 : 0;
    cf.Sin  = S0;
    cf.Sout = S1;
    cf.size = comm->size;
    if (fold) {
      cf.rec0   = rec_ptr(RA, 0);
      cf.flags0 = flag_ptr(0);
      cf.seq0   = comm->seq[0];
    } else {
      if (p2p) PB_CHK(k_ctrl_A_p2p(S0, comm->d_win, comm->my_slot, comm->my_flag, comm->seq[0]));
      else PB_CHK(k_ctrl_A(S0, RA.d_all));
    }
    if (fused_push) return k_fused_B(v, cf, red(RB, 1, true), H->d_ranges + 1, ++H->hseq[1]);
    return k_fused_B(v, cf, red(RB, 1, true), nullptr, 0);
  };
  auto step_C = [&](bool ctrl_done) -> int {   // [all-gather] -> ctrl_B -> K_C (+ p halo push)
    CtrlFold cf;
    cf.fold = (fold && !ctrl_done) ? 1 : 0;
    cf.Sin  = fold ? S1 : S0;
    cf.Sout = S0;
    cf.size = comm->size;
    if (cf.fold) {
      cf.rec0   = rec_ptr(RB, 1);
      cf.rec1   = rec_ptr(RB, 2);
      cf.flags0 = flag_ptr(1);
      cf.flags1 = flag_ptr(2);
      cf.seq0   = comm->seq[1];
      cf.seq1   = comm->seq[2];
    }
    if (fused_push) return k_fused_C(v, cf, RC.rb, H->d_ranges, ++H->hseq[0]);
    return k_fused_C(v, cf, RC.rb, nullptr, 0);
  };
  auto ctrl_B_standalone = [&]() -> int {
    if (p2p) return k_ctrl_B_p2p(S0, comm->d_win, comm->my_slot, comm->my_flag, comm->seq[1], comm->seq[2]);
    return k_ctrl_B(S0, RB.d_all);
  };
  auto host_step = [&](bool *stop) -> int {   // per-iteration host involvement (monitors / user test)
    PB_CUDA(cudaMemcpyAsync(hS, S0, sizeof(MpgpCtl), cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaStreamSynchronize(s));
    qps->iteration  = hS->iteration;
    qps->rnorm      = hS->rnorm;
    gfnorm          = sqrt(hS->gf2);
    gcnorm          = sqrt(hS->gc2);
    currentStepType = (char)hS->step;
    if (inner_smalxe) PB_CHK(smalxe_read_ctl(qps, hS));
    PB_CHK(qps_monitor(qps, qps->iteration, qps->rnorm));   // mpgp.c:524-528
    PB_CHK(qps->convergencetest(qps, &qps->reason));        // mpgp.c:531
    *stop = (qps->reason != KSP_CONVERGED_ITERATING);
    if (*stop) {
      hS->reason = qps->reason;
      PB_CUDA(cudaMemcpyAsync((char *)S0 + offsetof(MpgpCtl, reason), &hS->reason, sizeof(int), cudaMemcpyHostToDevice, s));
    }
    return 0;
  };

  pt_pre.reset();
  PhaseTimer pt_loop("MPGP fused: initial phase + iterations");
  // ---- initial phase: x = P(x); g = A x - b; split; p = gf  (mpgp.c:497-507)
  PB_CHK(k_fused_project(v, S1, red(RB, 1, true)));
  if (v.m > 0) PB_CHK(gather_ctrl_E());
  PB_CHK(second_spmv(false));
  if (!p2p) PB_CHK(RB.gather());
  bool stop = false;
  if (!fold) {
    PB_CHK(ctrl_B_standalone());
    if (host_conv) PB_CHK(host_step(&stop));
  }
  if (!stop) PB_CHK(step_C(!fold));

  // ---- main loop
  // iterations still allowed by max_it (qps.c:684: DIVERGED_ITS once i > max_it; the SMALXE inner rule counts the accumulated
  // inner iterations, smalxe.c:633): the last batch is cut to that, so that no launch is enqueued behind the stopping iteration
  long long allowed = (long long)S.max_it + 1 - (inner_smalxe ? (long long)S.inner_iter_accu : 0);
  if (allowed < 1) allowed = 1;
  long long enq = 0;
  while (!stop) {
    int nb = host_conv ? 1 : batch;
    if (!host_conv && allowed - enq >= 1 && allowed - enq < nb) nb = (int)(allowed - enq);
    enq += nb;
    for (int it = 0; it < nb && !stop; it++) {
      const double *xin = v.p;
      if (prod) {
        PB_CHK(k_spmv_gated(M2->Ad, v.p, v.t, S0, 0));
        xin = v.t;
      }
      if (H) {
        if (p2p) {
          if (!fused_push) PB_CHK(k_halo_push(H->push[0], v.p, 0, ++H->hseq[0], S0));
        } else {
          PB_CHK(mat_halo_begin(M1, v.p));
        }
      }
      if (H && !p2p) PB_CHK(mat_halo_end(M1));
      PB_CHK(k_fused_A(M1->Ad, xin, v, S0, red(RA, 0, true), ghost_merge(0)));
      PB_CHK(step_B());
      if (v.m > 0) PB_CHK(gather_ctrl_E());
      PB_CHK(second_spmv(fused_push));
      if (!p2p) PB_CHK(RB.gather());
      if (!fold) {
        PB_CHK(ctrl_B_standalone());
        if (host_conv) {
          PB_CHK(host_step(&stop));
          if (stop) break;
        }
      }
      PB_CHK(step_C(!fold));
    }
    if (!host_conv) {
      PB_CUDA(cudaMemcpyAsync(hS, S0, sizeof(MpgpCtl), cudaMemcpyDeviceToHost, s));
      PB_CUDA(cudaStreamSynchronize(s));
      stop = (hS->reason != 0);
    }
  }
  if (host_conv) {
    PB_CUDA(cudaMemcpyAsync(hS, S0, sizeof(MpgpCtl), cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaStreamSynchronize(s));
    hS->reason = qps->reason;
  }
  qps->iteration  = hS->iteration;
  qps->reason     = (KSPConvergedReason)hS->reason;
  qps->rnorm      = hS->rnorm;
  gfnorm          = sqrt(hS->gf2);
  gcnorm          = sqrt(hS->gc2);
  currentStepType = (char)hS->step;
  if (inner_smalxe) PB_CHK(smalxe_read_ctl(qps, hS));
  ncg += hS->ncg; nexp += hS->nexp; nmv += hS->nmv; nprop += hS->nprop;   // mpgp.c:643-648
  return 0;
}

// ---- the generic, host-driven driver (reference operation order, one kernel per Vec/Mat call) ------------
int MpgpImpl::grads(QPS qps, Vec x, Vec g)
{   // MPGPGrads mpgp.c:198-223
  QPC qpc = qps->solQP->qpc;
  PB_CHK(QPCGrads(qpc, x, g, work[1], work[2]));
  PB_CHK(QPCGradReduced(qpc, x, work[1], alpha, work[6]));
  return VecWAXPY(work[0], 1.0, work[1], work[2]);
}
int MpgpImpl::expansion_length(QPS qps)
{   // MPGPExpansionLength mpgp.c:233-287
  QP     qp = qps->solQP;
  double d0, d1;
  switch (explengthtype) {
  case QPS_MPGP_EXPANSION_LENGTH_FIXED: break;
  case QPS_MPGP_EXPANSION_LENGTH_OPT:
    PB_CHK(mat_mult(qp->A, explengthvec, work[5]));
    nmv++;
    PB_CHK(vec_mdot2(explengthvec, work[3], work[5], &d0, &d1));
    if (d1 == .0 && resetalpha) alpha = alpha / maxeig;
    else alpha = alpha_user * (d0 / d1);
    break;
  case QPS_MPGP_EXPANSION_LENGTH_OPTAPPROX:
    if (work[3] != explengthvec) {
      PB_CHK(vec_mdot2(explengthvec, work[3], explengthvec, &d0, &d1));
      alpha = alpha_user * (d0 / d1);
    } else {
      alpha = alpha_user;
    }
    alpha = alpha / maxeig;
    break;
  case QPS_MPGP_EXPANSION_LENGTH_BB:
    PB_CHK(VecAYPX(explengthvecold, -1.0, explengthvec));
    PB_CHK(VecAYPX(xold, -1.0, qp->x));
    PB_CHK(vec_mdot2(explengthvecold, explengthvecold, xold, &d0, &d1));
    if (d1 == .0 && resetalpha) alpha = alpha / maxeig;
    else alpha = alpha_user * (d0 / d1);
    break;
  default: return err(PETSC_ERR_PLIB, "Unknown MPGP expansion length type");
  }
  return 0;
}
int MpgpImpl::expansion_std(QPS qps, double afeas, double)
{   // MPGPExpansion_Std mpgp.c:299-323
  Vec x = qps->solQP->x, g = work[3], p = work[4], Ap = work[5];
  PB_CHK(VecAXPY(x, -afeas, p));
  PB_CHK(VecAXPY(g, -afeas, Ap));
  PB_CHK(grads(qps, x, g));
  PB_CHK(expansion_length(qps));
  return VecAXPY(x, -alpha, expdirection);
}

int MpgpImpl::solve_generic(QPS qps)
{   // QPSSolve_MPGP mpgp.c:438-650
  QP     qp = qps->solQP;
  QPC    qpc = qp->qpc;
  Mat    A = qp->A;
  Vec    b = qp->b, x = qp->x;
  Vec    gP = work[0], gf = work[1], gc = work[2], g = work[3], p = work[4], Ap = work[5], gold = nullptr;
  double gamma2, acg, bcg, afeas, pAp, gcTgc, gfTgf, f, fold;
  PetscInt lnmv = 0, lncg = 0, lnprop = 0, lnexp = 0, lnfinc = 0, lnfall = 0;

  if (explengthtype == QPS_MPGP_EXPANSION_LENGTH_BB) {
    explengthvecold = work[7];
    xold            = work[8];
    if (fallback || fallback2) gold = work[9];
  } else if (fallback || fallback2) {
    xold = work[7];
    gold = work[8];
  }
  gamma2 = gamma * gamma;
  PB_CHK(QPCProject(qpc, x, x));
  PB_CHK(mat_mult(A, x, g));
  lnmv++;
  PB_CHK(VecAXPY(g, -1.0, b));
  PB_CHK(grads(qps, x, g));
  PB_CHK(VecCopy(gf, p));
  currentStepType = ' ';
  qps->iteration  = 0;
  while (1) {
    PB_CHK(vec_norm2(gP, &qps->rnorm));
    PB_CHK(vec_dot(gc, gc, &gcTgc));
    PB_CHK(vec_dot(gf, gf, &gfTgf));
    if (!qps->monitors.empty()) {
      gfnorm = sqrt(gfTgf);
      gcnorm = sqrt(gcTgc);
      PB_CHK(qps_monitor(qps, qps->iteration, qps->rnorm));
    }
    PB_CHK(qps->convergencetest(qps, &qps->reason));
    if (qps->reason != KSP_CONVERGED_ITERATING) break;
    if (gcTgc <= gamma2 * gfTgf) {
      PB_CHK(mat_mult(A, p, Ap));
      lnmv++;
      PB_CHK(vec_dot(p, Ap, &pAp));
      PB_CHK(vec_dot(g, p, &acg));
      acg = acg / pAp;
      PB_CHK(QPCFeas(qpc, x, p, &afeas));
      if (acg <= afeas) {
        lncg++;
        currentStepType = 'c';
        PB_CHK(VecAXPY(x, -acg, p));
        PB_CHK(VecAXPY(g, -acg, Ap));
        PB_CHK(grads(qps, x, g));
        PB_CHK(vec_dot(Ap, gf, &bcg));
        bcg = bcg / pAp;
        PB_CHK(VecAYPX(p, -bcg, gf));
      } else {
        lnexp++;
        currentStepType = 'e';
        if (explengthtype == QPS_MPGP_EXPANSION_LENGTH_BB || fallback || fallback2) {
          PB_CHK(VecCopy(x, xold));
          if (explengthtype == QPS_MPGP_EXPANSION_LENGTH_BB) PB_CHK(VecCopy(explengthvec, explengthvecold));
        }
        if (exptype == QPS_MPGP_EXPANSION_PROJCG) PB_CHK(VecAXPY(x, -acg, p));   // MPGPExpansion_ProjCG :335-349
        else PB_CHK(expansion_std(qps, afeas, acg));
        if (expproject) PB_CHK(QPCProject(qpc, x, x));
        if (fallback || fallback2) PB_CHK(VecCopy(g, gold));
        PB_CHK(mat_mult(A, x, g));
        lnmv++;
        PB_CHK(VecAXPY(g, -1.0, b));
        if (fallback || fallback2) {
          PB_CHK(QPComputeObjectiveFromGradient(qp, xold, gold, &fold));
          PB_CHK(QPComputeObjectiveFromGradient(qp, x, g, &f));
          if (f > fold) {
            lnfinc++;
            if (fallback2) {
              PB_CHK(grads(qps, x, g));
              PB_CHK(vec_dot(gc, gc, &gcTgc));
              PB_CHK(vec_dot(gf, gf, &gfTgf));
              fallback = !(gcTgc <= gamma2 * gfTgf);
            }
            if (fallback) {
              lnfall++;
              currentStepType = 'f';
              PB_CHK(VecCopy(xold, x));
              PB_CHK(VecCopy(gold, g));
              if (fallback2) PB_CHK(grads(qps, xold, gold));
              PB_CHK(expansion_std(qps, afeas, acg));
              PB_CHK(QPCProject(qpc, x, x));
              PB_CHK(mat_mult(A, x, g));
              lnmv++;
              PB_CHK(VecAXPY(g, -1.0, b));
            }
          }
        }
        PB_CHK(grads(qps, x, g));
        PB_CHK(VecCopy(gf, p));
      }
    } else {
      lnprop++;
      currentStepType = 'p';
      PB_CHK(VecCopy(gc, p));
      PB_CHK(mat_mult(A, p, Ap));
      lnmv++;
      PB_CHK(vec_dot(p, Ap, &pAp));
      PB_CHK(vec_dot(g, p, &acg));
      acg = acg / pAp;
      PB_CHK(VecAXPY(x, -acg, p));
      PB_CHK(VecAXPY(g, -acg, Ap));
      PB_CHK(grads(qps, x, g));
      PB_CHK(VecCopy(gf, p));
    }
    qps->iteration++;
  }
  ncg += lncg; nexp += lnexp; nmv += lnmv; nprop += lnprop; nfinc += lnfinc; nfall += lnfall;
  return 0;
}

PetscErrorCode MpgpImpl::solve(QPS qps)
{
  if (fused_eligible(qps)) return solve_fused(qps);
  return solve_generic(qps);
}

static PetscErrorCode QPSCreate_MPGP(QPS qps)
{   // mpgp.c:819-871
  qps->impl = new MpgpImpl;
  return 0;
}

#define MPGP_OR_FAIL(qps)                                                      \
  MpgpImpl *mpgp = mpgp_of(qps);                                               \
  if (!mpgp) return err(PETSC_ERR_ARG_WRONG, "QPS is not of type mpgp")

PetscErrorCode QPSMPGPGetCurrentStepType(QPS qps, char *stepType)
{
  *stepType = ' ';
  MpgpImpl *mpgp = mpgp_of(qps);
  if (mpgp) *stepType = mpgp->currentStepType;
  return 0;
}
PetscErrorCode QPSMPGPSetAlpha(QPS qps, PetscReal alpha, QPSScalarArgType argtype)
{
  MPGP_OR_FAIL(qps);
  mpgp->alpha_user = alpha;
  mpgp->alpha_type = argtype;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSMPGPGetAlpha(QPS qps, PetscReal *alpha, QPSScalarArgType *argtype)
{
  MPGP_OR_FAIL(qps);
  if (alpha) *alpha = mpgp->alpha_user;
  if (argtype) *argtype = mpgp->alpha_type;
  return 0;
}
PetscErrorCode QPSMPGPSetGamma(QPS qps, PetscReal gamma)
{
  MPGP_OR_FAIL(qps);
  mpgp->gamma = gamma;
  return 0;
}
PetscErrorCode QPSMPGPGetGamma(QPS qps, PetscReal *gamma)
{
  MPGP_OR_FAIL(qps);
  *gamma = mpgp->gamma;
  return 0;
}
PetscErrorCode QPSMPGPGetOperatorMaxEigenvalue(QPS qps, PetscReal *maxeig)
{
  MPGP_OR_FAIL(qps);
  *maxeig = mpgp->maxeig;
  return 0;
}
PetscErrorCode QPSMPGPSetOperatorMaxEigenvalue(QPS qps, PetscReal maxeig)
{
  MPGP_OR_FAIL(qps);
  mpgp->maxeig     = maxeig;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSMPGPUpdateMaxEigenvalue(QPS qps, PetscReal maxeig_update)
{   // mpgp.c:119-143
  MPGP_OR_FAIL(qps);
  if (!qps->setupcalled) return err(PETSC_ERR_ARG_WRONGSTATE, "this routine is intended to be called after QPSSetUp");
  mpgp->maxeig = mpgp->maxeig * maxeig_update;
  if (mpgp->alpha_type == QPS_ARG_MULTIPLE) mpgp->alpha = mpgp->alpha / maxeig_update;
  return 0;
}
PetscErrorCode QPSMPGPSetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal tol)
{
  MPGP_OR_FAIL(qps);
  mpgp->maxeig_tol = tol;
  return 0;
}
PetscErrorCode QPSMPGPGetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal *tol)
{
  MPGP_OR_FAIL(qps);
  *tol = mpgp->maxeig_tol;
  return 0;
}
PetscErrorCode QPSMPGPGetOperatorMaxEigenvalueIterations(QPS qps, PetscInt *numit)
{
  MPGP_OR_FAIL(qps);
  *numit = mpgp->maxeig_iter;
  return 0;
}
PetscErrorCode QPSMPGPSetOperatorMaxEigenvalueIterations(QPS qps, PetscInt numit)
{
  MPGP_OR_FAIL(qps);
  mpgp->maxeig_iter = numit;
  return 0;
}
PetscErrorCode QPSMPGPGetStepCounts(QPS qps, PetscInt *nmv, PetscInt *ncg, PetscInt *nexp, PetscInt *nprop)
{
  MPGP_OR_FAIL(qps);
  if (nmv) *nmv = mpgp->nmv;
  if (ncg) *ncg = mpgp->ncg;
  if (nexp) *nexp = mpgp->nexp;
  if (nprop) *nprop = mpgp->nprop;
  return 0;
}

// =====================================================================================================
// SMALXE
// =====================================================================================================
struct SmalxeImpl : QPSImpl {   // QPS_SMALXE smalxeimpl.h:13-67
  QPS              inner = nullptr;
  QP               qp_penalized = nullptr;
  SmalxeInnerCtx  *cctx_inner = nullptr;
  double           M1_user = 1e2, M1_initial = 0, M1_update = 2.0, M1 = 0;
  QPSScalarArgType M1_type = QPS_ARG_MULTIPLE, rho_type = QPS_ARG_MULTIPLE, eta_type = QPS_ARG_MULTIPLE;
  PetscInt         M1_updates = 0, M1_hits = 0, eta_hits = 0, rho_updates = 0;
  double           rtol_E = 1.0, rho_user = 1.1, rho_update = 1.0, rho_update_late = 2.0;
  double           eta_user = 1e-1, eta = 0, update_threshold = 0.0;
  double           maxeig = PETSC_DECIDE, maxeig_tol = PETSC_DECIDE;
  PetscInt         maxeig_iter = PETSC_DECIDE;
  bool             inject_maxeig = false, inject_maxeig_set = false;
  bool             monitor = false, monitor_outer = false, get_lambda = false, get_Bt_lambda = true, knoll = false;
  PetscInt         inner_iter_min = 1, inner_no_gtol_stop = 0;
  int              state = 1;
  PetscInt         inner_iter_accu = 0;
  bool             setfromoptionscalled = false;
  // lagged ||B u|| update (smalxe.c:1190-1200 defaults; :289-370)
  bool             lag_enabled = false, lag_monitor = false, lag_compare = false;
  PetscInt         lag_offset = 2, Jstart = 10, Jstep = 5, Jend = 20;
  double           lag_lower = 0.1, lag_upper = 1.1;
  double           lag_normBu0 = 0.0;
  PetscInt         lag_II = 0, lag_J = 0, lag_neval = 0, lag_niter = 0;
  double           normBu = NAN, normBu_old = NAN, normBu_prev = NAN, enorm = NAN;
  Vec              BtBu = nullptr;

  ~SmalxeImpl() override
  {
    pb::unref(BtBu);
    QPSDestroy(&inner);
  }
  PetscErrorCode setup(QPS qps) override;
  PetscErrorCode solve(QPS qps) override;
  PetscErrorCode reset(QPS qps) override
  {   // QPSReset_SMALXE smalxe.c:1023-1041
    if (qps->solQP) QPRemoveChild(qps->solQP);
    qp_penalized = nullptr;
    normBu = enorm = NAN;
    state           = 1;
    inner_iter_accu = 0;
    M1_updates = M1_hits = eta_hits = rho_updates = 0;
    pb::unref(BtBu);
    if (inner) PB_CHK(QPSReset(inner));
    return 0;
  }
  PetscErrorCode setfromoptions(QPS qps) override;
  PetscErrorCode isqpcompatible(QPS, QP qp, PetscBool *flg) override
  {   // smalxe.c:1080-1091
    *flg = qp->BE ? PETSC_TRUE : PETSC_FALSE;
    return 0;
  }
  PetscErrorCode viewconvergence(QPS, PetscViewer v) override
  {   // smalxe.c:1001-1019
    vprintf_viewer(v, "Total number of inner iterations %d\n", (int)inner_iter_accu);
    vprintf_viewer(v, "#hits    of M1, eta: %3d, %3d\n", (int)M1_hits, (int)eta_hits);
    vprintf_viewer(v, "#updates of M1, rho: %3d, %3d\n", (int)M1_updates, (int)rho_updates);
    vprintf_viewer(v, "inner ");
    return QPSViewConvergence(inner, v);
  }
  int get_inner(QPS qps)
  {   // QPSSMALXEGetInnerQPS_SMALXE smalxe.c:492-506
    if (!inner) {
      PB_CHK(QPSCreate(qps->comm, &inner));
      inner->prefix = qps->prefix + "smalxe_";
    }
    return 0;
  }
  int update_normBu(QPS qps, Vec u, double *nBu, double *en);
  int update_normBu_on(QPS qps, Vec u, double *nBu, double *en);
  int update_normBu_lag_on(QPS qps, Vec u, double *nBu, double *en);
};

static SmalxeImpl *smalxe_of(QPS qps) { return (qps->impl && qps->type == QPSSMALXE) ? static_cast<SmalxeImpl *>(qps->impl) : nullptr; }

PetscErrorCode SmalxeImpl::setfromoptions(QPS qps)
{   // smalxe.c:696-768
  const std::string &p = qps->prefix;
  double             v;
  PetscInt           iv;
  bool               flg1, flg2, direct;
  if (options_real(p, "-qps_smalxe_maxeig", &v)) maxeig = v;
  if (options_real(p, "-qps_smalxe_maxeig_tol", &v)) maxeig_tol = v;
  if (options_int(p, "-qps_smalxe_maxeig_iter", &iv)) maxeig_iter = iv;
  bool inj;
  if (options_bool(p, "-qps_smalxe_maxeig_inject", &inj)) {
    inject_maxeig     = inj;
    inject_maxeig_set = true;
  }
  direct = false; v = eta_user;
  flg1 = options_bool(p, "-qps_smalxe_eta_direct", &direct);
  flg2 = options_real(p, "-qps_smalxe_eta", &v);
  if (flg1 || flg2) { eta_user = v; eta_type = direct ? QPS_ARG_DIRECT : QPS_ARG_MULTIPLE; }
  direct = false; v = rho_user;
  flg1 = options_bool(p, "-qps_smalxe_rho_direct", &direct);
  flg2 = options_real(p, "-qps_smalxe_rho", &v);
  if (flg1 || flg2) { rho_user = v; rho_type = direct ? QPS_ARG_DIRECT : QPS_ARG_MULTIPLE; }
  options_real(p, "-qps_smalxe_rho_update", &rho_update);
  options_real(p, "-qps_smalxe_rho_update_late", &rho_update_late);
  direct = false; v = M1_user;
  flg1 = options_bool(p, "-qps_smalxe_M1_direct", &direct);
  flg2 = options_real(p, "-qps_smalxe_M1", &v);
  if (flg1 || flg2) { M1_user = v; M1_type = direct ? QPS_ARG_DIRECT : QPS_ARG_MULTIPLE; }
  options_real(p, "-qps_smalxe_M1_update", &M1_update);
  options_real(p, "-qps_smalxe_rtol_E", &rtol_E);
  options_bool(p, "-qps_smalxe_get_lambda", &get_lambda);
  options_bool(p, "-qps_smalxe_get_Bt_lambda", &get_Bt_lambda);
  options_bool(p, "-qps_smalxe_monitor", &monitor);
  if (monitor) monitor_outer = true;
  options_bool(p, "-qps_smalxe_monitor_outer", &monitor_outer);
  options_int(p, "-qps_smalxe_inner_iter_min", &inner_iter_min);
  options_int(p, "-qps_smalxe_inner_no_gtol_stop", &inner_no_gtol_stop);
  options_real(p, "-qps_smalxe_update_threshold", &update_threshold);
  options_bool(p, "-qps_smalxe_knoll", &knoll);
  // smalxe.c:754-762.  As in the reference the lag switches only take effect when B_E has no MatMult (the dummy left behind by
  // QPTOrthonormalizeEq(MAT_ORTH_IMPLICIT), smalxe.c:878-886); with an ordinary equality matrix ||B u|| is evaluated exactly in every
  // inner iteration (on the fused path it costs no extra pass: K_B reduces B u of the new iterate).
  options_bool(p, "-qps_smalxe_norm_update_lag", &lag_enabled);
  options_bool(p, "-qps_smalxe_norm_update_lag_monitor", &lag_monitor);
  options_bool(p, "-qps_smalxe_norm_update_lag_compare", &lag_compare);
  options_int(p, "-qps_smalxe_norm_update_lag_offset", &lag_offset);
  options_int(p, "-qps_smalxe_norm_update_lag_start", &Jstart);
  options_int(p, "-qps_smalxe_norm_update_lag_step", &Jstep);
  options_int(p, "-qps_smalxe_norm_update_lag_end", &Jend);
  options_real(p, "-qps_smalxe_norm_update_lag_lower", &lag_lower);
  options_real(p, "-qps_smalxe_norm_update_lag_upper", &lag_upper);
  setfromoptionscalled = true;
  qps->setupcalled     = false;
  return 0;
}

// QPSSMALXEUpdateNormBu_SMALXE smalxe.c:247-261 (c = 0 after homogenisation)
int SmalxeImpl::update_normBu(QPS qps, Vec u, double *nBu, double *en)
{
  QPPF          pf = qps->solQP->pf;
  if (qps->solQP->BE && qps->solQP->BE->kind == MK_DUMMY)   // smalxe.c:878-886: B_E has no MatMult (implicit orthonormalisation)
    return lag_enabled ? update_normBu_lag_on(qps, u, nBu, en) : update_normBu_on(qps, u, nBu, en);
  const double *Bd, *du;
  int           m;
  PB_CHK(qppf_dense_rows(pf, &Bd, &m));
  PB_CHK(vec_dev_read(u, &du));
  double t[PB_MAXEQ_ALL], s = 0.0;
  PB_CHK(dense_rows_mult_host(qps->comm, u->n, m, Bd, du, t));
  for (int j = 0; j < m; j++) s += t[j] * t[j];
  *nBu = sqrt(s);
  *en  = *nBu / rtol_E;
  return 0;
}

// QPSSMALXEUpdateNormBu_SMALXEON smalxe.c:265-285: ||B u|| = sqrt(u' B'B u) with B'B the penalised term of the inner Hessian
// (Q = B'(BB')^-1 B for implicitly orthonormal rows); B'B u is left in work[0] for the multiplier update
int SmalxeImpl::update_normBu_on(QPS qps, Vec u, double *nBu, double *en)
{
  double dot;
  PB_CHK(QPPFApplyGtG(qps->solQP->pf, u, BtBu));
  PB_CHK(vec_dot(u, BtBu, &dot));
  *nBu = sqrt(dot);
  *en  = *nBu / rtol_E;
  return 0;
}
// QPSSMALXEUpdateNormBu_Lag_SMALXEON smalxe.c:289-370: the norm is re-evaluated every J-th inner iteration only (J grows from Jstart to
// Jend in steps of Jstep while consecutive exact values stay within [lower, upper) of each other); in between the last exact value is used.
// The reference keeps the counters in function statics; here they live in the solver object.
int SmalxeImpl::update_normBu_lag_on(QPS qps, Vec u, double *nBu, double *en)
{
  double normBu_approx, normBu_exact = 0.0, enorm_exact, rdiff;
  bool   eval = false;
  if (inner->iteration <= lag_offset) {
    PB_CHK(update_normBu_on(qps, u, &normBu_exact, &enorm_exact));
    eval = true;
    lag_neval++;
    lag_normBu0   = normBu_exact;
    normBu_approx = lag_normBu0;
    lag_J         = Jstart;
    lag_II        = 0;
  } else {
    if (lag_II == 0) {
      PB_CHK(update_normBu_on(qps, u, &normBu_exact, &enorm_exact));
      eval = true;
      lag_neval++;
      rdiff = fabs(normBu_exact / lag_normBu0);
      if (rdiff >= lag_upper || rdiff < lag_lower) {
        lag_II = 0;
        lag_J  = Jstart;
      } else {
        lag_II++;
      }
      lag_normBu0 = normBu_exact;
    } else {
      lag_II++;
    }
    normBu_approx = lag_normBu0;
  }
  lag_niter++;
  if (lag_II == lag_J) {
    lag_II = 0;
    if (lag_J < Jend) lag_J += Jstep;
  }
  if (lag_compare) {
    if (!eval) PB_CHK(update_normBu_on(qps, u, &normBu_exact, &enorm_exact));
    rdiff           = fabs(normBu_approx - normBu_exact) / normBu_exact;
    const char sign = (normBu_exact > normBu_approx) ? '>' : ((normBu_exact < normBu_approx) ? '<' : '=');
    vprintf_viewer(nullptr, "QPSSMALXEUpdateNormBu_Lag_SMALXEON: out %3d in %4d   II=%2d J=%2d niter=%4d neval=%4d   ||Bu||=%.4e  %c  %.4e=~||Bu|| relative_difference=%.4e %c\n",
                   (int)qps->iteration, (int)inner->iteration, (int)lag_II, (int)lag_J, (int)lag_niter, (int)lag_neval, normBu_exact, sign, normBu_approx, rdiff, rdiff > 10 ? sign : ' ');
  } else if (lag_monitor) {
    vprintf_viewer(nullptr, "QPSSMALXEUpdateNormBu_Lag_SMALXEON: out %3d in %4d   II=%2d J=%2d niter=%4d neval=%4d\n", (int)qps->iteration, (int)inner->iteration, (int)lag_II,
                   (int)lag_J, (int)lag_niter, (int)lag_neval);
  }
  *nBu = normBu_approx;
  *en  = *nBu / rtol_E;
  return 0;
}

// host version of the inner stopping rule (used with monitors / the generic driver)
extern "C" PetscErrorCode QPSConverged_Inner_SMALXE(QPS qps_inner, KSPConvergedReason *reason)
{   // smalxe.c:610-692
  SmalxeInnerCtx *cctx = (SmalxeInnerCtx *)qps_inner->cnvctx;
  QPS             qps_outer = cctx->qps_outer;
  SmalxeImpl     *sm = cctx->smalxe;
  const PetscInt  i = qps_inner->iteration;
  const double    gnorm = qps_inner->rnorm;
  *reason = KSP_CONVERGED_ITERATING;
  PB_CHK(sm->update_normBu(qps_outer, qps_inner->solQP->x, &sm->normBu, &sm->enorm));
  qps_outer->rnorm = std::max(sm->enorm, gnorm);
  cctx->MNormBu    = sm->M1 * sm->normBu;
  qps_inner->atol  = std::min(cctx->MNormBu, sm->eta);
  if (sm->monitor) vprintf_viewer(nullptr, "  %4d %c  %.8e  %.8e  %c = %.8e %c %.8e  %.8e %c %.8e = %-8s  %.8e\n", (int)i, mpgp_of(qps_inner) ? mpgp_of(qps_inner)->currentStepType : ' ', gnorm,
                                  sm->enorm, (gnorm > sm->enorm) ? 'G' : 'E', qps_outer->rnorm, (qps_outer->rnorm < cctx->ttol_outer) ? '<' : '>', cctx->ttol_outer, gnorm,
                                  (gnorm < qps_inner->atol) ? '<' : '>', qps_inner->atol, (cctx->MNormBu < sm->eta) ? "M1||Bu||" : "eta", cctx->MNormBu);
  if (i > qps_inner->max_it - sm->inner_iter_accu) {
    *reason           = KSP_DIVERGED_ITS;
    qps_outer->reason = KSP_DIVERGED_BREAKDOWN;
    return 0;
  }
  if (pb_isnanorinf(gnorm)) {
    *reason           = KSP_DIVERGED_NANORINF;
    qps_outer->reason = KSP_DIVERGED_BREAKDOWN;
    return 0;
  }
  PB_CHK(qps_outer->convergencetest(qps_outer, &qps_outer->reason));
  if (qps_outer->reason) {
    *reason = (qps_outer->reason > 0) ? KSP_CONVERGED_HAPPY_BREAKDOWN : KSP_DIVERGED_BREAKDOWN;
    return 0;
  }
  if (gnorm < qps_inner->atol) {
    *reason = KSP_CONVERGED_ATOL;
    if (cctx->MNormBu < sm->eta) sm->M1_hits++;
    else sm->eta_hits++;
    return 0;
  }
  if (sm->state == 3 && (i < sm->inner_iter_min || sm->inner_no_gtol_stop)) return 0;
  if (gnorm <= cctx->gtol) {
    if (!(qps_inner->rnorm > sm->enorm)) {
      if (sm->inner_no_gtol_stop < 2) *reason = KSP_CONVERGED_RTOL;
      if (sm->state != 3) sm->state = 3;
    }
  }
  return 0;
}

// the same rule, handed to the device-driven inner MPGP as numbers
int smalxe_fill_ctl(QPS inner, MpgpCtl *S, bool *host_needed)
{
  SmalxeInnerCtx *cctx = (SmalxeInnerCtx *)inner->cnvctx;
  QPS             outer = cctx->qps_outer;
  SmalxeImpl     *sm = cctx->smalxe;
  *host_needed = sm->monitor || (outer->convergencetest != QPSConvergedDefault);
  S->M1 = sm->M1; S->eta = sm->eta; S->rtol_E = sm->rtol_E; S->gtol = cctx->gtol;
  QPSConvergedDefaultCtx *oc = (QPSConvergedDefaultCtx *)outer->cnvctx;
  if (outer->convergencetest == QPSConvergedDefault) {
    if (!oc->setup_called) PB_CHK(QPSConvergedDefaultSetUp(outer));   // first call inside the first inner iteration (qps.c:686)
    S->outer_ttol = oc->ttol;
    S->outer_norm_rhs_div = oc->norm_rhs_div;
  }
  S->outer_atol = outer->atol; S->outer_divtol = outer->divtol;
  S->outer_max_it = outer->max_it; S->outer_iteration = outer->iteration;
  S->smalxe_state = sm->state; S->inner_iter_min = sm->inner_iter_min; S->inner_no_gtol_stop = sm->inner_no_gtol_stop;
  S->inner_iter_accu = sm->inner_iter_accu;
  S->M1_hits = 0; S->eta_hits = 0;
  S->outer_reason = outer->reason;
  return 0;
}
int smalxe_read_ctl(QPS inner, const MpgpCtl *S)
{
  SmalxeInnerCtx *cctx = (SmalxeInnerCtx *)inner->cnvctx;
  QPS             outer = cctx->qps_outer;
  SmalxeImpl     *sm = cctx->smalxe;
  if (S->host_conv) return 0;   // the host test keeps these fields itself
  sm->normBu = S->normBu; sm->enorm = S->enorm; sm->state = S->smalxe_state;
  sm->M1_hits += S->M1_hits; sm->eta_hits += S->eta_hits;
  cctx->MNormBu = S->MNormBu;
  inner->atol   = S->atol;
  outer->rnorm  = S->outer_rnorm;
  outer->reason = (KSPConvergedReason)S->outer_reason;
  return 0;
}

PetscErrorCode SmalxeImpl::setup(QPS qps)
{   // QPSSetUp_SMALXE smalxe.c:772-888
  QP qp = qps->solQP;
  if (qp->cE) {   // :782-787
    PB_CHK(QPTHomogenizeEq(qp));
    QP last;
    PB_CHK(QPChainGetLast(qp, &last));
    pb::ref(last);
    pb::unref(qps->solQP);
    qps->solQP = last;
    qp         = last;
    PB_CHK(QPSetUp(qp));
  }
  PB_CHK(get_inner(qps));
  Mat A = qp->A;
  pb::unref(BtBu);
  PB_CHK(VecDuplicate(qp->x, &BtBu));   // QPSSetWorkVecs(qps,1)
  PB_CHK(VecInvalidate(qp->lambda_E));
  PB_CHK(VecZeroEntries(qp->Bt_lambda));
  eta = eta_user;   // :806-811
  if (eta_type == QPS_ARG_MULTIPLE) {
    double normb;
    PB_CHK(vec_norm2(qp->b, &normb));
    eta *= normb;
  }
  M1_initial = M1_user;   // :814-818
  if (M1_type == QPS_ARG_MULTIPLE) {
    if (maxeig == PETSC_DECIDE) PB_CHK(MatGetMaxEigenvalue(A, NULL, &maxeig, maxeig_tol, maxeig_iter));
    M1_initial *= maxeig;
  }
  double rho;   // :821-826
  if (rho_type == QPS_ARG_MULTIPLE) {
    if (maxeig == PETSC_DECIDE) PB_CHK(MatGetMaxEigenvalue(A, NULL, &maxeig, maxeig_tol, maxeig_iter));
    rho = rho_user * maxeig;
  } else {
    rho = rho_user;
  }
  PB_CHK(QPPFSetUp(qp->pf));   // :834
  PB_CHK(QPRemoveChild(qp));   // :837
  PB_CHK(QPTEnforceEqByPenalty(qp, rho, PETSC_TRUE));
  PB_CHK(QPChainGetLast(qp, &qp_penalized));
  QP qp_inner = qp_penalized;
  if (qp_inner == qp) return err(PETSC_ERR_PLIB, "penalised child was not created (rho = 0?)");
  Vec b_inner;   // :850-853 independent copy of b
  PB_CHK(VecDuplicate(qp->b, &b_inner));
  PB_CHK(VecCopy(qp->b, b_inner));
  PB_CHK(QPSetRhs(qp_inner, b_inner));
  PB_CHK(VecDestroy(&b_inner));
  PB_CHK(QPSSetQP(inner, qp_inner));   // :856
  if (setfromoptionscalled) PB_CHK(QPSSetFromOptions(inner));
  else if (!inner->impl) PB_CHK(QPSSetDefaultType(inner));
  double    maxeig_inner = std::max(rho, maxeig);   // :865
  PetscBool orth;
  PB_CHK(QPPFGetGHasOrthonormalRows(qp->pf, &orth));
  if (!inject_maxeig_set) inject_maxeig = orth;
  if (inject_maxeig) PB_CHK(QPSMPGPSetOperatorMaxEigenvalue(inner, maxeig_inner));
  PB_CHK(QPSSetAutoPostSolve(inner, PETSC_FALSE));
  PB_CHK(QPSSetUp(inner));   // :871
  cctx_inner            = new SmalxeInnerCtx;   // :874-875
  cctx_inner->qps_outer = qps;
  cctx_inner->smalxe    = this;
  PB_CHK(QPSSetConvergenceTest(inner, QPSConverged_Inner_SMALXE, cctx_inner, [](void *c) -> PetscErrorCode {
    delete (SmalxeInnerCtx *)c;
    return 0;
  }));
  return 0;
}

PetscErrorCode SmalxeImpl::solve(QPS qps)
{   // QPSSolve_SMALXE smalxe.c:893-997
  QP     qp = qps->solQP, qp_inner = qp_penalized;
  Vec    b = qp->b, u = qp->x, Btmu = qp->Bt_lambda, b_inner = qp_inner->b;
  Mat    A_inner = qp_inner->A;
  double Lag, Lag_old, rho = A_inner->rho;
  const PetscInt maxits = qps->max_it;
  PetscInt       i;
  M1 = M1_initial;
  PB_CHK(VecZeroEntries(Btmu));   // :935
  if (knoll) PB_CHK(QPPFApplyP(qp->pf, b, u));   // :938-943
  PB_CHK(QPSetUp(qp_inner));
  PB_CHK(QPComputeObjective(qp_inner, u, &Lag_old));   // :946
  PB_CHK(update_normBu(qps, u, &normBu_old, &enorm));  // :949
  normBu_prev     = normBu_old;
  qps->iteration  = 0;
  inner_iter_accu = 0;
  qps->reason     = KSP_CONVERGED_ITERATING;
  PB_CHK(QPSResetStatistics(inner));   // :955
  QPSConvergedDefaultCtx *oc = (qps->convergencetest == QPSConvergedDefault) ? (QPSConvergedDefaultCtx *)qps->cnvctx : nullptr;
  for (i = 0; i < maxits; i++) {   // :957
    // QPSSMALXEUpdateLambda_SMALXE :402-435: Btmu += rho * B'B u
    PB_CHK(QPPFApplyGtG(qp->pf, u, BtBu));
    PB_CHK(VecAXPY(Btmu, rho, BtBu));
    if (qps->reason) break;   // :962
    PB_CHK(VecWAXPY(b_inner, -1.0, Btmu, b));   // :965
    inner->divtol = qps->divtol;                // :968
    {   // QPSConvergedSetUp_Inner_SMALXE :537-557
      PB_CHK(vec_norm2(b, &cctx_inner->norm_rhs_outer));
      cctx_inner->gtol       = qps->rtol * cctx_inner->norm_rhs_outer;
      cctx_inner->ttol_outer = std::max(qps->rtol * cctx_inner->norm_rhs_outer, qps->atol);
      if (oc) PB_CHK(vec_norm2(b_inner, &oc->norm_rhs_div));   // QPSConvergedDefaultSetRhsForDivergence qps.c:736-744
    }
    PB_CHK(QPSSolve(inner));   // :970
    inner_iter_accu += inner->iteration;
    qps->iteration = i + 1;
    PB_CHK(update_normBu(qps, u, &normBu, &enorm));   // :976
    rho = A_inner->rho;                               // :979
    PB_CHK(QPComputeObjective(qp_inner, u, &Lag));    // :982
    {   // QPSSMALXEUpdate_SMALXE :439-488
      const double t = 0.5 * rho * normBu * normBu, t2 = Lag - (Lag_old + t);
      const bool   flag = (t2 < update_threshold);
      if (monitor_outer) {
        vprintf_viewer(nullptr, "END   outer %3d:  Lagrangian L       L-L_old      L-(L_old+1/2*rho*||Bu||^2) %c threshold    1/2*rho*||Bu||^2\n", (int)qps->iteration, flag ? '<' : '>');
        vprintf_viewer(nullptr, "                  %+.10e  %+.3e                   %+.3e %c %+.3e   %.3e\n", Lag, Lag - Lag_old, t2, flag ? '<' : '>', update_threshold, t);
      }
      if (flag && M1_update != 1.0) {
        if (inner->reason == KSP_CONVERGED_ATOL) {
          M1 = M1 / M1_update;
          M1_updates++;
        }
      }
      if (!(inner->rnorm > enorm)) {   // :482; QPSSMALXEUpdateRho_SMALXE :373-398
        const double ru = (state == 3) ? rho_update_late : rho_update;
        const bool   lagflag = (state == 3) ? true : flag;
        if (lagflag && ru != 1.0) {
          PB_CHK(MatPenalizedUpdatePenalty(A_inner, ru));
          PB_CHK(QPSMPGPUpdateMaxEigenvalue(inner, ru));
          rho_updates++;
        }
      }
    }
    Lag_old    = Lag;
    normBu_old = normBu;
  }
  if (i == maxits && !qps->reason) qps->reason = KSP_DIVERGED_ITS;   // :986-989
  if (get_lambda) {   // :994
    PB_CHK(QPPFApplyHalfQ(qp->pf, qp->Bt_lambda, qp->lambda_E));
    qp->lambda_E->invalidated = false;
  }
  pb::vec_mark_invalid(qp->Bt_lambda, !get_Bt_lambda);   // :995
  return 0;
}

static PetscErrorCode QPSCreate_SMALXE(QPS qps)
{   // smalxe.c:1095-1209
  qps->impl   = new SmalxeImpl;
  qps->max_it = 100;   // :1203
  return 0;
}

#define SMALXE_OR_FAIL(qps)                                                    \
  SmalxeImpl *sm = smalxe_of(qps);                                             \
  if (!sm) return err(PETSC_ERR_ARG_WRONG, "QPS is not of type smalxe")

PetscErrorCode QPSSMALXEGetInnerQPS(QPS qps, QPS *inner)
{
  SMALXE_OR_FAIL(qps);
  PB_CHK(sm->get_inner(qps));
  *inner = sm->inner;
  return 0;
}
PetscErrorCode QPSSMALXESetOperatorMaxEigenvalue(QPS qps, PetscReal maxeig)
{
  SMALXE_OR_FAIL(qps);
  sm->maxeig       = maxeig;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalue(QPS qps, PetscReal *maxeig)
{
  SMALXE_OR_FAIL(qps);
  *maxeig = sm->maxeig;
  return 0;
}
PetscErrorCode QPSSMALXESetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal tol)
{
  SMALXE_OR_FAIL(qps);
  sm->maxeig_tol = tol;
  return 0;
}
PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal *tol)
{
  SMALXE_OR_FAIL(qps);
  *tol = sm->maxeig_tol;
  return 0;
}
PetscErrorCode QPSSMALXESetOperatorMaxEigenvalueIterations(QPS qps, PetscInt numit)
{
  SMALXE_OR_FAIL(qps);
  sm->maxeig_iter = numit;
  return 0;
}
PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalueIterations(QPS qps, PetscInt *numit)
{
  SMALXE_OR_FAIL(qps);
  *numit = sm->maxeig_iter;
  return 0;
}
PetscErrorCode QPSSMALXESetInjectOperatorMaxEigenvalue(QPS qps, PetscBool flg)
{
  SMALXE_OR_FAIL(qps);
  sm->inject_maxeig     = flg;
  sm->inject_maxeig_set = true;
  return 0;
}
PetscErrorCode QPSSMALXEGetInjectOperatorMaxEigenvalue(QPS qps, PetscBool *flg)
{
  SMALXE_OR_FAIL(qps);
  *flg = sm->inject_maxeig ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode QPSSMALXESetEta(QPS qps, PetscReal eta, QPSScalarArgType argtype)
{
  SMALXE_OR_FAIL(qps);
  sm->eta_user     = eta;
  sm->eta_type     = argtype;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSSMALXEGetEta(QPS qps, PetscReal *eta, QPSScalarArgType *argtype)
{
  SMALXE_OR_FAIL(qps);
  if (eta) *eta = sm->eta_user;
  if (argtype) *argtype = sm->eta_type;
  return 0;
}
PetscErrorCode QPSSMALXESetM1Initial(QPS qps, PetscReal M1_initial, QPSScalarArgType argtype)
{
  SMALXE_OR_FAIL(qps);
  sm->M1_user      = M1_initial;
  sm->M1_type      = argtype;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSSMALXEGetM1Initial(QPS qps, PetscReal *M1_initial, QPSScalarArgType *argtype)
{
  SMALXE_OR_FAIL(qps);
  if (M1_initial) *M1_initial = sm->M1_user;
  if (argtype) *argtype = sm->M1_type;
  return 0;
}
PetscErrorCode QPSSMALXESetM1Update(QPS qps, PetscReal M1_update)
{
  SMALXE_OR_FAIL(qps);
  sm->M1_update = M1_update;
  return 0;
}
PetscErrorCode QPSSMALXEGetM1Update(QPS qps, PetscReal *M1_update)
{
  SMALXE_OR_FAIL(qps);
  *M1_update = sm->M1_update;
  return 0;
}
PetscErrorCode QPSSMALXESetRhoInitial(QPS qps, PetscReal rho_initial, QPSScalarArgType argtype)
{
  SMALXE_OR_FAIL(qps);
  sm->rho_user     = rho_initial;
  sm->rho_type     = argtype;
  qps->setupcalled = false;
  return 0;
}
PetscErrorCode QPSSMALXEGetRhoInitial(QPS qps, PetscReal *rho_initial, QPSScalarArgType *argtype)
{
  SMALXE_OR_FAIL(qps);
  if (rho_initial) *rho_initial = sm->rho_user;
  if (argtype) *argtype = sm->rho_type;
  return 0;
}
PetscErrorCode QPSSMALXESetRhoUpdate(QPS qps, PetscReal rho_update)
{
  SMALXE_OR_FAIL(qps);
  sm->rho_update = rho_update;
  return 0;
}
PetscErrorCode QPSSMALXEGetRhoUpdate(QPS qps, PetscReal *rho_update)
{
  SMALXE_OR_FAIL(qps);
  *rho_update = sm->rho_update;
  return 0;
}
PetscErrorCode QPSSMALXESetRhoUpdateLate(QPS qps, PetscReal rho_update_late)
{
  SMALXE_OR_FAIL(qps);
  sm->rho_update_late = rho_update_late;
  return 0;
}
PetscErrorCode QPSSMALXEGetRhoUpdateLate(QPS qps, PetscReal *rho_update_late)
{
  SMALXE_OR_FAIL(qps);
  *rho_update_late = sm->rho_update_late;
  return 0;
}
PetscErrorCode QPSSMALXESetMonitor(QPS qps, PetscBool flg)
{
  SMALXE_OR_FAIL(qps);
  sm->monitor = flg;
  return 0;
}
PetscErrorCode QPSSMALXEGetStatistics(QPS qps, PetscInt *inner_iter_accu, PetscInt *M1_hits, PetscInt *eta_hits, PetscInt *M1_updates, PetscInt *rho_updates)
{
  SMALXE_OR_FAIL(qps);
  if (inner_iter_accu) *inner_iter_accu = sm->inner_iter_accu;
  if (M1_hits) *M1_hits = sm->M1_hits;
  if (eta_hits) *eta_hits = sm->eta_hits;
  if (M1_updates) *M1_updates = sm->M1_updates;
  if (rho_updates) *rho_updates = sm->rho_updates;
  return 0;
}
