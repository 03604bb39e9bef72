// qps_lin.cpp -- the two linear QPS types next to the hot path (SURVEY 8f rank 4), on the same device kernels:
//   "ksp"  : QPSKSP  (src/qps/impls/ksp/qpsksp.c) = unpreconditioned CG for unconstrained QPs, the default type when a QP has
//            no constraints (qps.c:448-451)
//   "pcpg" : QPSPCPG (src/qps/impls/pcpg/pcpg.c) = projected CG for equality-constrained QPs
// One kernel per reference Vec/Mat call (SpMV, dot, axpy), in the reference's order; no PETSc KSP object exists here, so the
// KSP-typed accessors of qpsksp.c are reduced to the type name ("cg").
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "objects.h"

using namespace pb;

namespace {
struct LinWork {
  std::vector<Vec> work;
  ~LinWork() { clear(); }
  void clear()
  {
    for (auto &w : work) pb::unref(w);
    work.clear();
  }
  int set(QPS qps, int nw)
  {
    clear();
    work.assign(nw, nullptr);
    for (int i = 0; i < nw; i++) PB_CHK(VecDuplicate(qps->solQP->x, &work[i]));
    return 0;
  }
};

// ---- QPSKSP ------------------------------------------------------------------------------------------
struct KspImpl : QPSImpl {
  LinWork W;
  PetscErrorCode isqpcompatible(QPS, QP qp, PetscBool *flg) override
  {   // QPSIsQPCompatible_KSP qpsksp.c:205-219
    *flg = (qp->BE || qp->cE || qp->qpc) ? PETSC_FALSE : PETSC_TRUE;
    return 0;
  }
  PetscErrorCode setup(QPS qps) override { return W.set(qps, 3); }
  PetscErrorCode reset(QPS) override
  {
    W.clear();
    return 0;
  }
  PetscErrorCode viewconvergence(QPS, PetscViewer v) override
  {   // QPSViewConvergence_KSP qpsksp.c:176-189
    vprintf_viewer(v, "KSPType: %s\n", "cg");
    return 0;
  }
  // QPSSolve_KSP (qpsksp.c:137-153) -> KSPSolve on KSPCG / PCNONE / KSP_NORM_UNPRECONDITIONED / non-zero initial guess
  // (QPSCreate_KSP qpsksp.c:232-253); the stopping test is the QPS one (QPSKSPConverged_KSP qpsksp.c:5-14).
  // Fused form for a packed AIJ or a dense Hessian on one GPU (-qps_ksp_b200_driver generic switches it off): per iteration ONE SpMV kernel that
  // also reduces p.Ap (the power-method skeleton, kernels.cu: EpiPower with s = 1), ONE update kernel (x += a p, r -= a w, r.r) and the
  // direction update -- 3 kernels and 2 host round trips instead of 7 and 4, 11 vector passes instead of 15.  Same recurrence, same
  // stopping test; the products p.w and r.r are summed by other kernels than in the un-fused form (deterministic, different order).
  bool fused_ok(QPS qps) const
  {
    Mat A = qps->solQP->A;
    std::string d = "auto";
    options_string(qps->prefix, "-qps_ksp_b200_driver", &d);
    if (d == "generic") return false;
    if ((A->kind != MK_AIJ && A->kind != MK_DENSE) || A->comm->size != 1 || A->m != A->n || A->eq_host) return false;
    if (mat_ensure_device(A)) return false;
    return A->Ad.kind == 3 || A->Ad.kind == 4 || A->Ad.kind == 6;
  }
  PetscErrorCode solve_fused(QPS qps)
  {
    QP       qp = qps->solQP;
    Mat      A = qp->A;
    Vec      b = qp->b, x = qp->x, R = W.work[0], P = W.work[1], Wv = W.work[2];
    double   beta, betaold = 1.0, dpi, dp;
    PetscInt i = 0;
    const PetscInt n = x->n;
    Reducer &Rd = reducer(qps->comm);
    PB_CHK(mat_mult(A, x, R));
    PB_CHK(VecAYPX(R, -1.0, b));
    PB_CHK(vec_dot(R, R, &beta));
    dp             = sqrt(beta);
    qps->iteration = 0;
    qps->rnorm     = dp;
    PB_CHK(qps->convergencetest(qps, &qps->reason));
    if (qps->reason) return 0;
    do {
      if (beta == 0.0) {
        qps->reason = KSP_CONVERGED_ATOL;
        break;
      }
      if (!i) {
        PB_CHK(VecCopy(R, P));
      } else {
        PB_CHK(VecAYPX(P, beta / betaold, R));
      }
      const double *dP, *dW;
      double       *dWw, *dx, *dR;
      PB_CHK(vec_dev_read(P, &dP));
      PB_CHK(vec_dev_write(Wv, &dWw));
      PB_CHK(k_power_step(A->Ad, dP, 1.0, dWw, Rd.rb));   // w = A p, out[0] = p.w
      PB_CHK(Rd.fetch());
      dpi     = Rd.sum(0);
      betaold = beta;
      if (!(dpi > 0.0)) {
        qps->reason = KSP_DIVERGED_INDEFINITE_MAT;
        break;
      }
      const double a = beta / dpi;
      PB_CHK(vec_dev_read(Wv, &dW));
      PB_CHK(vec_dev_rw(x, &dx));
      PB_CHK(vec_dev_rw(R, &dR));
      PB_CHK(k_cg_update(n, a, dP, dW, dx, dR, Rd.rb));
      PB_CHK(Rd.fetch());
      beta           = Rd.sum(0);
      dp             = sqrt(beta);
      qps->iteration = i + 1;
      qps->rnorm     = dp;
      PB_CHK(qps->convergencetest(qps, &qps->reason));
      i++;
      if (qps->reason) break;
    } while (i < qps->max_it);
    if (!qps->reason) qps->reason = KSP_DIVERGED_ITS;
    qps->iteration = i;
    return 0;
  }
  PetscErrorCode solve(QPS qps) override
  {
    if (fused_ok(qps)) return solve_fused(qps);
    QP     qp = qps->solQP;
    Mat    A = qp->A;
    Vec    b = qp->b, x = qp->x, R = W.work[0], P = W.work[1], Wv = W.work[2];
    double beta, betaold = 1.0, dpi, dp;
    PetscInt i = 0;
    PB_CHK(mat_mult(A, x, R));
    PB_CHK(VecAYPX(R, -1.0, b));
    PB_CHK(vec_norm2(R, &dp));
    qps->iteration = 0;
    qps->rnorm     = dp;
    PB_CHK(qps->convergencetest(qps, &qps->reason));
    if (qps->reason) return 0;
    PB_CHK(vec_dot(R, R, &beta));
    do {
      if (beta == 0.0) {
        qps->reason = KSP_CONVERGED_ATOL;
        break;
      }
      if (!i) {
        PB_CHK(VecCopy(R, P));
      } else {
        PB_CHK(VecAYPX(P, beta / betaold, R));
      }
      PB_CHK(mat_mult(A, P, Wv));
      PB_CHK(vec_dot(P, Wv, &dpi));
      betaold = beta;
      if (!(dpi > 0.0)) {
        qps->reason = KSP_DIVERGED_INDEFINITE_MAT;
        break;
      }
      const double a = beta / dpi;
      PB_CHK(VecAXPY(x, a, P));
      PB_CHK(VecAXPY(R, -a, Wv));
      PB_CHK(vec_norm2(R, &dp));
      qps->iteration = i + 1;
      qps->rnorm     = dp;
      PB_CHK(qps->convergencetest(qps, &qps->reason));
      i++;
      if (qps->reason) break;
      PB_CHK(vec_dot(R, R, &beta));
    } while (i < qps->max_it);
    if (!qps->reason) qps->reason = KSP_DIVERGED_ITS;
    qps->iteration = i;
    return 0;
  }
};

// ---- QPSPCPG -----------------------------------------------------------------------------------------
struct PcpgImpl : QPSImpl {
  LinWork W;
  PetscErrorCode isqpcompatible(QPS, QP qp, PetscBool *flg) override
  {   // QPSIsQPCompatible_PCPG pcpg.c:13-22
    *flg = (qp->qpc || !qp->BE) ? PETSC_FALSE : PETSC_TRUE;
    return 0;
  }
  PetscErrorCode setup(QPS qps) override
  {   // QPSSetup_PCPG pcpg.c:31-41
    if (qps->solQP->cE) {
      QP last;
      PB_CHK(QPTHomogenizeEq(qps->solQP));
      PB_CHK(QPChainGetLast(qps->solQP, &last));
      pb::ref(last);
      QPDestroy(&qps->solQP);
      qps->solQP = last;
      PB_CHK(QPChainSetUp(last));   // the child gets its x (a copy of the parent's) before the work vectors are shaped after it
    }
    return W.set(qps, 6);
  }
  PetscErrorCode reset(QPS) override
  {
    W.clear();
    return 0;
  }
  PetscErrorCode solve(QPS qps) override
  {   // QPSSolve_PCPG pcpg.c:49-131, PCNONE branch (y = w)
    QP     qp = qps->solQP;
    Mat    A = qp->A;
    QPPF   cp;
    Vec    lm = qp->x, rhs = qp->b, p = W.work[0], r = W.work[1], w = W.work[2], Ap = W.work[5];
    double alpha, alpha1, beta, beta1 = 0.0, beta2;
    PB_CHK(QPGetQPPF(qp, &cp));
    PB_CHK(mat_mult(A, lm, r));
    PB_CHK(VecAYPX(r, -1.0, rhs));
    qps->iteration = 0;
    do {
      PB_CHK(QPPFApplyP(cp, r, w));
      PB_CHK(vec_norm2(w, &qps->rnorm));
      PB_CHK(qps->convergencetest(qps, &qps->reason));
      if (qps->reason) break;
      beta2 = beta1;
      PB_CHK(vec_dot(w, w, &beta1));
      if (!qps->iteration) {
        beta = 0;
        PB_CHK(VecCopy(w, p));
      } else {
        beta = beta1 / beta2;
        PB_CHK(VecAYPX(p, beta, w));
      }
      PB_CHK(mat_mult(A, p, Ap));
      PB_CHK(vec_dot(p, Ap, &alpha1));
      alpha = beta1 / alpha1;
      PB_CHK(VecAXPY(lm, alpha, p));
      PB_CHK(VecAXPY(r, -alpha, Ap));
      qps->iteration++;
    } while (qps->iteration < qps->max_it);
    return 0;
  }
};
}   // namespace

PetscErrorCode QPSCreate_KSP(QPS qps)
{
  qps->impl = new KspImpl;
  return 0;
}
PetscErrorCode QPSCreate_PCPG(QPS qps)
{
  qps->impl = new PcpgImpl;
  return 0;
}

PetscErrorCode QPSKSPSetType(QPS qps, const char *type)
{   // qpsksp.c:83-96: only CG exists on this path
  if (qps->type != QPSKSP) return err(PETSC_ERR_SUP, "This is a QPSKSP specific routine!");
  if (!type || strcmp(type, "cg")) return err(PETSC_ERR_SUP, "the B200 QPSKSP provides the \"cg\" Krylov method only (got %s)", type ? type : "NULL");
  return 0;
}
PetscErrorCode QPSKSPGetType(QPS qps, const char **type)
{   // qpsksp.c:100-113
  if (qps->type != QPSKSP) return err(PETSC_ERR_SUP, "This is a QPSKSP specific routine!");
  *type = "cg";
  return 0;
}
