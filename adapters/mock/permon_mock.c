/* permon_mock.c -- TEST INFRASTRUCTURE: implementation of adapters/mock/permon_mock.h (sequential host-array Mat / Vec, a QP container and
 * the part of the QPS front end that dispatches through _QPSOps: registration by name, QPSSetType, QPSSetUp, QPSSolve, QPSViewConvergence).
 * The dispatch order follows the reference: src/qps/interface/qpsregis.c:29-36, qps.c:379-406 (SetType), :198-221 (SetUp), :537-555 (Solve),
 * :968-1000 (ViewConvergence). */
#include "permon_mock.h"
#include <stdarg.h>

struct _p_PetscViewer PETSC_VIEWER_STDOUT_WORLD_OBJ = {{"ascii", NULL, PETSC_COMM_WORLD, 0}, NULL};

MPI_Comm PetscObjectComm(PetscObject o) { return o ? o->comm : PETSC_COMM_SELF; }
PetscErrorCode PetscObjectTypeCompare(PetscObject o, const char *type, PetscBool *same)
{
  *same = (o && o->type_name && !strcmp(o->type_name, type)) ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode PetscObjectGetOptionsPrefix(PetscObject o, const char **prefix) { *prefix = o->prefix; return 0; }
PetscErrorCode PetscObjectStateIncrease(PetscObject o) { o->state++; return 0; }

static char g_options[4096];
PetscErrorCode PetscOptionsSetValue(void *options, const char *name, const char *value)
{
  (void)options;
  strncat(g_options, name, sizeof g_options - strlen(g_options) - 2);
  strncat(g_options, " ", sizeof g_options - strlen(g_options) - 2);
  if (value) {
    strncat(g_options, value, sizeof g_options - strlen(g_options) - 2);
    strncat(g_options, " ", sizeof g_options - strlen(g_options) - 2);
  }
  return 0;
}
PetscErrorCode PetscOptionsGetAll(void *options, char **copts)
{
  (void)options;
  *copts = strdup(g_options);
  return *copts ? 0 : 55;
}
PetscErrorCode PetscViewerASCIIPrintf(PetscViewer v, const char *fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  vfprintf((v && v->f) ? v->f : stdout, fmt, ap);
  va_end(ap);
  return 0;
}

/* ---- Vec ---------------------------------------------------------------------------------------------------------------------------- */
PetscErrorCode VecCreateSeqWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, const PetscScalar *a, Vec *v)
{
  (void)bs;
  PetscCall(PetscNew(v));
  (*v)->hdr.type_name = "seq";
  (*v)->hdr.comm      = comm;
  (*v)->n             = n;
  (*v)->a             = (PetscScalar *)a;
  return 0;
}
static PetscErrorCode VecCreateOwned(PetscInt n, Vec *v)
{
  PetscCall(VecCreateSeqWithArray(PETSC_COMM_SELF, 1, n, (PetscScalar *)calloc((size_t)(n > 0 ? n : 1), sizeof(PetscScalar)), v));
  (*v)->owned = PETSC_TRUE;
  return 0;
}
PetscErrorCode VecDestroy(Vec *v)
{
  if (!*v) return 0;
  if ((*v)->owned) free((*v)->a);
  free(*v);
  *v = NULL;
  return 0;
}
PetscErrorCode VecSet(Vec v, PetscScalar a) { for (PetscInt i = 0; i < v->n; i++) v->a[i] = a; return 0; }
PetscErrorCode VecGetSize(Vec v, PetscInt *N) { *N = v->n; return 0; }
PetscErrorCode VecGetLocalSize(Vec v, PetscInt *n) { *n = v->n; return 0; }
PetscErrorCode VecGetArray(Vec v, PetscScalar **a) { *a = v->a; return 0; }
PetscErrorCode VecRestoreArray(Vec v, PetscScalar **a) { (void)v; *a = NULL; return 0; }
PetscErrorCode VecGetArrayRead(Vec v, const PetscScalar **a) { *a = v->a; return 0; }
PetscErrorCode VecRestoreArrayRead(Vec v, const PetscScalar **a) { (void)v; *a = NULL; return 0; }

/* ---- Mat ---------------------------------------------------------------------------------------------------------------------------- */
PetscErrorCode MatCreateSeqAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt *i, PetscInt *j, PetscScalar *a, Mat *A)
{
  PetscCall(PetscNew(A));
  (*A)->hdr.type_name = MATSEQAIJ;
  (*A)->hdr.comm      = comm;
  (*A)->m = m; (*A)->n = n; (*A)->ia = i; (*A)->ja = j; (*A)->a = a;
  return 0;
}
PetscErrorCode MatCreateOneRow(Vec a, Mat *A)
{   /* src/mat/impls/onerow/onerow.c:97-113 */
  PetscCall(PetscNew(A));
  (*A)->hdr.type_name = MATONEROW;
  (*A)->hdr.comm      = a->hdr.comm;
  (*A)->m = 1; (*A)->n = a->n; (*A)->row = a;
  return 0;
}
PetscErrorCode MatCreateSeqDense(MPI_Comm comm, PetscInt m, PetscInt n, PetscScalar *data, Mat *A)
{   /* column-major, entry (i, j) at data[i + j * lda], lda = m until MatDenseSetLDA (the user's array; no allocation by the mock) */
  PetscCall(PetscNew(A));
  (*A)->hdr.type_name = MATSEQDENSE;
  (*A)->hdr.comm      = comm;
  (*A)->m = m; (*A)->n = n; (*A)->a = data; (*A)->lda = m > 0 ? m : 1;
  return 0;
}
PetscErrorCode MatDenseSetLDA(Mat A, PetscInt lda)
{
  PetscCheck(lda >= A->m, PETSC_COMM_SELF, PETSC_ERR_SUP, "lda %d < %d rows", (int)lda, (int)A->m);
  A->lda = lda;
  return 0;
}
PetscErrorCode MatDenseGetLDA(Mat A, PetscInt *lda) { *lda = A->lda; return 0; }
PetscErrorCode MatDenseGetArrayRead(Mat A, const PetscScalar **a) { *a = A->a; return 0; }
PetscErrorCode MatDenseRestoreArrayRead(Mat A, const PetscScalar **a) { (void)A; *a = NULL; return 0; }
PetscErrorCode MatDestroy(Mat *A) { free(*A); *A = NULL; return 0; }
PetscErrorCode MatGetSize(Mat A, PetscInt *M, PetscInt *N) { *M = A->m; *N = A->n; return 0; }
PetscErrorCode MatGetLocalSize(Mat A, PetscInt *m, PetscInt *n) { *m = A->m; *n = A->n; return 0; }
PetscErrorCode MatMPIAIJGetLocalMat(Mat A, MatReuse scall, Mat *Aloc)
{
  (void)scall;
  return MatCreateSeqAIJWithArrays(A->hdr.comm, A->m, A->n, A->ia, A->ja, A->a, Aloc);
}
PetscErrorCode MatGetRowIJ(Mat A, PetscInt shift, PetscBool symmetric, PetscBool inodecompressed, PetscInt *n, const PetscInt **ia, const PetscInt **ja, PetscBool *done)
{
  (void)shift; (void)symmetric; (void)inodecompressed;
  *n = A->m; *ia = A->ia; *ja = A->ja; *done = A->ia ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode MatRestoreRowIJ(Mat A, PetscInt shift, PetscBool symmetric, PetscBool inodecompressed, PetscInt *n, const PetscInt **ia, const PetscInt **ja, PetscBool *done)
{
  (void)A; (void)shift; (void)symmetric; (void)inodecompressed; (void)n;
  *ia = *ja = NULL; *done = PETSC_TRUE;
  return 0;
}
PetscErrorCode MatSeqAIJGetArrayRead(Mat A, const PetscScalar **a) { *a = A->a; return 0; }
PetscErrorCode MatSeqAIJRestoreArrayRead(Mat A, const PetscScalar **a) { (void)A; *a = NULL; return 0; }
PetscErrorCode MatCreateVecs(Mat A, Vec *right, Vec *left)
{
  if (right) PetscCall(VecCreateOwned(A->n, right));
  if (left) PetscCall(VecCreateOwned(A->m, left));
  return 0;
}
PetscErrorCode MatMultTranspose(Mat A, Vec x, Vec y)
{
  if (A->row) {   /* onerow.c:41-50: y = a * x_0 */
    for (PetscInt i = 0; i < A->n; i++) y->a[i] = A->row->a[i] * x->a[0];
    return 0;
  }
  for (PetscInt i = 0; i < A->n; i++) y->a[i] = 0.0;
  for (PetscInt r = 0; r < A->m; r++)
    for (PetscInt k = A->ia[r]; k < A->ia[r + 1]; k++) y->a[A->ja[k]] += A->a[k] * x->a[r];
  return 0;
}

/* ---- QP container (src/qp/interface/qp.c: setters take what the user passes, getters return borrowed pointers) -------------------------- */
PetscErrorCode QPCreate(MPI_Comm comm, QP *qp)
{
  PetscCall(PetscNew(qp));
  (*qp)->hdr.type_name = "qp";
  (*qp)->hdr.comm      = comm;
  return 0;
}
PetscErrorCode QPDestroy(QP *qp)
{
  if (!*qp) return 0;
  free((*qp)->qpc);
  free(*qp);
  *qp = NULL;
  return 0;
}
PetscErrorCode QPSetOperator(QP qp, Mat A) { qp->A = A; return 0; }
PetscErrorCode QPSetRhs(QP qp, Vec b) { qp->b = b; return 0; }
PetscErrorCode QPSetInitialVector(QP qp, Vec x) { qp->x = x; return 0; }
PetscErrorCode QPSetBox(QP qp, IS is, Vec lb, Vec ub)
{
  (void)is;
  free(qp->qpc);
  qp->qpc = NULL;
  if (lb || ub) {
    PetscCall(PetscNew(&qp->qpc));
    qp->qpc->hdr.type_name = QPCBOX;
    qp->qpc->lb = lb; qp->qpc->ub = ub;
  }
  return 0;
}
PetscErrorCode QPSetEq(QP qp, Mat BE, Vec cE) { qp->BE = BE; qp->cE = cE; return 0; }
PetscErrorCode QPGetOperator(QP qp, Mat *A) { *A = qp->A; return 0; }
PetscErrorCode QPGetRhs(QP qp, Vec *b) { *b = qp->b; return 0; }
PetscErrorCode QPGetSolutionVector(QP qp, Vec *x) { *x = qp->x; return 0; }
PetscErrorCode QPGetBox(QP qp, IS *is, Vec *lb, Vec *ub)
{
  if (is) *is = NULL;
  if (lb) *lb = qp->qpc ? qp->qpc->lb : NULL;
  if (ub) *ub = qp->qpc ? qp->qpc->ub : NULL;
  return 0;
}
PetscErrorCode QPGetEq(QP qp, Mat *BE, Vec *cE) { if (BE) *BE = qp->BE; if (cE) *cE = qp->cE; return 0; }
PetscErrorCode QPGetIneq(QP qp, Mat *BI, Vec *cI) { (void)qp; if (BI) *BI = NULL; if (cI) *cI = NULL; return 0; }
PetscErrorCode QPGetQPC(QP qp, QPC *qpc) { *qpc = qp->qpc; return 0; }

/* ---- QPS front end ------------------------------------------------------------------------------------------------------------------ */
static struct { const char *name; PetscErrorCode (*create)(QPS); } g_types[16];
static int g_ntypes;
PetscErrorCode QPSRegister(const char sname[], PetscErrorCode (*function)(QPS))
{   /* qpsregis.c:29-36: a later registration of the same name overrides the earlier one (PetscFunctionListAdd) */
  for (int k = 0; k < g_ntypes; k++)
    if (!strcmp(g_types[k].name, sname)) { g_types[k].create = function; return 0; }
  PetscCheck(g_ntypes < 16, PETSC_COMM_SELF, PETSC_ERR_SUP, "too many QPS types");
  g_types[g_ntypes].name = sname; g_types[g_ntypes].create = function; g_ntypes++;
  return 0;
}
PetscErrorCode QPSCreate(MPI_Comm comm, QPS *qps)
{   /* qps.c:61-100: defaults qps.c:73-76 */
  PetscCall(PetscNew(qps));
  (*qps)->hdr.comm = comm;
  (*qps)->rtol = 1e-5; (*qps)->atol = 1e-50; (*qps)->divtol = 1e4; (*qps)->max_it = 10000;
  return 0;
}
PetscErrorCode QPSDestroy(QPS *qps)
{
  if (!*qps) return 0;
  if ((*qps)->ops->destroy) PetscCall((*qps)->ops->destroy(*qps));
  free(*qps);
  *qps = NULL;
  return 0;
}
PetscErrorCode QPSSetType(QPS qps, const char *type)
{   /* qps.c:379-406 */
  for (int k = 0; k < g_ntypes; k++)
    if (!strcmp(g_types[k].name, type)) {
      if (qps->ops->destroy) PetscCall(qps->ops->destroy(qps));
      memset(qps->ops, 0, sizeof(struct _QPSOps));
      qps->setupcalled   = PETSC_FALSE;
      qps->hdr.type_name = g_types[k].name;
      return g_types[k].create(qps);
    }
  PetscCheck(0, PETSC_COMM_SELF, PETSC_ERR_ARG_UNKNOWN_TYPE, "Unable to find requested QPS type %s", type);
  return 0;
}
PetscErrorCode QPSSetQP(QPS qps, QP qp) { qps->topQP = qps->solQP = qp; qps->setupcalled = PETSC_FALSE; return 0; }
PetscErrorCode QPSSetTolerances(QPS qps, PetscReal rtol, PetscReal atol, PetscReal dtol, PetscInt maxits)
{
  qps->rtol = rtol; qps->atol = atol; qps->divtol = dtol; qps->max_it = maxits;
  return 0;
}
PetscErrorCode QPSSetUp(QPS qps)
{   /* qps.c:198-221 */
  PetscBool flg = PETSC_TRUE;
  if (qps->setupcalled) return 0;
  PetscCheck(qps->ops->setup, PETSC_COMM_SELF, PETSC_ERR_SUP, "QPS type not set");
  if (qps->ops->isqpcompatible) PetscCall(qps->ops->isqpcompatible(qps, qps->solQP, &flg));
  PetscCheck(flg, PETSC_COMM_SELF, PETSC_ERR_SUP, "QPS solver %s is not compatible with its attached QP", qps->hdr.type_name);
  PetscCall(qps->ops->setup(qps));
  qps->setupcalled = PETSC_TRUE;
  return 0;
}
PetscErrorCode QPSSolve(QPS qps)
{   /* qps.c:537-555 */
  PetscCall(QPSSetUp(qps));
  PetscCall(qps->ops->solve(qps));
  qps->iterations_accumulated += qps->iteration;
  qps->nsolves++;
  return 0;
}
PetscErrorCode QPSViewConvergence(QPS qps, PetscViewer v)
{   /* qps.c:968-1000: the type-specific part comes from _QPSOps::viewconvergence */
  if (qps->ops->viewconvergence) PetscCall(qps->ops->viewconvergence(qps, v));
  return 0;
}
