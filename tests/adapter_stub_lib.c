/* TEST INFRASTRUCTURE: a stand-in for libpermon_b200.so with the slice of the C ABI that adapters/qpsb200.c binds.  Every call succeeds
 * and does nothing, except that the matrix constructors report on stdout what the adapter handed over, so that the adapter's upload
 * routes can be checked on a machine without a GPU (tests/test_adapter_dense.py).  Loaded through PERMON_B200_LIBRARY. */
#include <stdio.h>

typedef int b200_int;
static int   g_handle_store[64];
static int   g_next;
void        *PETSC_COMM_WORLD = &g_handle_store[63];

static void *handle(void) { return &g_handle_store[g_next++ % 62]; }
#define NEW(out) (*(out) = handle(), 0)

int         PermonInitialize(int *argc, char ***args, const char *file, const char *help) { (void)argc; (void)args; (void)file; (void)help; return 0; }
int         PermonB200GetUniqueId(void *id) { (void)id; return 0; }
int         PermonB200CommInitRank(int n, int r, const void *id) { (void)n; (void)r; (void)id; return 0; }
const char *PermonB200GetLastErrorMessage(void) { return ""; }
int         PetscOptionsInsertString(void *o, const char *s) { (void)o; (void)s; return 0; }
int MatCreateMPIAIJWithArrays(void *c, b200_int m, b200_int n, b200_int M, b200_int N, const b200_int *i, const b200_int *j, const double *a, void **A)
{
  (void)c; (void)i; (void)j;
  *A = handle();
  printf("stub MatCreateMPIAIJWithArrays m %d n %d M %d N %d values %p handle %p\n", m, n, M, N, (const void *)a, *A);
  return 0;
}
int MatCreateSeqDense(void *c, b200_int m, b200_int n, double *data, void **A)
{
  (void)c;
  *A = handle();
  printf("stub MatCreateSeqDense m %d n %d data %p handle %p\n", m, n, (void *)data, *A);
  return 0;
}
int MatDenseSetLDA(void *A, b200_int lda)
{
  printf("stub MatDenseSetLDA lda %d handle %p\n", lda, A);
  return 0;
}
int MatCreateOneRow(void *row, void **A) { (void)row; return NEW(A); }
int MatDestroy(void **A) { *A = 0; return 0; }
int VecCreateMPIWithArray(void *c, b200_int bs, b200_int n, b200_int N, const double *a, void **v) { (void)c; (void)bs; (void)n; (void)N; (void)a; return NEW(v); }
int VecGetArrayRead(void *v, const double **a) { (void)v; *a = 0; return 0; }
int VecRestoreArrayRead(void *v, const double **a) { (void)v; *a = 0; return 0; }
int VecDestroy(void **v) { *v = 0; return 0; }
int QPCreate(void *c, void **qp) { (void)c; return NEW(qp); }
int QPDestroy(void **qp) { *qp = 0; return 0; }
int QPSetOperator(void *qp, void *A) { (void)qp; (void)A; return 0; }
int QPSetRhs(void *qp, void *b) { (void)qp; (void)b; return 0; }
int QPSetInitialVector(void *qp, void *x) { (void)qp; (void)x; return 0; }
int QPSetBox(void *qp, void *is, void *lb, void *ub) { (void)qp; (void)is; (void)lb; (void)ub; return 0; }
int QPSetEq(void *qp, void *B, void *c) { (void)qp; (void)B; (void)c; return 0; }
int QPSCreate(void *c, void **q) { (void)c; return NEW(q); }
int QPSDestroy(void **q) { *q = 0; return 0; }
int QPSSetType(void *q, const char *t) { (void)q; (void)t; return 0; }
int QPSSetQP(void *q, void *qp) { (void)q; (void)qp; return 0; }
int QPSSetTolerances(void *q, double r, double a, double d, b200_int m) { (void)q; (void)r; (void)a; (void)d; (void)m; return 0; }
int QPSSetOptionsPrefix(void *q, const char *p) { (void)q; (void)p; return 0; }
int QPSSetFromOptions(void *q) { (void)q; return 0; }
int QPSSetAutoPostSolve(void *q, int f) { (void)q; (void)f; return 0; }
int QPSSetUp(void *q) { (void)q; return 0; }
int QPSSolve(void *q) { (void)q; return 0; }
int QPSReset(void *q) { (void)q; return 0; }
int QPSResetStatistics(void *q) { (void)q; return 0; }
int QPSGetIterationNumber(void *q, b200_int *i) { (void)q; *i = 0; return 0; }
int QPSGetConvergedReason(void *q, int *r) { (void)q; *r = 2; return 0; }
int QPSGetResidualNorm(void *q, double *r) { (void)q; *r = 0.0; return 0; }
int QPSViewConvergence(void *q, void *v) { (void)q; (void)v; return 0; }
int QPSMonitorDefault(void *q, b200_int n, double r, void *v) { (void)q; (void)n; (void)r; (void)v; return 0; }
int PetscViewerASCIIOpen(void *c, const char *name, void **v) { (void)c; (void)name; return NEW(v); }
int PetscViewerDestroy(void **v) { *v = 0; return 0; }
