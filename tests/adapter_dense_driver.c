/* TEST INFRASTRUCTURE: "PERMON user code" on the mock PETSc (adapters/mock) whose Hessian is a MATSEQDENSE matrix, solved through
 * adapters/qpsb200.c.  The matrix is column-major with a leading dimension lda >= n (MatCreateSeqDense + MatDenseSetLDA), as a PETSc
 * user would hold it.  usage: adapter_dense_driver problem.bin x_out.bin type
 * problem.bin: int32 n, lda, has_lb; fp64 a[lda * n] (column-major), b[n], x0[n], [lb[n]] */
#include "../adapters/mock/permon_mock.h"

PetscErrorCode PermonB200RegisterQPS(void);

static void *rd(FILE *f, size_t bytes)
{
  void *p = malloc(bytes ? bytes : 1);
  if (bytes && fread(p, 1, bytes, f) != bytes) exit(3);
  return p;
}

int main(int argc, char **argv)
{
  if (argc < 4) return 2;
  FILE *f = fopen(argv[1], "rb");
  if (!f) return 2;
  int hdr[3];   /* n, lda, has_lb */
  if (fread(hdr, sizeof(int), 3, f) != 3) return 3;
  const int n = hdr[0], lda = hdr[1];
  double   *a = rd(f, 8 * (size_t)lda * (size_t)n), *b = rd(f, 8 * (size_t)n), *x = rd(f, 8 * (size_t)n);
  double   *lb = hdr[2] ? rd(f, 8 * (size_t)n) : NULL;
  fclose(f);

  Mat A;
  Vec vb, vx, vlb = NULL;
  QP  qp;
  QPS qps;
  PetscCall(PermonB200RegisterQPS());
  PetscCall(MatCreateSeqDense(PETSC_COMM_WORLD, n, n, a, &A));
  if (lda != n) PetscCall(MatDenseSetLDA(A, lda));
  printf("user MatCreateSeqDense n %d lda %d data %p\n", n, lda, (void *)a);
  PetscCall(VecCreateSeqWithArray(PETSC_COMM_WORLD, 1, n, b, &vb));
  PetscCall(VecCreateSeqWithArray(PETSC_COMM_WORLD, 1, n, x, &vx));
  if (lb) PetscCall(VecCreateSeqWithArray(PETSC_COMM_WORLD, 1, n, lb, &vlb));
  PetscCall(QPCreate(PETSC_COMM_WORLD, &qp));
  PetscCall(QPSetOperator(qp, A));
  PetscCall(QPSetRhs(qp, vb));
  PetscCall(QPSetInitialVector(qp, vx));
  PetscCall(QPSetBox(qp, NULL, vlb, NULL));
  PetscCall(QPSCreate(PETSC_COMM_WORLD, &qps));
  PetscCall(QPSSetType(qps, argv[3]));
  PetscCall(QPSSetQP(qps, qp));
  PetscCall(QPSSolve(qps));
  printf("reason %d iterations %d rnorm %.10e\n", (int)qps->reason, (int)qps->iteration, (double)qps->rnorm);
  PetscCall(QPSViewConvergence(qps, PETSC_VIEWER_STDOUT_WORLD));
  f = fopen(argv[2], "wb");
  if (!f || fwrite(x, 8, (size_t)n, f) != (size_t)n) return 4;
  fclose(f);
  PetscCall(QPSDestroy(&qps));
  PetscCall(QPDestroy(&qp));
  PetscCall(MatDestroy(&A));
  PetscCall(VecDestroy(&vb)); PetscCall(VecDestroy(&vx)); PetscCall(VecDestroy(&vlb));
  free(a); free(b); free(x); free(lb);
  return 0;
}
