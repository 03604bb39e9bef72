/* permon_mock.h -- TEST INFRASTRUCTURE: the smallest stand-in for the PETSc / PERMON headers that adapters/qpsb200.c touches, so that the
 * adapter compiles and RUNS in this repository, where PETSc does not exist.  Shapes follow the reference (include/permon/private/
 * qpsimpl.h:12-71 for _QPSOps / _p_QPS; petscsys.h conventions for PetscCall / PetscCheck / PetscObject).  Sequential only (one rank);
 * Mat = host CSR or a column-major dense array (MATSEQDENSE), Vec = host array.  Not part of the product: libpermon_b200.so never sees this file. */
#ifndef PERMON_MOCK_H
#define PERMON_MOCK_H
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

typedef int    PetscErrorCode;
typedef int    PetscInt;
typedef int    PetscMPIInt;
typedef double PetscReal;
typedef double PetscScalar;
typedef long   PetscObjectState;
typedef enum { PETSC_FALSE, PETSC_TRUE } PetscBool;
typedef int MPI_Comm;
typedef int MPI_Datatype;
typedef void *PetscOptionItems;
typedef enum {
  KSP_CONVERGED_ITERATING = 0, KSP_CONVERGED_RTOL = 2, KSP_CONVERGED_ATOL = 3, KSP_CONVERGED_ITS = 4, KSP_CONVERGED_HAPPY_BREAKDOWN = 7,
  KSP_DIVERGED_ITS = -3, KSP_DIVERGED_DTOL = -4, KSP_DIVERGED_BREAKDOWN = -5, KSP_DIVERGED_NANORINF = -9
} KSPConvergedReason;
typedef enum { MAT_INITIAL_MATRIX, MAT_REUSE_MATRIX } MatReuse;

#define PETSC_SUCCESS 0
#define PETSC_ERR_SUP 56
#define PETSC_ERR_LIB 76
#define PETSC_ERR_FILE_OPEN 65
#define PETSC_ERR_ARG_UNKNOWN_TYPE 86
#define PETSC_COMM_WORLD 1
#define PETSC_COMM_SELF 2
#define MPI_BYTE 1
#define PetscInt_FMT "d"
#define PERMON_EXTERN extern
#define MATSEQAIJ "seqaij"
#define MATSEQDENSE "seqdense"
#define MATONEROW "onerow"
#define QPCBOX "box"
#define QPSMPGP "mpgp"
#define QPSSMALXE "smalxe"

#define PetscFunctionBegin
#define PetscFunctionReturn(v) return (v)
#define PetscCall(call)                              \
  do {                                               \
    PetscErrorCode ierr_mock_ = (call);              \
    if (ierr_mock_) return ierr_mock_;               \
  } while (0)
#define PetscCallMPI(call) PetscCall(call)
#define PetscCheck(cond, comm, code, ...)                                  \
  do {                                                                     \
    if (!(cond)) {                                                         \
      fprintf(stderr, "[mock PETSc] error %d at %s:%d: ", (int)(code), __FILE__, __LINE__); \
      fprintf(stderr, __VA_ARGS__);                                        \
      fprintf(stderr, "\n");                                               \
      return (code);                                                       \
    }                                                                      \
  } while (0)
#define PetscNew(p) ((*(p) = calloc(1, sizeof(**(p)))) ? 0 : 55)
#define PetscFree(p) (free(p), (p) = NULL, 0)

static inline int MPI_Comm_size(MPI_Comm c, int *s) { (void)c; *s = 1; return 0; }
static inline int MPI_Comm_rank(MPI_Comm c, int *r) { (void)c; *r = 0; return 0; }
static inline int MPI_Bcast(void *b, int n, MPI_Datatype t, int root, MPI_Comm c) { (void)b; (void)n; (void)t; (void)root; (void)c; return 0; }

/* ---- objects --------------------------------------------------------------------------------------------------------------- */
struct _p_PetscObject {
  const char      *type_name;
  const char      *prefix;
  MPI_Comm         comm;
  PetscObjectState state;
};
typedef struct _p_PetscObject *PetscObject;
#define PETSCHEADER(OpsType) \
  struct _p_PetscObject hdr; \
  OpsType               ops[1]

typedef struct _p_Vec *Vec;
typedef struct _p_Mat *Mat;
typedef struct _p_IS  *IS;
typedef struct _p_QPC *QPC;
typedef struct _p_QP  *QP;
typedef struct _p_QPS *QPS;
typedef struct _p_PetscViewer *PetscViewer;
struct _p_PetscViewer { struct _p_PetscObject hdr; FILE *f; };
struct _p_Vec { struct _p_PetscObject hdr; PetscInt n; PetscScalar *a; PetscBool owned; };
struct _p_Mat { struct _p_PetscObject hdr; PetscInt m, n; PetscInt *ia, *ja; PetscScalar *a; Vec row; /* MATONEROW */ PetscInt lda; /* MATSEQDENSE */ };
struct _p_QPC { struct _p_PetscObject hdr; Vec lb, ub; };
struct _p_QP  { struct _p_PetscObject hdr; Mat A, BE; Vec b, x, cE; QPC qpc; };

/* include/permon/private/qpsimpl.h:12-24 */
struct _QPSOps {
  PetscErrorCode (*solve)(QPS);
  PetscErrorCode (*setup)(QPS);
  PetscErrorCode (*destroy)(QPS);
  PetscErrorCode (*view)(QPS, PetscViewer);
  PetscErrorCode (*viewconvergence)(QPS, PetscViewer);
  PetscErrorCode (*setfromoptions)(QPS, PetscOptionItems);
  PetscErrorCode (*reset)(QPS);
  PetscErrorCode (*resetstatistics)(QPS);
  PetscErrorCode (*isqpcompatible)(QPS, QP, PetscBool *);
  PetscErrorCode (*monitor)(QPS, PetscInt, PetscViewer);
  PetscErrorCode (*monitorcostfunction)(QPS, PetscInt, PetscViewer);
};
/* include/permon/private/qpsimpl.h:26-71 (the fields a solver implementation reads or writes) */
struct _p_QPS {
  PETSCHEADER(struct _QPSOps);
  QP                 topQP, solQP;
  PetscReal          rtol, atol, divtol;
  PetscInt           max_it;
  PetscBool          autoPostSolve, user_type;
  void              *data;
  PetscReal          rnorm;
  PetscInt           iteration, iterations_accumulated, nsolves;
  PetscBool          setupcalled, postsolvecalled;
  KSPConvergedReason reason;
};

/* ---- the PETSc / PERMON calls the adapter makes ---------------------------------------------------------------------------------- */
MPI_Comm       PetscObjectComm(PetscObject o);
PetscErrorCode PetscObjectTypeCompare(PetscObject o, const char *type, PetscBool *same);
PetscErrorCode PetscObjectGetOptionsPrefix(PetscObject o, const char **prefix);
PetscErrorCode PetscObjectStateIncrease(PetscObject o);
PetscErrorCode PetscOptionsGetAll(void *options, char **copts);
PetscErrorCode PetscOptionsSetValue(void *options, const char *name, const char *value);
PetscErrorCode PetscViewerASCIIPrintf(PetscViewer v, const char *fmt, ...);

PetscErrorCode MatCreateSeqAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt *i, PetscInt *j, PetscScalar *a, Mat *A);
PetscErrorCode MatCreateOneRow(Vec a, Mat *A);
PetscErrorCode MatCreateSeqDense(MPI_Comm comm, PetscInt m, PetscInt n, PetscScalar *data, Mat *A);
PetscErrorCode MatDenseSetLDA(Mat A, PetscInt lda);
PetscErrorCode MatDenseGetLDA(Mat A, PetscInt *lda);
PetscErrorCode MatDenseGetArrayRead(Mat A, const PetscScalar **a);
PetscErrorCode MatDenseRestoreArrayRead(Mat A, const PetscScalar **a);
PetscErrorCode MatDestroy(Mat *A);
PetscErrorCode MatGetSize(Mat A, PetscInt *M, PetscInt *N);
PetscErrorCode MatGetLocalSize(Mat A, PetscInt *m, PetscInt *n);
PetscErrorCode MatMPIAIJGetLocalMat(Mat A, MatReuse scall, Mat *Aloc);
PetscErrorCode MatGetRowIJ(Mat A, PetscInt shift, PetscBool symmetric, PetscBool inodecompressed, PetscInt *n, const PetscInt **ia, const PetscInt **ja, PetscBool *done);
PetscErrorCode MatRestoreRowIJ(Mat A, PetscInt shift, PetscBool symmetric, PetscBool inodecompressed, PetscInt *n, const PetscInt **ia, const PetscInt **ja, PetscBool *done);
PetscErrorCode MatSeqAIJGetArrayRead(Mat A, const PetscScalar **a);
PetscErrorCode MatSeqAIJRestoreArrayRead(Mat A, const PetscScalar **a);
PetscErrorCode MatCreateVecs(Mat A, Vec *right, Vec *left);
PetscErrorCode MatMultTranspose(Mat A, Vec x, Vec y);

PetscErrorCode VecCreateSeqWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, const PetscScalar *a, Vec *v);
PetscErrorCode VecDestroy(Vec *v);
PetscErrorCode VecSet(Vec v, PetscScalar a);
PetscErrorCode VecGetSize(Vec v, PetscInt *N);
PetscErrorCode VecGetLocalSize(Vec v, PetscInt *n);
PetscErrorCode VecGetArray(Vec v, PetscScalar **a);
PetscErrorCode VecRestoreArray(Vec v, PetscScalar **a);
PetscErrorCode VecGetArrayRead(Vec v, const PetscScalar **a);
PetscErrorCode VecRestoreArrayRead(Vec v, const PetscScalar **a);

PetscErrorCode QPCreate(MPI_Comm comm, QP *qp);
PetscErrorCode QPDestroy(QP *qp);
PetscErrorCode QPSetOperator(QP qp, Mat A);
PetscErrorCode QPSetRhs(QP qp, Vec b);
PetscErrorCode QPSetInitialVector(QP qp, Vec x);
PetscErrorCode QPSetBox(QP qp, IS is, Vec lb, Vec ub);
PetscErrorCode QPSetEq(QP qp, Mat BE, Vec cE);
PetscErrorCode QPGetOperator(QP qp, Mat *A);
PetscErrorCode QPGetRhs(QP qp, Vec *b);
PetscErrorCode QPGetSolutionVector(QP qp, Vec *x);
PetscErrorCode QPGetBox(QP qp, IS *is, Vec *lb, Vec *ub);
PetscErrorCode QPGetEq(QP qp, Mat *BE, Vec *cE);
PetscErrorCode QPGetIneq(QP qp, Mat *BI, Vec *cI);
PetscErrorCode QPGetQPC(QP qp, QPC *qpc);

/* src/qps/interface/qpsregis.c:29-36, qps.c:61-100, :379-406, :198-221, :537-555, :968-1000 */
PetscErrorCode QPSRegister(const char sname[], PetscErrorCode (*function)(QPS));
PetscErrorCode QPSCreate(MPI_Comm comm, QPS *qps);
PetscErrorCode QPSDestroy(QPS *qps);
PetscErrorCode QPSSetType(QPS qps, const char *type);
PetscErrorCode QPSSetQP(QPS qps, QP qp);
PetscErrorCode QPSSetTolerances(QPS qps, PetscReal rtol, PetscReal atol, PetscReal dtol, PetscInt maxits);
PetscErrorCode QPSSetUp(QPS qps);
PetscErrorCode QPSSolve(QPS qps);
PetscErrorCode QPSViewConvergence(QPS qps, PetscViewer v);
extern struct _p_PetscViewer PETSC_VIEWER_STDOUT_WORLD_OBJ;
#define PETSC_VIEWER_STDOUT_WORLD (&PETSC_VIEWER_STDOUT_WORLD_OBJ)
#endif
