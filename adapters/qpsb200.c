/* qpsb200.c -- PERMON plug-in that runs QPSMPGP / QPSSMALXE on libpermon_b200.so (SURVEY.md 8f rank 1: the PETSc upload adapter).
 *
 * Where it goes in a PERMON + PETSc build:  src/qps/impls/b200/qpsb200.c, compiled with -DPERMON_B200_HAVE_PETSC, and
 *     PermonB200RegisterQPS();                      // once after PermonInitialize(): QPSRegister("mpgp" | "smalxe", ...) override
 * or, as a dynamic plug-in, PetscDLLibraryRegister_permonb200() (the pattern of src/sys/permoninit.c:125-131).
 *
 * What it replaces (reference file:line):
 *   QPSRegister / QPSRegisterAll           src/qps/interface/qpsregis.c:17-36
 *   struct _QPSOps, struct _p_QPS          include/permon/private/qpsimpl.h:12-71   (every slot of the vtable is filled below)
 *   QPSCreate_MPGP / QPSCreate_SMALXE      src/qps/impls/mpgp/mpgp.c:819-869, src/qps/impls/smalxe/smalxe.c:1143-1207
 *   Mat_MPIAIJ row-partitioned layout      include/permon/private/petsc/mpiaij.h:49-83 (read through MatMPIAIJGetLocalMat)
 *   MATSEQDENSE Hessians                   column-major host array + leading dimension (MatDenseGetArrayRead, MatDenseGetLDA)
 *
 * The adapter is thin on purpose: it reads the PETSc objects of the QP (host CSR of the local rows with GLOBAL column indices, host
 * arrays of the vectors), hands them to the C ABI of libpermon_b200.so (include/permon_b200.h) -- "uploaded once" -- and lets the whole
 * iteration run on the device; the user's x Vec is the solution storage on both sides (src/qp/interface/qp.c:1987-1991).
 * libpermon_b200.so deliberately exports PERMON's own names (QPCreate, QPSSolve, ...), so it is loaded with dlopen(RTLD_LOCAL) and
 * reached through dlsym: no symbol of it is visible to the PERMON build.
 *
 * Without PETSc (this repository) the file compiles against adapters/mock/ (-DPERMON_B200_MOCK_PETSC), a minimal stand-in for the PETSc /
 * PERMON headers the adapter touches, and tests/test_adapter.py runs the reference's ex1 tutorial through it on the GPU.
 */
#if defined(PERMON_B200_HAVE_PETSC)
  #include <permon/private/qpsimpl.h>
  #include <permonqps.h>
#elif defined(PERMON_B200_MOCK_PETSC)
  #include "mock/permon_mock.h"
#endif

#if defined(PERMON_B200_HAVE_PETSC) || defined(PERMON_B200_MOCK_PETSC)
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

/* ---- the slice of libpermon_b200.so's C ABI the adapter binds (include/permon_b200.h; ints are PetscErrorCode) -------------------- */
typedef int b200_int; /* PetscInt of the B200 build: int32 */
typedef struct {
  void *lib;
  void **comm_world;
  int (*PermonInitialize)(int *, char ***, const char *, const char *);
  int (*PermonB200GetUniqueId)(void *);
  int (*PermonB200CommInitRank)(int, int, const void *);
  const char *(*PermonB200GetLastErrorMessage)(void);
  int (*PetscOptionsInsertString)(void *, const char *);
  int (*MatCreateMPIAIJWithArrays)(void *, b200_int, b200_int, b200_int, b200_int, const b200_int *, const b200_int *, const double *, void **);
  int (*MatCreateOneRow)(void *, void **);
  int (*MatCreateSeqDense)(void *, b200_int, b200_int, double *, void **);
  int (*MatDenseSetLDA)(void *, b200_int);
  int (*MatDestroy)(void **);
  int (*VecCreateMPIWithArray)(void *, b200_int, b200_int, b200_int, const double *, void **);
  int (*VecGetArrayRead)(void *, const double **);
  int (*VecRestoreArrayRead)(void *, const double **);
  int (*VecDestroy)(void **);
  int (*QPCreate)(void *, void **);
  int (*QPDestroy)(void **);
  int (*QPSetOperator)(void *, void *);
  int (*QPSetRhs)(void *, void *);
  int (*QPSetInitialVector)(void *, void *);
  int (*QPSetBox)(void *, void *, void *, void *);
  int (*QPSetEq)(void *, void *, void *);
  int (*QPSCreate)(void *, void **);
  int (*QPSDestroy)(void **);
  int (*QPSSetType)(void *, const char *);
  int (*QPSSetQP)(void *, void *);
  int (*QPSSetTolerances)(void *, double, double, double, b200_int);
  int (*QPSSetOptionsPrefix)(void *, const char *);
  int (*QPSSetFromOptions)(void *);
  int (*QPSSetAutoPostSolve)(void *, int);
  int (*QPSSetUp)(void *);
  int (*QPSSolve)(void *);
  int (*QPSReset)(void *);
  int (*QPSResetStatistics)(void *);
  int (*QPSGetIterationNumber)(void *, b200_int *);
  int (*QPSGetConvergedReason)(void *, int *);
  int (*QPSGetResidualNorm)(void *, double *);
  int (*QPSViewConvergence)(void *, void *);
  int (*QPSMonitorDefault)(void *, b200_int, double, void *);
  int (*PetscViewerASCIIOpen)(void *, const char *, void **);
  int (*PetscViewerDestroy)(void **);
} B200Api;

static B200Api g_b200;

#define B200_BIND(name)                                                                                                              \
  do {                                                                                                                               \
    *(void **)(&g_b200.name) = dlsym(g_b200.lib, #name);                                                                             \
    PetscCheck(g_b200.name, PETSC_COMM_SELF, PETSC_ERR_LIB, "libpermon_b200.so does not export %s", #name);                          \
  } while (0)
#define B200_CALL(call)                                                                                                              \
  do {                                                                                                                               \
    int b200_ierr_ = (call);                                                                                                         \
    PetscCheck(!b200_ierr_, PETSC_COMM_SELF, PETSC_ERR_LIB, "libpermon_b200: error %d in %s: %s", b200_ierr_, #call,                 \
               g_b200.PermonB200GetLastErrorMessage ? g_b200.PermonB200GetLastErrorMessage() : "");                                   \
  } while (0)

static PetscErrorCode B200Load(void)
{
  const char *path;

  PetscFunctionBegin;
  if (g_b200.lib) PetscFunctionReturn(PETSC_SUCCESS);
  path = getenv("PERMON_B200_LIBRARY");
  g_b200.lib = dlopen(path ? path : "libpermon_b200.so", RTLD_NOW | RTLD_LOCAL);
  PetscCheck(g_b200.lib, PETSC_COMM_SELF, PETSC_ERR_LIB, "cannot load libpermon_b200.so (set PERMON_B200_LIBRARY): %s", dlerror());
  g_b200.comm_world = (void **)dlsym(g_b200.lib, "PETSC_COMM_WORLD");
  PetscCheck(g_b200.comm_world, PETSC_COMM_SELF, PETSC_ERR_LIB, "libpermon_b200.so does not export PETSC_COMM_WORLD");
  B200_BIND(PermonInitialize); B200_BIND(PermonB200GetUniqueId); B200_BIND(PermonB200CommInitRank); B200_BIND(PermonB200GetLastErrorMessage);
  B200_BIND(PetscOptionsInsertString);
  B200_BIND(MatCreateMPIAIJWithArrays); B200_BIND(MatCreateOneRow); B200_BIND(MatCreateSeqDense); B200_BIND(MatDenseSetLDA); B200_BIND(MatDestroy);
  B200_BIND(VecCreateMPIWithArray); B200_BIND(VecGetArrayRead); B200_BIND(VecRestoreArrayRead); B200_BIND(VecDestroy);
  B200_BIND(QPCreate); B200_BIND(QPDestroy); B200_BIND(QPSetOperator); B200_BIND(QPSetRhs); B200_BIND(QPSetInitialVector); B200_BIND(QPSetBox); B200_BIND(QPSetEq);
  B200_BIND(QPSCreate); B200_BIND(QPSDestroy); B200_BIND(QPSSetType); B200_BIND(QPSSetQP); B200_BIND(QPSSetTolerances); B200_BIND(QPSSetOptionsPrefix);
  B200_BIND(QPSSetFromOptions); B200_BIND(QPSSetAutoPostSolve); B200_BIND(QPSSetUp); B200_BIND(QPSSolve); B200_BIND(QPSReset); B200_BIND(QPSResetStatistics);
  B200_BIND(QPSGetIterationNumber); B200_BIND(QPSGetConvergedReason); B200_BIND(QPSGetResidualNorm); B200_BIND(QPSViewConvergence); B200_BIND(QPSMonitorDefault);
  B200_BIND(PetscViewerASCIIOpen); B200_BIND(PetscViewerDestroy);
  B200_CALL(g_b200.PermonInitialize(NULL, NULL, NULL, NULL));
  {
    /* one process per GPU: the MPI communicator maps onto the library's NCCL communicator of the same ranks; the 128-byte id travels
       over MPI (with one rank there is nothing to do) */
    PetscMPIInt size, rank;
    char        id[128];
    PetscCallMPI(MPI_Comm_size(PETSC_COMM_WORLD, &size));
    PetscCallMPI(MPI_Comm_rank(PETSC_COMM_WORLD, &rank));
    if (size > 1) {
      memset(id, 0, sizeof id);
      if (!rank) B200_CALL(g_b200.PermonB200GetUniqueId(id));
      PetscCallMPI(MPI_Bcast(id, 128, MPI_BYTE, 0, PETSC_COMM_WORLD));
      B200_CALL(g_b200.PermonB200CommInitRank(size, rank, id));
    }
  }
  {
    /* the -qps_* / -qps_mpgp_* / -qps_smalxe_* keys live in PETSc's options database: the library reads the same keys from its own */
    char *all = NULL;
    PetscCall(PetscOptionsGetAll(NULL, &all));
    if (all && all[0]) B200_CALL(g_b200.PetscOptionsInsertString(NULL, all));
    PetscCall(PetscFree(all));
  }
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* ---- per-solver state ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  const char *type; /* "mpgp" | "smalxe" */
  void       *qp, *qps, *A, *b, *x, *lb, *ub, *BE, *BErow, *cE;
  /* PETSc side: what was borrowed in set-up and has to be given back */
  Mat                Aloc;
  PetscBool          Aloc_owned;
  const PetscInt    *ia, *ja;
  const PetscScalar *a, *pb, *plb, *pub, *pbe, *pce;
  const PetscScalar *ad; /* MATSEQDENSE Hessian: its column-major array (of Adense), borrowed until the next set-up / reset */
  Mat                Adense;
  PetscScalar       *px;
  Vec                vb, vx, vlb, vub, vbe, vce;
  PetscInt           nrows;
  b200_int          *ia32, *ja32; /* only when PetscInt is 64 bit */
} QPS_B200;

static PetscErrorCode B200ReleaseBorrowed(QPS_B200 *ctx)
{
  PetscBool done;

  PetscFunctionBegin;
  if (ctx->pb) PetscCall(VecRestoreArrayRead(ctx->vb, &ctx->pb));
  if (ctx->px) PetscCall(VecRestoreArray(ctx->vx, &ctx->px));
  if (ctx->plb) PetscCall(VecRestoreArrayRead(ctx->vlb, &ctx->plb));
  if (ctx->pub) PetscCall(VecRestoreArrayRead(ctx->vub, &ctx->pub));
  if (ctx->pbe) {
    PetscCall(VecRestoreArrayRead(ctx->vbe, &ctx->pbe));
    PetscCall(VecDestroy(&ctx->vbe));
  }
  if (ctx->pce) PetscCall(VecRestoreArrayRead(ctx->vce, &ctx->pce));
  if (ctx->a) PetscCall(MatSeqAIJRestoreArrayRead(ctx->Aloc, &ctx->a));
  if (ctx->ad) PetscCall(MatDenseRestoreArrayRead(ctx->Adense, &ctx->ad));
  if (ctx->ia) PetscCall(MatRestoreRowIJ(ctx->Aloc, 0, PETSC_FALSE, PETSC_FALSE, &ctx->nrows, &ctx->ia, &ctx->ja, &done));
  if (ctx->Aloc_owned) PetscCall(MatDestroy(&ctx->Aloc));
  free(ctx->ia32);
  free(ctx->ja32);
  ctx->pb = ctx->plb = ctx->pub = ctx->pbe = ctx->pce = NULL;
  ctx->px = NULL;
  ctx->a  = NULL;
  ctx->ad = NULL;
  ctx->Adense = NULL;
  ctx->ia = ctx->ja = NULL;
  ctx->ia32 = ctx->ja32 = NULL;
  ctx->Aloc             = NULL;
  ctx->Aloc_owned       = PETSC_FALSE;
  PetscFunctionReturn(PETSC_SUCCESS);
}

static PetscErrorCode B200DestroyDeviceSide(QPS_B200 *ctx)
{
  PetscFunctionBegin;
  if (ctx->qps) B200_CALL(g_b200.QPSDestroy(&ctx->qps));
  if (ctx->qp) B200_CALL(g_b200.QPDestroy(&ctx->qp));
  if (ctx->BE) B200_CALL(g_b200.MatDestroy(&ctx->BE));
  if (ctx->BErow) B200_CALL(g_b200.VecDestroy(&ctx->BErow));
  if (ctx->cE) B200_CALL(g_b200.VecDestroy(&ctx->cE));
  if (ctx->b) B200_CALL(g_b200.VecDestroy(&ctx->b));
  if (ctx->x) B200_CALL(g_b200.VecDestroy(&ctx->x));
  if (ctx->lb) B200_CALL(g_b200.VecDestroy(&ctx->lb));
  if (ctx->ub) B200_CALL(g_b200.VecDestroy(&ctx->ub));
  if (ctx->A) B200_CALL(g_b200.MatDestroy(&ctx->A));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::setup -- QPSSetup_MPGP mpgp.c:359-428 / QPSSetUp_SMALXE smalxe.c:772-888: here "upload once" */
static PetscErrorCode QPSSetUp_B200(QPS qps)
{
  QPS_B200   *ctx = (QPS_B200 *)qps->data;
  QP          qp  = qps->solQP;
  Mat         A, BE = NULL;
  Vec         b, x, lb = NULL, ub = NULL, cE = NULL;
  IS          is = NULL;
  PetscInt    m, n, M, N;
  PetscBool   done, isseq, isdense;
  void       *comm;
  const char *prefix = NULL;

  PetscFunctionBegin;
  PetscCall(B200Load());
  comm = *g_b200.comm_world;
  PetscCall(B200DestroyDeviceSide(ctx));
  PetscCall(B200ReleaseBorrowed(ctx));
  PetscCall(QPGetOperator(qp, &A));
  PetscCall(QPGetRhs(qp, &b));
  PetscCall(QPGetSolutionVector(qp, &x));
  PetscCall(QPGetBox(qp, &is, &lb, &ub));
  PetscCall(QPGetEq(qp, &BE, &cE));
  PetscCheck(!is, PetscObjectComm((PetscObject)qps), PETSC_ERR_SUP, "box constraints on an index subset: expand lb / ub to full length (-infinity / +infinity) first");

  PetscCall(MatGetSize(A, &M, &N));
  PetscCall(MatGetLocalSize(A, &m, &n));
  PetscCall(PetscObjectTypeCompare((PetscObject)A, MATSEQDENSE, &isdense));
  if (isdense) {
    /* dense Hessian (one rank): PETSc's column-major array (entry (i, j) at a[i + j*lda]) and its leading dimension go over as they are.
       The library copies the array to the device at the first use (QPSSetUp below); it stays borrowed until the next set-up or reset */
    PetscInt lda;
    PetscCall(MatDenseGetLDA(A, &lda));
    PetscCall(MatDenseGetArrayRead(A, &ctx->ad));
    ctx->Adense = A;
    B200_CALL(g_b200.MatCreateSeqDense(comm, (b200_int)M, (b200_int)N, (double *)ctx->ad, &ctx->A));
    if (lda != M) B200_CALL(g_b200.MatDenseSetLDA(ctx->A, (b200_int)lda));
  } else {
    /* AIJ Hessian: local rows, GLOBAL column indices (what MatCreateMPIAIJWithArrays of either side takes).  MPIAIJ keeps a diagonal and
       an off-diagonal block with compressed local columns (mpiaij.h:49-83); MatMPIAIJGetLocalMat merges them back */
    PetscCall(PetscObjectTypeCompare((PetscObject)A, MATSEQAIJ, &isseq));
    if (isseq) {
      ctx->Aloc       = A;
      ctx->Aloc_owned = PETSC_FALSE;
    } else {
      PetscCall(MatMPIAIJGetLocalMat(A, MAT_INITIAL_MATRIX, &ctx->Aloc));
      ctx->Aloc_owned = PETSC_TRUE;
    }
    PetscCall(MatGetRowIJ(ctx->Aloc, 0, PETSC_FALSE, PETSC_FALSE, &ctx->nrows, &ctx->ia, &ctx->ja, &done));
    PetscCheck(done && ctx->nrows == m, PetscObjectComm((PetscObject)qps), PETSC_ERR_SUP, "the Hessian must be an assembled (MPI)AIJ matrix");
    PetscCall(MatSeqAIJGetArrayRead(ctx->Aloc, &ctx->a));
    {
      const b200_int *ia = (const b200_int *)ctx->ia, *ja = (const b200_int *)ctx->ja;
      if (sizeof(PetscInt) != sizeof(b200_int)) { /* 64-bit-index PETSc: the device CSR is int32 */
        PetscInt k, nz = ctx->ia[m];
        PetscCheck(M < 2147483647 && nz < 2147483647, PetscObjectComm((PetscObject)qps), PETSC_ERR_SUP, "local block too large for 32-bit indices");
        ctx->ia32 = (b200_int *)malloc(sizeof(b200_int) * (size_t)(m + 1));
        ctx->ja32 = (b200_int *)malloc(sizeof(b200_int) * (size_t)(nz > 0 ? nz : 1));
        for (k = 0; k <= m; k++) ctx->ia32[k] = (b200_int)ctx->ia[k];
        for (k = 0; k < nz; k++) ctx->ja32[k] = (b200_int)ctx->ja[k];
        ia = ctx->ia32;
        ja = ctx->ja32;
      }
      B200_CALL(g_b200.MatCreateMPIAIJWithArrays(comm, (b200_int)m, (b200_int)n, (b200_int)M, (b200_int)N, ia, ja, ctx->a, &ctx->A));
    }
  }

  /* vectors: the library adopts the host arrays; x stays the solution storage */
  ctx->vb = b;
  ctx->vx = x;
  PetscCall(VecGetArrayRead(b, &ctx->pb));
  PetscCall(VecGetArray(x, &ctx->px));
  B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)m, (b200_int)M, ctx->pb, &ctx->b));
  B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)n, (b200_int)N, ctx->px, &ctx->x));
  if (lb) {
    ctx->vlb = lb;
    PetscCall(VecGetArrayRead(lb, &ctx->plb));
    B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)n, (b200_int)N, ctx->plb, &ctx->lb));
  }
  if (ub) {
    ctx->vub = ub;
    PetscCall(VecGetArrayRead(ub, &ctx->pub));
    B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)n, (b200_int)N, ctx->pub, &ctx->ub));
  }
  B200_CALL(g_b200.QPCreate(comm, &ctx->qp));
  B200_CALL(g_b200.QPSetOperator(ctx->qp, ctx->A));
  B200_CALL(g_b200.QPSetRhs(ctx->qp, ctx->b));
  B200_CALL(g_b200.QPSetInitialVector(ctx->qp, ctx->x));
  if (ctx->lb || ctx->ub) B200_CALL(g_b200.QPSetBox(ctx->qp, NULL, ctx->lb, ctx->ub));

  /* equality constraints (SMALXE): one row B_E (the SVM-type constraint y'a = c of BASELINE config 4; MATONEROW in PERMON,
     src/mat/impls/onerow/onerow.c:97-113, or any other Mat type).  The row is read through the public interface only: B_E^T e_1 */
  if (BE) {
    Vec      e = NULL, row = NULL;
    PetscInt mE, nE, nb;
    PetscCall(MatGetSize(BE, &mE, &nE));
    PetscCheck(mE == 1, PetscObjectComm((PetscObject)qps), PETSC_ERR_SUP, "this adapter forwards a single equality row; %" PetscInt_FMT " rows given", mE);
    PetscCall(MatCreateVecs(BE, &row, &e));
    PetscCall(VecSet(e, 1.0));
    PetscCall(MatMultTranspose(BE, e, row));
    PetscCall(VecDestroy(&e));
    PetscCall(VecGetLocalSize(row, &nb));
    ctx->vbe = row; /* owned: destroyed in B200ReleaseBorrowed */
    PetscCall(VecGetArrayRead(row, &ctx->pbe));
    B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)nb, (b200_int)N, ctx->pbe, &ctx->BErow));
    B200_CALL(g_b200.MatCreateOneRow(ctx->BErow, &ctx->BE));
    if (cE) {
      PetscInt nc, Nc;
      PetscCall(VecGetLocalSize(cE, &nc));
      PetscCall(VecGetSize(cE, &Nc));
      ctx->vce = cE;
      PetscCall(VecGetArrayRead(cE, &ctx->pce));
      B200_CALL(g_b200.VecCreateMPIWithArray(comm, 1, (b200_int)nc, (b200_int)Nc, ctx->pce, &ctx->cE));
    }
    B200_CALL(g_b200.QPSetEq(ctx->qp, ctx->BE, ctx->cE));
  }

  B200_CALL(g_b200.QPSCreate(comm, &ctx->qps));
  B200_CALL(g_b200.QPSSetType(ctx->qps, ctx->type));
  B200_CALL(g_b200.QPSSetQP(ctx->qps, ctx->qp));
  B200_CALL(g_b200.QPSSetTolerances(ctx->qps, qps->rtol, qps->atol, qps->divtol, (b200_int)qps->max_it));
  PetscCall(PetscObjectGetOptionsPrefix((PetscObject)qps, &prefix));
  if (prefix) B200_CALL(g_b200.QPSSetOptionsPrefix(ctx->qps, prefix));
  B200_CALL(g_b200.QPSSetFromOptions(ctx->qps)); /* the same -qps_mpgp_* / -qps_smalxe_* keys, read from the forwarded database */
  B200_CALL(g_b200.QPSSetAutoPostSolve(ctx->qps, 0)); /* PERMON's own QPSPostSolve computes multipliers from x on its side */
  B200_CALL(g_b200.QPSSetUp(ctx->qps));              /* packs + uploads the matrix, power method (alpha = 2 / maxeig) */
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::solve -- QPSSolve_MPGP mpgp.c:438-650 / QPSSolve_SMALXE smalxe.c:893-997: the whole iteration on the device */
static PetscErrorCode QPSSolve_B200(QPS qps)
{
  QPS_B200     *ctx = (QPS_B200 *)qps->data;
  const double *sol;
  b200_int      its;
  int           reason;
  double        rnorm;

  PetscFunctionBegin;
  B200_CALL(g_b200.QPSSetTolerances(ctx->qps, qps->rtol, qps->atol, qps->divtol, (b200_int)qps->max_it));
  B200_CALL(g_b200.QPSSolve(ctx->qps));
  B200_CALL(g_b200.QPSGetIterationNumber(ctx->qps, &its));
  B200_CALL(g_b200.QPSGetConvergedReason(ctx->qps, &reason));
  B200_CALL(g_b200.QPSGetResidualNorm(ctx->qps, &rnorm));
  qps->iteration = (PetscInt)its;
  qps->reason    = (KSPConvergedReason)reason;
  qps->rnorm     = (PetscReal)rnorm;
  /* D2H: the iterate lands in the array the library adopted, i.e. in the PETSc Vec x itself */
  B200_CALL(g_b200.VecGetArrayRead(ctx->x, &sol));
  B200_CALL(g_b200.VecRestoreArrayRead(ctx->x, &sol));
  PetscCall(PetscObjectStateIncrease((PetscObject)ctx->vx));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::reset (qps.c:236-249 calls it) */
static PetscErrorCode QPSReset_B200(QPS qps)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;

  PetscFunctionBegin;
  PetscCall(B200DestroyDeviceSide(ctx));
  PetscCall(B200ReleaseBorrowed(ctx));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::destroy -- QPSDestroy_MPGP mpgp.c:667-692 */
static PetscErrorCode QPSDestroy_B200(QPS qps)
{
  PetscFunctionBegin;
  PetscCall(QPSReset_B200(qps));
  PetscCall(PetscFree(qps->data));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::resetstatistics -- QPSResetStatistics_MPGP mpgp.c:654-664 */
static PetscErrorCode QPSResetStatistics_B200(QPS qps)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;

  PetscFunctionBegin;
  if (ctx->qps) B200_CALL(g_b200.QPSResetStatistics(ctx->qps));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::isqpcompatible -- QPSIsQPCompatible_MPGP mpgp.c:695-711, QPSIsQPCompatible_SMALXE smalxe.c:1009-1027 */
static PetscErrorCode QPSIsQPCompatible_B200(QPS qps, QP qp, PetscBool *flg)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;
  Mat       Beq = NULL, Bineq = NULL;
  Vec       ceq = NULL, cineq = NULL;
  QPC       qpc = NULL;

  PetscFunctionBegin;
  PetscCall(QPGetEq(qp, &Beq, &ceq));
  PetscCall(QPGetIneq(qp, &Bineq, &cineq));
  PetscCall(QPGetQPC(qp, &qpc));
  *flg = PETSC_FALSE;
  if (Bineq || cineq) PetscFunctionReturn(PETSC_SUCCESS);
  if (!strcmp(ctx->type, "mpgp")) {
    if (Beq || ceq) PetscFunctionReturn(PETSC_SUCCESS);
    if (qpc) PetscCall(PetscObjectTypeCompare((PetscObject)qpc, QPCBOX, flg));
  } else {
    *flg = Beq ? PETSC_TRUE : PETSC_FALSE;
  }
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::setfromoptions -- QPSSetFromOptions_MPGP mpgp.c:715-747: the keys are parsed by the library from the forwarded database */
static PetscErrorCode QPSSetFromOptions_B200(QPS qps, PetscOptionItems PetscOptionsObject)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;

  PetscFunctionBegin;
  (void)PetscOptionsObject;
  if (ctx->qps) B200_CALL(g_b200.QPSSetFromOptions(ctx->qps));
  qps->setupcalled = PETSC_FALSE; /* options may change alpha / expansion type: set up again before the next solve */
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* the library prints into its own ASCII viewer: route it through a temporary file into the PETSc viewer.  PERMON's QPSViewConvergence
   (qps.c:968-1000) prints the generic lines itself and calls _QPSOps::viewconvergence for the type-specific ones, so only the lines after
   "<type> specific:" are forwarded (the viewer's own tab level indents them) */
static PetscErrorCode B200ViewThrough(PetscViewer v, int (*fn)(void *, void *), void *obj)
{
  char  name[] = "/tmp/permon_b200_viewXXXXXX", line[1024];
  int   fd     = mkstemp(name), specific = 0;
  void *bv     = NULL;
  FILE *f;

  PetscFunctionBegin;
  PetscCheck(fd >= 0, PETSC_COMM_SELF, PETSC_ERR_FILE_OPEN, "cannot create a temporary file");
  close(fd);
  B200_CALL(g_b200.PetscViewerASCIIOpen(*g_b200.comm_world, name, &bv));
  B200_CALL(fn(obj, bv));
  B200_CALL(g_b200.PetscViewerDestroy(&bv));
  f = fopen(name, "r");
  if (f) {
    while (fgets(line, sizeof line, f)) {
      const char *p = line;
      while (*p == ' ') p++;
      if (specific) PetscCall(PetscViewerASCIIPrintf(v, "%s", p));
      else if (strstr(p, "specific:")) specific = 1;
    }
    fclose(f);
  }
  remove(name);
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::viewconvergence -- QPSViewConvergence_MPGP mpgp.c:751-770 ("number of Hessian multiplications ..." lines of the golden files) */
static PetscErrorCode QPSViewConvergence_B200(QPS qps, PetscViewer v)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;

  PetscFunctionBegin;
  if (ctx->qps) PetscCall(B200ViewThrough(v, g_b200.QPSViewConvergence, ctx->qps));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::view */
static PetscErrorCode QPSView_B200(QPS qps, PetscViewer v)
{
  QPS_B200 *ctx = (QPS_B200 *)qps->data;

  PetscFunctionBegin;
  PetscCall(PetscViewerASCIIPrintf(v, "  %s on libpermon_b200.so (B200, device-resident iteration)\n", ctx->type));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* _QPSOps::monitor -- QPSMonitorDefault_MPGP mpgp.c:21-34; _QPSOps::monitorcostfunction -- mpgp.c:38-58 (not provided on the device path) */
static PetscErrorCode QPSMonitor_B200(QPS qps, PetscInt n, PetscViewer v)
{
  PetscFunctionBegin;
  PetscCall(PetscViewerASCIIPrintf(v, "%3" PetscInt_FMT " %s ||gp||=%.10e\n", n, ((QPS_B200 *)qps->data)->type, (double)qps->rnorm));
  PetscFunctionReturn(PETSC_SUCCESS);
}
static PetscErrorCode QPSMonitorCostFunction_B200(QPS qps, PetscInt n, PetscViewer v)
{
  PetscFunctionBegin;
  PetscCall(QPSMonitor_B200(qps, n, v));
  PetscFunctionReturn(PETSC_SUCCESS);
}

static PetscErrorCode QPSCreate_B200(QPS qps, const char *type)
{
  QPS_B200 *ctx;

  PetscFunctionBegin;
  PetscCall(PetscNew(&ctx));
  ctx->type = type;
  qps->data = (void *)ctx;
  qps->ops->solve               = QPSSolve_B200;
  qps->ops->setup               = QPSSetUp_B200;
  qps->ops->destroy             = QPSDestroy_B200;
  qps->ops->view                = QPSView_B200;
  qps->ops->viewconvergence     = QPSViewConvergence_B200;
  qps->ops->setfromoptions      = QPSSetFromOptions_B200;
  qps->ops->reset               = QPSReset_B200;
  qps->ops->resetstatistics     = QPSResetStatistics_B200;
  qps->ops->isqpcompatible      = QPSIsQPCompatible_B200;
  qps->ops->monitor             = QPSMonitor_B200;
  qps->ops->monitorcostfunction = QPSMonitorCostFunction_B200;
  PetscFunctionReturn(PETSC_SUCCESS);
}
PERMON_EXTERN PetscErrorCode QPSCreate_MPGP_B200(QPS qps)
{
  PetscFunctionBegin;
  PetscCall(QPSCreate_B200(qps, "mpgp"));
  PetscFunctionReturn(PETSC_SUCCESS);
}
PERMON_EXTERN PetscErrorCode QPSCreate_SMALXE_B200(QPS qps)
{
  PetscFunctionBegin;
  PetscCall(QPSCreate_B200(qps, "smalxe"));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* registration: the names of the stock solvers are overridden, user code (-qps_type mpgp, QPSSetType(qps, QPSMPGP)) is unchanged */
PERMON_EXTERN PetscErrorCode PermonB200RegisterQPS(void)
{
  PetscFunctionBegin;
  PetscCall(QPSRegister(QPSMPGP, QPSCreate_MPGP_B200));
  PetscCall(QPSRegister(QPSSMALXE, QPSCreate_SMALXE_B200));
  PetscFunctionReturn(PETSC_SUCCESS);
}
PERMON_EXTERN PetscErrorCode PetscDLLibraryRegister_permonb200(void)
{
  PetscFunctionBegin;
  PetscCall(PermonB200RegisterQPS());
  PetscFunctionReturn(PETSC_SUCCESS);
}
#endif /* PERMON_B200_HAVE_PETSC || PERMON_B200_MOCK_PETSC */
