/*
 * permon_b200.h -- C ABI of libpermon_b200.so: PERMON's QP / QPC / QPPF / QPS surface for the
 * QPSMPGP + QPSSMALXE hot path, executed on NVIDIA B200 (sm_100a).
 *
 * The entry points below are exactly the functions a PERMON user (or PERMON's own registry, see
 * INTEGRATION.md) binds for this path; every declaration cites the reference interface it replaces
 * (file:line into the permon/permon tree).  PETSc itself is not available in this environment, so a
 * minimal stand-in for the PETSc types the path needs (Vec, Mat, IS, options, MPI_Comm) is part of this
 * header ("shim" section).  Signatures contain only plain pointers, integers and doubles.
 *
 * Conventions (identical to the reference, SURVEY.md 8b):
 *  - every function returns PetscErrorCode (0 == PETSC_SUCCESS); numerical failure is NOT an error but a
 *    negative KSPConvergedReason (QPSGetConvergedReason / QPIsSolved);
 *  - objects are reference counted: setters take a reference, the caller keeps and destroys its own;
 *    XxxDestroy(&obj) decrements and nulls the handle;
 *  - data are uploaded to the device once (QPSSetUp); the iteration stays on the device; results are
 *    brought back when the caller asks for host arrays (VecGetArray[Read]);
 *  - one process drives one GPU; a multi-GPU "communicator" is one process per GPU joined over NCCL.
 *  - there is NO CPU execution path: every call that computes fails with PETSC_ERR_GPU when no CUDA
 *    device is usable.
 */
#ifndef PERMON_B200_H
#define PERMON_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PERMON_EXTERN __attribute__((visibility("default")))
#else
#define PERMON_EXTERN
#endif

/* ===================================================================================================
 * PETSc stand-in ("shim"): the subset of petscsys.h / petscvec.h / petscmat.h / petscksp.h the path uses
 * =================================================================================================== */
typedef int     PetscErrorCode;
typedef int32_t PetscInt;      /* default PETSc build: 32-bit indices */
typedef double  PetscReal;
typedef double  PetscScalar;
typedef int     PetscMPIInt;
typedef int64_t PetscObjectState;
typedef enum { PETSC_FALSE = 0, PETSC_TRUE = 1 } PetscBool;

#define PETSC_SUCCESS 0
#define PETSC_ERR_MEM 55
#define PETSC_ERR_NOT_CONVERGED 82
#define PETSC_ERR_SUP 56
#define PETSC_ERR_ORDER 58
#define PETSC_ERR_ARG_SIZ 60
#define PETSC_ERR_ARG_WRONG 62
#define PETSC_ERR_ARG_OUTOFRANGE 63
#define PETSC_ERR_ARG_WRONGSTATE 73
#define PETSC_ERR_ARG_INCOMP 75
#define PETSC_ERR_LIB 76
#define PETSC_ERR_PLIB 77
#define PETSC_ERR_ARG_NULL 85
#define PETSC_ERR_ARG_UNKNOWN_TYPE 86
#define PETSC_ERR_GPU 97
#define PETSC_ERR_GPU_RESOURCE 98

#define PETSC_DECIDE (-1)
#define PETSC_DEFAULT (-2)
#define PETSC_DETERMINE PETSC_DECIDE
#define PETSC_MACHINE_EPSILON 2.2204460492503131e-16
#define PETSC_MAX_REAL 1.7976931348623157e+308
#define PETSC_INFINITY (PETSC_MAX_REAL / 4)
#define PETSC_NINFINITY (-PETSC_INFINITY)
#define PETSC_SMALL 1.e-10

/* petscksp.h: KSPConvergedReason (only the values QPS produces) */
typedef enum {
  KSP_CONVERGED_RTOL            = 2,
  KSP_CONVERGED_ATOL            = 3,
  KSP_CONVERGED_ITS             = 4,
  KSP_CONVERGED_HAPPY_BREAKDOWN = 7,
  KSP_DIVERGED_NULL             = -2,
  KSP_DIVERGED_ITS              = -3,
  KSP_DIVERGED_DTOL             = -4,
  KSP_DIVERGED_BREAKDOWN        = -5,
  KSP_DIVERGED_NANORINF         = -9,
  KSP_DIVERGED_INDEFINITE_MAT   = -10,
  KSP_CONVERGED_ITERATING       = 0
} KSPConvergedReason;

typedef enum { NORM_1 = 0, NORM_2 = 1, NORM_INFINITY = 3 } NormType;

typedef struct _p_PermonComm *MPI_Comm;     /* communicator = the set of GPU-owning processes */
typedef struct _p_Vec        *Vec;
typedef struct _p_Mat        *Mat;
typedef struct _p_IS         *IS;
typedef struct _p_PetscViewer *PetscViewer; /* ASCII viewer on a FILE*; NULL == stdout */
typedef void(PetscCtxDestroyFn)(void **);

extern PERMON_EXTERN MPI_Comm PETSC_COMM_WORLD;
extern PERMON_EXTERN MPI_Comm PETSC_COMM_SELF;

/* --- library life cycle: include/permonsys.h:136-137, src/sys/permoninit.c:36,104 --- */
PERMON_EXTERN PetscErrorCode PermonInitialize(int *argc, char ***args, const char file[], const char help[]);
PERMON_EXTERN PetscErrorCode PermonFinalize(void);

/* --- B200 specific boundary helpers (no reference counterpart: they replace mpiexec / PETSc device setup) --- */
/* number of visible CUDA devices (0 => every compute call fails with PETSC_ERR_GPU) */
PERMON_EXTERN PetscErrorCode PermonB200GetDeviceCount(int *count);
/* choose the CUDA device of this process (default: LOCAL_RANK or 0) -- before any object is created */
PERMON_EXTERN PetscErrorCode PermonB200SetDevice(int device);
/* run all kernels on a caller-owned cudaStream_t (e.g. torch's current stream); NULL = library stream */
PERMON_EXTERN PetscErrorCode PermonB200SetStream(void *cuda_stream);
PERMON_EXTERN PetscErrorCode PermonB200GetStream(void **cuda_stream);
PERMON_EXTERN PetscErrorCode PermonB200Synchronize(void);
/* multi-GPU bootstrap: rank 0 creates a 128-byte NCCL unique id, the host language broadcasts it, every rank joins */
PERMON_EXTERN PetscErrorCode PermonB200GetUniqueId(void *id128);
PERMON_EXTERN PetscErrorCode PermonB200CommInitRank(int nranks, int rank, const void *id128);
/* setup-time host exchange used to build halo plans: all-gather of variable-length byte strings.
   Default implementation runs over NCCL; a host language may install its own (e.g. gloo in CPU tests). */
typedef int (*PermonB200AllGatherV)(void *ctx, const void *sendbuf, int64_t sendbytes, void *recvbuf,
                                    const int64_t *recvbytes /* size entries */);
typedef int (*PermonB200AllGatherI64)(void *ctx, int64_t value, int64_t *all /* size entries */);
PERMON_EXTERN PetscErrorCode PermonB200CommSetHostExchange(int nranks, int rank, PermonB200AllGatherI64 agi, PermonB200AllGatherV agv, void *ctx);
/* kernel-level instrumentation for bench.py: CUDA-event timing of every launch of one kernel family */
PERMON_EXTERN PetscErrorCode PermonB200ProfileBegin(void);
PERMON_EXTERN PetscErrorCode PermonB200ProfileEnd(int *nfamilies);
PERMON_EXTERN PetscErrorCode PermonB200ProfileGet(int family, const char **name, int64_t *launches, double *total_ms, double *bytes_per_launch);
PERMON_EXTERN PetscErrorCode PermonB200ProfileGetWorking(int family, int64_t *launches, double *total_ms);   /* launches that did work (device-driven kernels exit at once when they have nothing to do) */
PERMON_EXTERN PetscErrorCode PermonB200ProfileDump(const char *csv_path);   /* per-launch timeline of the last profiled region */
PERMON_EXTERN PetscErrorCode PermonB200GetLaunchCount(int64_t *launches);
PERMON_EXTERN const char    *PermonB200GetLastErrorMessage(void);

/* --- options database (petscoptions.h) --- */
PERMON_EXTERN PetscErrorCode PetscOptionsSetValue(void *options, const char name[], const char value[]);
PERMON_EXTERN PetscErrorCode PetscOptionsClearValue(void *options, const char name[]);
PERMON_EXTERN PetscErrorCode PetscOptionsClear(void *options);
PERMON_EXTERN PetscErrorCode PetscOptionsInsertString(void *options, const char in_str[]);
PERMON_EXTERN PetscErrorCode PetscOptionsHasName(void *options, const char pre[], const char name[], PetscBool *set);

/* --- viewers --- */
PERMON_EXTERN PetscErrorCode PetscViewerASCIIOpen(MPI_Comm comm, const char name[], PetscViewer *viewer);
PERMON_EXTERN PetscErrorCode PetscViewerDestroy(PetscViewer *viewer);

/* --- IS (petscis.h) --- */
PERMON_EXTERN PetscErrorCode ISCreateStride(MPI_Comm comm, PetscInt n, PetscInt first, PetscInt step, IS *is);
PERMON_EXTERN PetscErrorCode ISCreateGeneral(MPI_Comm comm, PetscInt n, const PetscInt idx[], int copymode, IS *is);
PERMON_EXTERN PetscErrorCode ISGetLocalSize(IS is, PetscInt *n);
PERMON_EXTERN PetscErrorCode ISDestroy(IS *is);

/* --- Vec (petscvec.h).  n = local length, N = global length.  "WithArray": the caller's host buffer is the
 *     host storage of the Vec (as in PETSc) -- results appear in it after VecGetArray[Read]/VecRestoreArray. --- */
PERMON_EXTERN PetscErrorCode VecCreateSeq(MPI_Comm comm, PetscInt n, Vec *v);
PERMON_EXTERN PetscErrorCode VecCreateMPI(MPI_Comm comm, PetscInt n, PetscInt N, Vec *v);
PERMON_EXTERN PetscErrorCode VecCreateSeqWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, const PetscScalar array[], Vec *v);
PERMON_EXTERN PetscErrorCode VecCreateMPIWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, PetscInt N, const PetscScalar array[], Vec *v);
/* device-resident input (PETSc: VecCreateSeqCUDAWithArray): `darray` is a CUDA device pointer owned by the caller */
PERMON_EXTERN PetscErrorCode VecCreateSeqCUDAWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, const PetscScalar darray[], Vec *v);
PERMON_EXTERN PetscErrorCode VecCreateMPICUDAWithArray(MPI_Comm comm, PetscInt bs, PetscInt n, PetscInt N, const PetscScalar darray[], Vec *v);
PERMON_EXTERN PetscErrorCode VecDuplicate(Vec v, Vec *newv);
PERMON_EXTERN PetscErrorCode VecDestroy(Vec *v);
PERMON_EXTERN PetscErrorCode VecGetSize(Vec v, PetscInt *N);
PERMON_EXTERN PetscErrorCode VecGetLocalSize(Vec v, PetscInt *n);
PERMON_EXTERN PetscErrorCode VecGetOwnershipRange(Vec v, PetscInt *low, PetscInt *high);
PERMON_EXTERN PetscErrorCode VecGetArray(Vec v, PetscScalar **a);
PERMON_EXTERN PetscErrorCode VecRestoreArray(Vec v, PetscScalar **a);
PERMON_EXTERN PetscErrorCode VecGetArrayRead(Vec v, const PetscScalar **a);
PERMON_EXTERN PetscErrorCode VecRestoreArrayRead(Vec v, const PetscScalar **a);
PERMON_EXTERN PetscErrorCode VecCUDAGetArray(Vec v, PetscScalar **d);      /* device pointer, read-write */
PERMON_EXTERN PetscErrorCode VecCUDARestoreArray(Vec v, PetscScalar **d);
PERMON_EXTERN PetscErrorCode VecCUDAGetArrayRead(Vec v, const PetscScalar **d);
PERMON_EXTERN PetscErrorCode VecCUDARestoreArrayRead(Vec v, const PetscScalar **d);
PERMON_EXTERN PetscErrorCode VecSet(Vec v, PetscScalar alpha);
PERMON_EXTERN PetscErrorCode VecZeroEntries(Vec v);
PERMON_EXTERN PetscErrorCode VecCopy(Vec x, Vec y);
PERMON_EXTERN PetscErrorCode VecScale(Vec x, PetscScalar alpha);
PERMON_EXTERN PetscErrorCode VecAXPY(Vec y, PetscScalar alpha, Vec x);
PERMON_EXTERN PetscErrorCode VecAYPX(Vec y, PetscScalar beta, Vec x);
PERMON_EXTERN PetscErrorCode VecWAXPY(Vec w, PetscScalar alpha, Vec x, Vec y);
PERMON_EXTERN PetscErrorCode VecPointwiseMax(Vec w, Vec x, Vec y);
PERMON_EXTERN PetscErrorCode VecPointwiseMin(Vec w, Vec x, Vec y);
PERMON_EXTERN PetscErrorCode VecDot(Vec x, Vec y, PetscScalar *val);
PERMON_EXTERN PetscErrorCode VecNorm(Vec x, NormType type, PetscReal *val);
/* include/permonvec.h:11-12, src/vec/interface/permonvecutils.c:266,303 */
PERMON_EXTERN PetscErrorCode VecInvalidate(Vec vec);
PERMON_EXTERN PetscErrorCode VecIsInvalidated(Vec vec, PetscBool *flg);

/* --- Mat (petscmat.h).  CSR arrays are host pointers with GLOBAL column indices; they are copied. --- */
PERMON_EXTERN PetscErrorCode MatCreateSeqAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt i[], PetscInt j[], PetscScalar a[], Mat *mat);
PERMON_EXTERN PetscErrorCode MatCreateMPIAIJWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt M, PetscInt N, const PetscInt i[], const PetscInt j[], const PetscScalar a[], Mat *mat);
/* same, from CUDA device pointers (int32 rowptr/cols, fp64 values): nothing crosses PCIe */
PERMON_EXTERN PetscErrorCode MatCreateSeqAIJCUSPARSEWithArrays(MPI_Comm comm, PetscInt m, PetscInt n, const PetscInt di[], const PetscInt dj[], const PetscScalar da[], Mat *mat);
/* include/permonmat.h:36, src/mat/impls/onerow/onerow.c:97: the 1 x n matrix a^T */
PERMON_EXTERN PetscErrorCode MatCreateOneRow(Vec a, Mat *A_new);
/* include/permonmat.h:28, src/mat/impls/composite/matprod.c:42: implicit product mats[nmat-1]*...*mats[0] (nmat <= 2) */
PERMON_EXTERN PetscErrorCode MatCreateProd(MPI_Comm comm, PetscInt nmat, const Mat *mats, Mat *mat);
PERMON_EXTERN PetscErrorCode MatDestroy(Mat *A);
PERMON_EXTERN PetscErrorCode MatGetSize(Mat A, PetscInt *M, PetscInt *N);
PERMON_EXTERN PetscErrorCode MatGetLocalSize(Mat A, PetscInt *m, PetscInt *n);
PERMON_EXTERN PetscErrorCode MatGetOwnershipRange(Mat A, PetscInt *low, PetscInt *high);
PERMON_EXTERN PetscErrorCode MatCreateVecs(Mat A, Vec *right, Vec *left);
PERMON_EXTERN PetscErrorCode MatMult(Mat A, Vec x, Vec y);
PERMON_EXTERN PetscErrorCode MatMultAdd(Mat A, Vec x, Vec y, Vec z);
PERMON_EXTERN PetscErrorCode MatMultTranspose(Mat A, Vec x, Vec y);
/* include/permonmat.h:132, src/mat/interface/permonmatutils.c:442-522 */
PERMON_EXTERN PetscErrorCode MatGetMaxEigenvalue(Mat A, Vec v, PetscReal *lambda_out, PetscReal tol, PetscInt maxits);
/* halo-plan introspection (host data; used by the CPU multi-rank tests) */
PERMON_EXTERN PetscErrorCode MatB200GetHaloInfo(Mat A, PetscInt *nghost, const PetscInt **garray, PetscInt *nneigh, const PetscInt **neigh_rank,
                                                const PetscInt **recv_off, const PetscInt **send_off, const PetscInt **send_idx, PetscInt *nboundary_rows);
/* host split of a row-partitioned matrix (diagonal block with local columns, compressed off-diagonal rows with ghost-buffer columns,
   the local row id of every off-diagonal row); valid until the matrix is first used on the device.  CPU multi-rank tests. */
PERMON_EXTERN PetscErrorCode MatB200GetHostSplit(Mat A, const PetscInt **dia, const PetscInt **dja, const PetscScalar **da, PetscInt *noffrows,
                                                 const PetscInt **oia, const PetscInt **oja, const PetscScalar **oa, const PetscInt **orow);
/* device storage introspection: kind 0/1/2 = CSR (tile-streamed / vector / TMA-staged), 3 = packed dictionary-coded tiles;
   stream_bytes = bytes one SpMV reads for the matrix itself (diagonal + off-diagonal block); coded_tiles / tiles of the packed form.
   Uploads a row-partitioned matrix if it is not on the device yet. */
PERMON_EXTERN PetscErrorCode MatB200GetStorageInfo(Mat A, PetscInt *kind, PetscReal *stream_bytes, PetscInt *coded_tiles, PetscInt *tiles);
/* like MatCreateMPIAIJWithArrays, but di / dj / da are CUDA device pointers (int32 row pointer, GLOBAL column ids, fp64 values) of the
   device the library runs on.  The arrays must be complete when the call is made (device-synchronised, or written on the stream of
   PermonB200GetStream).  The matrix is re-coded on the GPU into the same stored form the host constructor builds; the call returns when
   the arrays are no longer read, and nothing of them is kept (the caller may free or overwrite them).  Null arrays: PETSC_ERR_ARG_NULL;
   host memory: PETSC_ERR_ARG_WRONG. */
PERMON_EXTERN PetscErrorCode MatB200CreateAIJWithDeviceArrays(MPI_Comm comm, PetscInt m, PetscInt n, PetscInt M, PetscInt N, const PetscInt di[], const PetscInt dj[],
                                                              const PetscScalar da[], Mat *mat);
/* parts of the stored form of an AIJ matrix (MatB200GetStoredForm): field + MATB200_FORM_OFFDIAG selects the off-diagonal block of a
   row-partitioned matrix instead of the diagonal block (the whole matrix on one rank) */
#define MATB200_FORM_SCALARS 0   /* 15 int64: kind, n, ncols, nnz, st_npat, st_nwin, st_lmax, st_dlo, st_dhi, pk_max, pk_bytes, pk_coded, stages, tile_cap, W */
#define MATB200_FORM_ST_MASKS 1  /* all-stencil form: presence byte per row (ntiles * 256) */
#define MATB200_FORM_ST_PID 2    /* pattern id per tile */
#define MATB200_FORM_ST_PATS 3   /* pattern table */
#define MATB200_FORM_PK_BLOB 4   /* packed tiles: blob (incl. its 16 trailing bytes) */
#define MATB200_FORM_PK_OFF 5    /* tile offsets in 16-byte units (ntiles + 1) */
#define MATB200_FORM_CSR_IA 6
#define MATB200_FORM_CSR_JA 7    /* up to nnz */
#define MATB200_FORM_CSR_A 8     /* up to nnz */
#define MATB200_FORM_ELL_VAL 9   /* tile-ELL arrays */
#define MATB200_FORM_ELL_COL 10
#define MATB200_FORM_ELL_LEN 11
#define MATB200_FORM_ELL_LT 12
#define MATB200_FORM_ELL_OFF 13
#define MATB200_FORM_ROWS 14     /* row id of every compressed row (off-diagonal block) */
#define MATB200_FORM_OFFDIAG 16
/* copy one part of the stored form into a host buffer of *nbytes bytes; buf == NULL returns the size of the part in *nbytes (0: the
   matrix has no such array).  Uploads a row-partitioned matrix if it is not on the device yet. */
PERMON_EXTERN PetscErrorCode MatB200GetStoredForm(Mat A, PetscInt part, void *buf, size_t *nbytes);
/* host-side packer of the device matrix format (permon_b200/csrc/pack.cpp), exposed so that the format can be checked without a
   GPU: tile t occupies blob[16*tile_off[t] .. 16*tile_off[t+1]).  *blob == NULL when the matrix cannot be packed. */
PERMON_EXTERN PetscErrorCode PermonB200PackTiles(PetscInt n, const PetscInt ia[], const PetscInt ja[], const PetscScalar a[], unsigned char **blob,
                                                 unsigned **tile_off, PetscInt *ntiles, PetscInt *coded_tiles);
PERMON_EXTERN PetscErrorCode PermonB200PackFree(unsigned char *blob, unsigned *tile_off);

/* ===================================================================================================
 * QPC -- separable constraints (box): include/permonqpc.h:21-56, src/qpc
 * =================================================================================================== */
typedef struct _p_QPC *QPC;
#define QPCType char *
#define QPCBOX  "box" /* permonqpc.h:11 */

PERMON_EXTERN PetscErrorCode QPCCreate(MPI_Comm comm, QPC *qpc);                                   /* permonqpc.h:21, qpc.c:14 */
PERMON_EXTERN PetscErrorCode QPCDestroy(QPC *qpc);                                                 /* permonqpc.h:24 */
PERMON_EXTERN PetscErrorCode QPCSetUp(QPC qpc);                                                    /* permonqpc.h:26, qpc.c:37 */
PERMON_EXTERN PetscErrorCode QPCSetType(QPC qpc, const QPCType type);                              /* permonqpc.h:29 */
PERMON_EXTERN PetscErrorCode QPCGetType(QPC qpc, const QPCType *type);                             /* permonqpc.h:32 */
PERMON_EXTERN PetscErrorCode QPCSetIS(QPC qpc, IS is);                                             /* permonqpc.h:30 */
PERMON_EXTERN PetscErrorCode QPCGetIS(QPC qpc, IS *is);                                            /* permonqpc.h:33 */
PERMON_EXTERN PetscErrorCode QPCGetBlockSize(QPC qpc, PetscInt *bs);                               /* permonqpc.h:41 */
PERMON_EXTERN PetscErrorCode QPCGetNumberOfConstraints(QPC qpc, PetscInt *num);                    /* permonqpc.h:44 */
PERMON_EXTERN PetscErrorCode QPCProject(QPC qpc, Vec x, Vec Px);                                   /* permonqpc.h:46, qpc.c:466 */
PERMON_EXTERN PetscErrorCode QPCGrads(QPC qpc, Vec x, Vec g, Vec gf, Vec gc);                      /* permonqpc.h:47, qpc.c:540 */
PERMON_EXTERN PetscErrorCode QPCGradReduced(QPC qpc, Vec x, Vec gf, PetscReal alpha, Vec gr);      /* permonqpc.h:48, qpc.c:589 */
PERMON_EXTERN PetscErrorCode QPCFeas(QPC qpc, Vec x, Vec d, PetscReal *alpha);                     /* permonqpc.h:49, qpc.c:503 */
PERMON_EXTERN PetscErrorCode QPCCreateBox(MPI_Comm comm, IS is, Vec lb, Vec ub, QPC *qpc);         /* permonqpc.h:53, qpcbox.c:554 */
PERMON_EXTERN PetscErrorCode QPCBoxSet(QPC qpc, Vec lb, Vec ub);                                   /* permonqpc.h:54 */
PERMON_EXTERN PetscErrorCode QPCBoxGet(QPC qpc, Vec *lb, Vec *ub);                                 /* permonqpc.h:55 */
PERMON_EXTERN PetscErrorCode QPCBoxGetMultipliers(QPC qpc, Vec *llb, Vec *lub);                    /* permonqpc.h:56 */
PERMON_EXTERN PetscErrorCode QPCViewKKT(QPC qpc, Vec x, PetscReal normb, PetscViewer v);           /* permonqpc.h:23, qpcbox.c:333 */

/* ===================================================================================================
 * QPPF -- projector factory on G = B_E: include/permonqppf.h:12-40, src/qppf/interface/qppf.c
 * =================================================================================================== */
typedef struct _p_QPPF *QPPF;

PERMON_EXTERN PetscErrorCode QPPFCreate(MPI_Comm comm, QPPF *cp);                    /* permonqppf.h:12, qppf.c:96 */
PERMON_EXTERN PetscErrorCode QPPFDestroy(QPPF *cp);                                  /* permonqppf.h:17 */
PERMON_EXTERN PetscErrorCode QPPFReset(QPPF cp);                                     /* permonqppf.h:13 */
PERMON_EXTERN PetscErrorCode QPPFSetUp(QPPF cp);                                     /* permonqppf.h:15, qppf.c:371 */
PERMON_EXTERN PetscErrorCode QPPFSetG(QPPF cp, Mat G);                               /* permonqppf.h:27 */
PERMON_EXTERN PetscErrorCode QPPFGetG(QPPF cp, Mat *G);                              /* permonqppf.h:36 */
PERMON_EXTERN PetscErrorCode QPPFGetGHasOrthonormalRows(QPPF cp, PetscBool *flg);    /* permonqppf.h:37 */
PERMON_EXTERN PetscErrorCode QPPFApplyP(QPPF cp, Vec v, Vec Pv);                     /* permonqppf.h:20, qppf.c:572 */
PERMON_EXTERN PetscErrorCode QPPFApplyQ(QPPF cp, Vec v, Vec Qv);                     /* permonqppf.h:21, qppf.c:454 */
PERMON_EXTERN PetscErrorCode QPPFApplyHalfQ(QPPF cp, Vec x, Vec y);                  /* permonqppf.h:22, qppf.c:507 */
PERMON_EXTERN PetscErrorCode QPPFApplyHalfQTranspose(QPPF cp, Vec x, Vec y);         /* permonqppf.h:23, qppf.c:535 */
PERMON_EXTERN PetscErrorCode QPPFApplyCP(QPPF cp, Vec x, Vec y);                     /* permonqppf.h:24, qppf.c:610 */
PERMON_EXTERN PetscErrorCode QPPFApplyGtG(QPPF cp, Vec v, Vec GtGv);                 /* permonqppf.h:25, qppf.c:580 */
PERMON_EXTERN PetscErrorCode QPPFCreateP(QPPF cp, Mat *P);                           /* permonqppf.h:32, qppf.c:685 */
PERMON_EXTERN PetscErrorCode QPPFCreateQ(QPPF cp, Mat *Q);                           /* permonqppf.h:31, qppf.c:650 */
PERMON_EXTERN PetscErrorCode QPPFCreateGtG(QPPF cp, Mat *GtG);                       /* permonqppf.h:34, qppf.c:705 */
PERMON_EXTERN PetscErrorCode QPPFSetFromOptions(QPPF cp);                            /* permonqppf.h:16, qppf.c:170: -qppf_explicit, -qppf_redundancy */
PERMON_EXTERN PetscErrorCode QPPFSetRedundancy(QPPF cp, PetscInt nred);              /* permonqppf.h:28, qppf.c:158 */
PERMON_EXTERN PetscErrorCode QPPFSetExplicitInv(QPPF cp, PetscBool explicitInv);     /* permonqppf.h:29, qppf.c:143 */
PERMON_EXTERN PetscErrorCode QPPFGetAlphaTilde(QPPF cp, Vec *alpha_tilde);           /* permonqppf.h:19, qppf.c:441 */
PERMON_EXTERN PetscErrorCode QPPFGetGGt(QPPF cp, Mat *GGt);                          /* permonqppf.h:38, qppf.c:744 */

/* ===================================================================================================
 * QP -- problem container: include/permonqp.h:21-123, src/qp/interface/qp.c
 * =================================================================================================== */
typedef struct _p_QP *QP;

PERMON_EXTERN PetscErrorCode QPCreate(MPI_Comm comm, QP *qp);                        /* permonqp.h:40, qp.c:94 */
PERMON_EXTERN PetscErrorCode QPDestroy(QP *qp);                                      /* permonqp.h:47 */
PERMON_EXTERN PetscErrorCode QPSetUp(QP qp);                                         /* permonqp.h:46, qp.c:614 */
PERMON_EXTERN PetscErrorCode QPSetOperator(QP qp, Mat A);                            /* permonqp.h:60, qp.c:1086 */
PERMON_EXTERN PetscErrorCode QPSetRhs(QP qp, Vec b);                                 /* permonqp.h:63, qp.c:1259 */
PERMON_EXTERN PetscErrorCode QPSetRhsPlus(QP qp, Vec b);                             /* permonqp.h:64, qp.c:1296 */
PERMON_EXTERN PetscErrorCode QPSetInitialVector(QP qp, Vec x);                       /* permonqp.h:59, qp.c:1978 */
PERMON_EXTERN PetscErrorCode QPSetBox(QP qp, IS is, Vec lb, Vec ub);                 /* permonqp.h:69, qp.c:1858 */
PERMON_EXTERN PetscErrorCode QPSetEq(QP qp, Mat Beq, Vec ceq);                       /* permonqp.h:66, qp.c:1467 */
PERMON_EXTERN PetscErrorCode QPSetQPC(QP qp, QPC qpc);                               /* permonqp.h:91 */
PERMON_EXTERN PetscErrorCode QPSetOptionsPrefix(QP qp, const char prefix[]);         /* permonqp.h:73 */
PERMON_EXTERN PetscErrorCode QPSetFromOptions(QP qp);                                /* permonqp.h:75 */
PERMON_EXTERN PetscErrorCode QPGetSolutionVector(QP qp, Vec *x);                     /* permonqp.h:78, qp.c:2018 */
PERMON_EXTERN PetscErrorCode QPGetOperator(QP qp, Mat *A);                           /* permonqp.h:79 */
PERMON_EXTERN PetscErrorCode QPGetRhs(QP qp, Vec *b);                                /* permonqp.h:82 */
PERMON_EXTERN PetscErrorCode QPGetEq(QP qp, Mat *Beq, Vec *ceq);                     /* permonqp.h:84 */
PERMON_EXTERN PetscErrorCode QPGetBox(QP qp, IS *is, Vec *lb, Vec *ub);              /* permonqp.h:85 */
PERMON_EXTERN PetscErrorCode QPGetQPC(QP qp, QPC *qpc);                              /* permonqp.h:92 */
PERMON_EXTERN PetscErrorCode QPGetQPPF(QP qp, QPPF *pf);                             /* permonqp.h:86 */
PERMON_EXTERN PetscErrorCode QPGetChild(QP qp, QP *child);                           /* permonqp.h:35 */
PERMON_EXTERN PetscErrorCode QPGetParent(QP qp, QP *parent);                         /* permonqp.h:36 */
PERMON_EXTERN PetscErrorCode QPIsSolved(QP qp, PetscBool *flg);                      /* permonqp.h:89 */
PERMON_EXTERN PetscErrorCode QPComputeObjective(QP qp, Vec x, PetscReal *f);         /* permonqp.h:55, qp.c:913 */
PERMON_EXTERN PetscErrorCode QPComputeObjectiveFromGradient(QP qp, Vec x, Vec g, PetscReal *f); /* permonqp.h:57, qp.c:981 */
PERMON_EXTERN PetscErrorCode QPComputeMissingBoxMultipliers(QP qp);                  /* permonqp.h:52, qp.c:829 */
PERMON_EXTERN PetscErrorCode QPComputeMissingEqMultiplier(QP qp);                    /* permonqp.h:51, qp.c:778 */
PERMON_EXTERN PetscErrorCode QPComputeLagrangianGradient(QP qp, Vec x, Vec r, char *kkt_name[]); /* permonqp.h:54, qp.c:668 */
PERMON_EXTERN PetscErrorCode QPGetEqMultiplier(QP qp, Vec *lambda_E, Vec *Bt_lambda);/* B200 helper: borrowed lambda_E / B^T lambda */
PERMON_EXTERN PetscErrorCode QPViewKKT(QP qp, PetscViewer v);                        /* permonqp.h:44, qp.c:245 */
PERMON_EXTERN PetscErrorCode QPChainGetLast(QP qp, QP *child);                       /* permonqp.h:26, qpchain.c:105 */
PERMON_EXTERN PetscErrorCode QPChainSetUp(QP qp);                                    /* permonqp.h:29, qpchain.c:135 */
PERMON_EXTERN PetscErrorCode QPChainPostSolve(QP qp);                                /* permonqp.h:27, qpchain.c:200 */
PERMON_EXTERN PetscErrorCode QPChainViewKKT(QP qp, PetscViewer v);                   /* permonqp.h:31 */
PERMON_EXTERN PetscErrorCode QPRemoveChild(QP qp);                                   /* permonqp.h:34 */
PERMON_EXTERN PetscErrorCode QPTEnforceEqByPenalty(QP qp, PetscReal rho_user, PetscBool rho_direct); /* permonqp.h:96, qptransform.c:329 */
PERMON_EXTERN PetscErrorCode QPTHomogenizeEq(QP qp);                                 /* permonqp.h:97, qptransform.c:437 */
PERMON_EXTERN PetscErrorCode QPTEnforceEqByProjector(QP qp);                        /* permonqp.h:98, qptransform.c:215 */
/* MatOrthType / MatOrthForm: include/permonmat.h:160-171.  The B200 path orthonormalises the (at most 4) dense equality rows with
   MAT_ORTH_GS or MAT_ORTH_CHOLESKY and always stores T*BE explicitly. */
typedef enum { MAT_ORTH_NONE = 0, MAT_ORTH_GS, MAT_ORTH_GS_LINGEN, MAT_ORTH_CHOLESKY, MAT_ORTH_IMPLICIT, MAT_ORTH_INEXACT } MatOrthType;
typedef enum { MAT_ORTH_FORM_IMPLICIT = 0, MAT_ORTH_FORM_EXPLICIT = 1 } MatOrthForm;
PERMON_EXTERN PetscErrorCode QPTOrthonormalizeEq(QP qp, MatOrthType type, MatOrthForm form); /* permonqp.h:101, qptransform.c:566 */
/* MatPenalized: permonqp.h:119-123, src/qp/utils/matpenalized.c */
PERMON_EXTERN PetscErrorCode MatCreatePenalized(QP qp, PetscReal rho, Mat *A_inner);
PERMON_EXTERN PetscErrorCode MatPenalizedSetPenalty(Mat Arho, PetscReal rho);
PERMON_EXTERN PetscErrorCode MatPenalizedUpdatePenalty(Mat Arho, PetscReal rho_update);
PERMON_EXTERN PetscErrorCode MatPenalizedGetPenalty(Mat Arho, PetscReal *rho);

/* ===================================================================================================
 * QPS -- solvers: include/permonqps.h:24-165, src/qps
 * =================================================================================================== */
typedef struct _p_QPS *QPS;
#define QPSType   char *
#define QPSMPGP   "mpgp"   /* permonqps.h:13 */
#define QPSSMALXE "smalxe" /* permonqps.h:16 */
#define QPSKSP    "ksp"    /* permonqps.h:12: unconstrained QPs, conjugate gradients */
#define QPSPCPG   "pcpg"   /* permonqps.h:15: equality-constrained QPs, projected conjugate gradients */

typedef enum { QPS_ARG_MULTIPLE = 0, QPS_ARG_DIRECT = 1 } QPSScalarArgType; /* permonqps.h:19-22 */

PERMON_EXTERN PetscErrorCode QPSRegister(const char sname[], PetscErrorCode (*create)(QPS)); /* permonqps.h:30, qpsregis.c:29 */
PERMON_EXTERN PetscErrorCode QPSCreate(MPI_Comm comm, QPS *qps_new);                  /* permonqps.h:32, qps.c:61 */
PERMON_EXTERN PetscErrorCode QPSDestroy(QPS *qps);                                    /* permonqps.h:35, qps.c:340 */
PERMON_EXTERN PetscErrorCode QPSSetFromOptions(QPS qps);                              /* permonqps.h:36, qps.c:859 */
PERMON_EXTERN PetscErrorCode QPSSetUp(QPS qps);                                       /* permonqps.h:37, qps.c:198 */
PERMON_EXTERN PetscErrorCode QPSReset(QPS qps);                                       /* permonqps.h:38, qps.c:236 */
PERMON_EXTERN PetscErrorCode QPSResetStatistics(QPS qps);                             /* permonqps.h:39, qps.c:265 */
PERMON_EXTERN PetscErrorCode QPSSolve(QPS qps);                                       /* permonqps.h:40, qps.c:537 */
PERMON_EXTERN PetscErrorCode QPSPostSolve(QPS qps);                                   /* permonqps.h:41, qps.c:579 */
PERMON_EXTERN PetscErrorCode QPSIsQPCompatible(QPS qps, QP qp, PetscBool *flg);       /* permonqps.h:42 */
PERMON_EXTERN PetscErrorCode QPSSetDefaultType(QPS qps);                              /* permonqps.h:44, qps.c:420 */
PERMON_EXTERN PetscErrorCode QPSSetType(QPS qps, const QPSType type);                 /* permonqps.h:46, qps.c:379 */
PERMON_EXTERN PetscErrorCode QPSGetType(QPS qps, const QPSType *type);                /* permonqps.h:54 */
PERMON_EXTERN PetscErrorCode QPSSetQP(QPS qps, QP qp);                                /* permonqps.h:47, qps.c:171 */
PERMON_EXTERN PetscErrorCode QPSGetQP(QPS qps, QP *qp);                               /* permonqps.h:55 */
PERMON_EXTERN PetscErrorCode QPSGetSolvedQP(QPS qps, QP *qp);                         /* permonqps.h:56 */
PERMON_EXTERN PetscErrorCode QPSSetTolerances(QPS qps, PetscReal rtol, PetscReal abstol, PetscReal dtol, PetscInt maxits); /* permonqps.h:48 */
PERMON_EXTERN PetscErrorCode QPSGetTolerances(QPS qps, PetscReal *rtol, PetscReal *abstol, PetscReal *dtol, PetscInt *maxits); /* permonqps.h:57 */
PERMON_EXTERN PetscErrorCode QPSSetOptionsPrefix(QPS qps, const char prefix[]);       /* permonqps.h:49 */
PERMON_EXTERN PetscErrorCode QPSAppendOptionsPrefix(QPS qps, const char prefix[]);    /* permonqps.h:50 */
PERMON_EXTERN PetscErrorCode QPSGetOptionsPrefix(QPS qps, const char *prefix[]);      /* permonqps.h:58 */
PERMON_EXTERN PetscErrorCode QPSSetConvergenceTest(QPS qps, PetscErrorCode (*converge)(QPS, KSPConvergedReason *), void *cctx, PetscErrorCode (*destroy)(void *)); /* permonqps.h:51, qps.c:617 */
PERMON_EXTERN PetscErrorCode QPSGetConvergenceContext(QPS qps, void **ctx);           /* permonqps.h:59 */
PERMON_EXTERN PetscErrorCode QPSSetAutoPostSolve(QPS qps, PetscBool flg);             /* permonqps.h:52 */
PERMON_EXTERN PetscErrorCode QPSGetAutoPostSolve(QPS qps, PetscBool *flg);            /* permonqps.h:65 */
PERMON_EXTERN PetscErrorCode QPSGetConvergedReason(QPS qps, KSPConvergedReason *reason); /* permonqps.h:60 */
PERMON_EXTERN PetscErrorCode QPSGetResidualNorm(QPS qps, PetscReal *rnorm);           /* permonqps.h:61 */
PERMON_EXTERN PetscErrorCode QPSGetIterationNumber(QPS qps, PetscInt *its);           /* permonqps.h:62 */
PERMON_EXTERN PetscErrorCode QPSGetAccumulatedIterationNumber(QPS qps, PetscInt *its);/* permonqps.h:63 */
PERMON_EXTERN PetscErrorCode QPSConvergedDefault(QPS qps, KSPConvergedReason *reason);/* permonqps.h:69, qps.c:675 */
PERMON_EXTERN PetscErrorCode QPSConvergedDefaultCreate(void **ctx);                   /* permonqps.h:73 */
PERMON_EXTERN PetscErrorCode QPSConvergedDefaultDestroy(void *ctx);                   /* permonqps.h:72 */
PERMON_EXTERN PetscErrorCode QPSConvergedSkip(QPS qps, KSPConvergedReason *reason);   /* permonqps.h:68, qps.c:775 */
PERMON_EXTERN PetscErrorCode QPSMonitorSet(QPS qps, PetscErrorCode (*monitor)(QPS, PetscInt, PetscReal, void *), void *mctx, PetscCtxDestroyFn *destroy); /* permonqps.h:80 */
PERMON_EXTERN PetscErrorCode QPSMonitorCancel(QPS qps);                               /* permonqps.h:81 */
PERMON_EXTERN PetscErrorCode QPSMonitorDefault(QPS qps, PetscInt n, PetscReal rnorm, void *dummy); /* permonqps.h:85, qps.c:1364 */
PERMON_EXTERN PetscErrorCode QPSViewConvergence(QPS qps, PetscViewer viewer);         /* permonqps.h:34, qps.c:968 */

/* MPGP: permonqps.h:100-128, src/qps/impls/mpgp/mpgp.c */
typedef enum { QPS_MPGP_EXPANSION_STD, QPS_MPGP_EXPANSION_PROJCG, QPS_MPGP_EXPANSION_GF, QPS_MPGP_EXPANSION_G, QPS_MPGP_EXPANSION_GFGR, QPS_MPGP_EXPANSION_GGR } QPSMPGPExpansionType;
typedef enum { QPS_MPGP_EXPANSION_LENGTH_FIXED, QPS_MPGP_EXPANSION_LENGTH_OPT, QPS_MPGP_EXPANSION_LENGTH_OPTAPPROX, QPS_MPGP_EXPANSION_LENGTH_BB } QPSMPGPExpansionLengthType;
PERMON_EXTERN PetscErrorCode QPSMPGPGetCurrentStepType(QPS qps, char *stepType);
/* QPSKSP: the Krylov method behind the "ksp" type; without PETSc's KSP the accessors reduce to the type name ("cg") */
PERMON_EXTERN PetscErrorCode QPSKSPSetType(QPS qps, const char *type);                 /* permonqps.h:91, qpsksp.c:83 */
PERMON_EXTERN PetscErrorCode QPSKSPGetType(QPS qps, const char **type);                /* permonqps.h:92, qpsksp.c:100 */
PERMON_EXTERN PetscErrorCode QPSMPGPSetAlpha(QPS qps, PetscReal alpha, QPSScalarArgType argtype);
PERMON_EXTERN PetscErrorCode QPSMPGPGetAlpha(QPS qps, PetscReal *alpha, QPSScalarArgType *argtype);
PERMON_EXTERN PetscErrorCode QPSMPGPSetGamma(QPS qps, PetscReal gamma);
PERMON_EXTERN PetscErrorCode QPSMPGPGetGamma(QPS qps, PetscReal *gamma);
PERMON_EXTERN PetscErrorCode QPSMPGPGetOperatorMaxEigenvalue(QPS qps, PetscReal *maxeig);
PERMON_EXTERN PetscErrorCode QPSMPGPSetOperatorMaxEigenvalue(QPS qps, PetscReal maxeig);
PERMON_EXTERN PetscErrorCode QPSMPGPUpdateMaxEigenvalue(QPS qps, PetscReal maxeig_update);
PERMON_EXTERN PetscErrorCode QPSMPGPSetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal tol);
PERMON_EXTERN PetscErrorCode QPSMPGPGetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal *tol);
PERMON_EXTERN PetscErrorCode QPSMPGPGetOperatorMaxEigenvalueIterations(QPS qps, PetscInt *numit);
PERMON_EXTERN PetscErrorCode QPSMPGPSetOperatorMaxEigenvalueIterations(QPS qps, PetscInt numit);
/* the counters QPSViewConvergence_MPGP prints (mpgp.c:751-770): Hessian mults, CG / expansion / proportioning steps */
PERMON_EXTERN PetscErrorCode QPSMPGPGetStepCounts(QPS qps, PetscInt *nmv, PetscInt *ncg, PetscInt *nexp, PetscInt *nprop);

/* SMALXE: permonqps.h:143-165, src/qps/impls/smalxe/smalxe.c */
PERMON_EXTERN PetscErrorCode QPSSMALXEGetInnerQPS(QPS qps, QPS *inner);
PERMON_EXTERN PetscErrorCode QPSSMALXESetOperatorMaxEigenvalue(QPS qps, PetscReal maxeig);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalue(QPS qps, PetscReal *maxeig);
PERMON_EXTERN PetscErrorCode QPSSMALXESetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal tol);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalueTolerance(QPS qps, PetscReal *tol);
PERMON_EXTERN PetscErrorCode QPSSMALXESetOperatorMaxEigenvalueIterations(QPS qps, PetscInt numit);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetOperatorMaxEigenvalueIterations(QPS qps, PetscInt *numit);
PERMON_EXTERN PetscErrorCode QPSSMALXESetInjectOperatorMaxEigenvalue(QPS qps, PetscBool flg);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetInjectOperatorMaxEigenvalue(QPS qps, PetscBool *flg);
PERMON_EXTERN PetscErrorCode QPSSMALXESetEta(QPS qps, PetscReal eta, QPSScalarArgType argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetEta(QPS qps, PetscReal *eta, QPSScalarArgType *argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXESetM1Initial(QPS qps, PetscReal M1_initial, QPSScalarArgType argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetM1Initial(QPS qps, PetscReal *M1_initial, QPSScalarArgType *argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXESetM1Update(QPS qps, PetscReal M1_update);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetM1Update(QPS qps, PetscReal *M1_update);
PERMON_EXTERN PetscErrorCode QPSSMALXESetRhoInitial(QPS qps, PetscReal rho_initial, QPSScalarArgType argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetRhoInitial(QPS qps, PetscReal *rho_initial, QPSScalarArgType *argtype);
PERMON_EXTERN PetscErrorCode QPSSMALXESetRhoUpdate(QPS qps, PetscReal rho_update);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetRhoUpdate(QPS qps, PetscReal *rho_update);
PERMON_EXTERN PetscErrorCode QPSSMALXESetRhoUpdateLate(QPS qps, PetscReal rho_update_late);
PERMON_EXTERN PetscErrorCode QPSSMALXEGetRhoUpdateLate(QPS qps, PetscReal *rho_update_late);
PERMON_EXTERN PetscErrorCode QPSSMALXESetMonitor(QPS qps, PetscBool flg);
/* the counters QPSViewConvergence_SMALXE prints (smalxe.c:1001-1019) */
PERMON_EXTERN PetscErrorCode QPSSMALXEGetStatistics(QPS qps, PetscInt *inner_iter_accu, PetscInt *M1_hits, PetscInt *eta_hits, PetscInt *M1_updates, PetscInt *rho_updates);

#ifdef __cplusplus
}
#endif
#endif /* PERMON_B200_H */
