"""ctypes binding of libpermon_b200.so -- the C ABI declared in include/permon_b200.h.

This is a *binding*, not an implementation: every call goes straight to the shared library (PERMON's own
function names and argument order), which runs CUDA kernels on the B200.  There is no CPU fallback: if the
library is missing, or no CUDA device is present, the calls raise.

Typical use (mirrors src/tutorials/ex1.c of the reference):

    from permon_b200 import api as P
    P.initialize()
    A  = P.MatCreateAIJ(ia, ja, a, n)          # MatCreateSeqAIJWithArrays / MatCreateMPIAIJWithArrays
    b  = P.VecFromArray(b_np); x = P.VecFromArray(x_np); lb = P.VecFromArray(lb_np)
    qp = P.QPCreate(); P.QPSetOperator(qp, A); P.QPSetRhs(qp, b); P.QPSetInitialVector(qp, x); P.QPSetBox(qp, None, lb, None)
    qps = P.QPSCreate(); P.QPSSetQP(qps, qp); P.QPSSetFromOptions(qps); P.QPSSolve(qps)
    sol = P.VecGetArray(x)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBPATH = os.path.join(_HERE, "libpermon_b200.so")
_lib = None

DECIDE = -1
DEFAULT = -2
INFINITY = 1.7976931348623157e308 / 4.0
NINFINITY = -INFINITY
QPS_ARG_MULTIPLE, QPS_ARG_DIRECT = 0, 1

REASONS = {2: "CONVERGED_RTOL", 3: "CONVERGED_ATOL", 4: "CONVERGED_ITS", 7: "CONVERGED_HAPPY_BREAKDOWN",
           -3: "DIVERGED_ITS", -4: "DIVERGED_DTOL", -5: "DIVERGED_BREAKDOWN", -9: "DIVERGED_NANORINF", 0: "ITERATING"}


class PermonError(RuntimeError):
    def __init__(self, code, where, msg):
        super().__init__(f"{where} failed with PetscErrorCode {code}: {msg}")
        self.code = code


def _preload_nccl():
    """libpermon_b200.so needs libnccl.so.2.  In a Python process that also imports torch, the copy bundled with torch
    (nvidia/nccl/lib, newer than the system one) must be the one that gets loaded first, otherwise torch's own import
    fails on missing symbols.  A plain C host simply picks up the system libnccl.so.2."""
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia")
        for base in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
            if os.path.exists(cand):
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                return
    except Exception:
        pass


def lib():
    """Load the shared library (must have been built: python -m permon_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIBPATH):
            raise ImportError(f"{_LIBPATH} is missing -- build it with `python -m permon_b200.build` "
                              "(the product has no fallback implementation)")
        _preload_nccl()
        _lib = C.CDLL(_LIBPATH, mode=C.RTLD_GLOBAL)
        _lib.PermonB200GetLastErrorMessage.restype = C.c_char_p
    return _lib


def _chk(code, where):
    if code != 0:
        raise PermonError(code, where, lib().PermonB200GetLastErrorMessage().decode(errors="replace"))


def call(name, *args):
    f = getattr(lib(), name)
    f.restype = C.c_int
    _chk(f(*args), name)


def _h(obj):
    """handle -> c_void_p"""
    if obj is None:
        return C.c_void_p(None)
    return obj if isinstance(obj, C.c_void_p) else C.c_void_p(obj)


_keepalive = {}


def _keep(handle, *arrays):
    _keepalive.setdefault(handle.value, []).extend(arrays)


def world():
    return C.c_void_p.in_dll(lib(), "PETSC_COMM_WORLD")


def device_count() -> int:
    n = C.c_int()
    call("PermonB200GetDeviceCount", C.byref(n))
    return n.value


def initialize(options: str = ""):
    call("PermonInitialize", None, None, None, None)
    if options:
        call("PetscOptionsInsertString", None, options.encode())


def finalize():
    call("PermonFinalize")


def options_set(name, value=""):
    call("PetscOptionsSetValue", None, name.encode(), str(value).encode())


def options_clear():
    call("PetscOptionsClear", None)


def set_stream(ptr):
    call("PermonB200SetStream", C.c_void_p(ptr))


def get_stream() -> int:
    """the CUDA stream the library launches on (its own non-blocking stream unless PermonB200SetStream handed it another)"""
    s = C.c_void_p()
    call("PermonB200GetStream", C.byref(s))
    return int(s.value or 0)


def synchronize():
    call("PermonB200Synchronize")


def launch_count() -> int:
    n = C.c_int64()
    call("PermonB200GetLaunchCount", C.byref(n))
    return n.value


def profile_begin():
    call("PermonB200ProfileBegin")


def profile_end():
    n = C.c_int()
    call("PermonB200ProfileEnd", C.byref(n))
    out = {}
    for f in range(n.value):
        name, cnt, ms, bpl = C.c_char_p(), C.c_int64(), C.c_double(), C.c_double()
        call("PermonB200ProfileGet", C.c_int(f), C.byref(name), C.byref(cnt), C.byref(ms), C.byref(bpl))
        wn, wms = C.c_int64(), C.c_double()
        call("PermonB200ProfileGetWorking", C.c_int(f), C.byref(wn), C.byref(wms))
        out[name.value.decode()] = dict(launches=cnt.value, total_ms=ms.value, bytes_per_launch=bpl.value, working_launches=wn.value, working_ms=wms.value)
    return out


def comm_init_rank(nranks, rank, id_bytes: bytes | None):
    buf = C.create_string_buffer(id_bytes if id_bytes else b"\0" * 128, 128)
    call("PermonB200CommInitRank", C.c_int(nranks), C.c_int(rank), buf)


def get_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    call("PermonB200GetUniqueId", buf)
    return buf.raw


_AGI = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64))
_AGV = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_int64))
_host_exchange_refs = []


def comm_set_host_exchange(nranks, rank, allgather_i64, allgather_bytes):
    """Install Python callbacks (e.g. over torch.distributed/gloo) for the set-up-time host exchange."""
    def agi(_ctx, value, out):
        try:
            vals = allgather_i64(int(value))
            for r in range(nranks):
                out[r] = int(vals[r])
            return 0
        except Exception:  # pragma: no cover
            import traceback
            traceback.print_exc()
            return 1

    def agv(_ctx, send, sendbytes, recv, recvbytes):
        try:
            data = C.string_at(send, sendbytes) if sendbytes else b""
            parts = allgather_bytes(data)
            off = 0
            for r in range(nranks):
                assert len(parts[r]) == recvbytes[r]
                C.memmove(recv + off, parts[r], len(parts[r]))
                off += len(parts[r])
            return 0
        except Exception:  # pragma: no cover
            import traceback
            traceback.print_exc()
            return 1

    a, b = _AGI(agi), _AGV(agv)
    _host_exchange_refs.extend([a, b])
    call("PermonB200CommSetHostExchange", C.c_int(nranks), C.c_int(rank), a, b, None)


# ---- Vec ---------------------------------------------------------------------------------------------
def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _iptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def VecFromArray(arr, N=DECIDE, comm=None):
    """VecCreate{Seq,MPI}WithArray: `arr` (float64, contiguous) is the host storage of the Vec."""
    assert arr.dtype == np.float64 and arr.flags.c_contiguous
    v = C.c_void_p()
    call("VecCreateMPIWithArray", comm or world(), C.c_int(1), C.c_int(arr.shape[0]), C.c_int(N), _dptr(arr), C.byref(v))
    _keep(v, arr)
    return v


def VecFromDevicePointer(ptr, n, N=DECIDE, comm=None, keep=None):
    v = C.c_void_p()
    call("VecCreateMPICUDAWithArray", comm or world(), C.c_int(1), C.c_int(n), C.c_int(N), C.c_void_p(ptr), C.byref(v))
    if keep is not None:
        _keep(v, keep)
    return v


def VecCreate(n, N=DECIDE, comm=None):
    v = C.c_void_p()
    call("VecCreateMPI", comm or world(), C.c_int(n), C.c_int(N), C.byref(v))
    return v


def VecDuplicate(v):
    w = C.c_void_p()
    call("VecDuplicate", v, C.byref(w))
    return w


def VecDestroy(v):
    _keepalive.pop(v.value, None)
    call("VecDestroy", C.byref(v))


def VecGetLocalSize(v) -> int:
    n = C.c_int()
    call("VecGetLocalSize", v, C.byref(n))
    return n.value


def VecGetArray(v) -> np.ndarray:
    """Copy of the current contents (downloads from the device when the device copy is newer)."""
    n = VecGetLocalSize(v)
    p = C.POINTER(C.c_double)()
    call("VecGetArrayRead", v, C.byref(p))
    out = np.ctypeslib.as_array(p, shape=(n,)).copy() if n else np.zeros(0)
    call("VecRestoreArrayRead", v, C.byref(p))
    return out


def VecSyncToHost(v):
    """VecGetArrayRead + Restore without a copy: the current contents land in the host buffer the Vec was created over
    (VecCreate*WithArray semantics: the user's array is the storage)."""
    p = C.POINTER(C.c_double)()
    call("VecGetArrayRead", v, C.byref(p))
    call("VecRestoreArrayRead", v, C.byref(p))


def VecSetArray(v, arr):
    n = VecGetLocalSize(v)
    p = C.POINTER(C.c_double)()
    call("VecGetArray", v, C.byref(p))
    np.ctypeslib.as_array(p, shape=(n,))[:] = arr
    call("VecRestoreArray", v, C.byref(p))


def VecCUDAGetArrayRead(v) -> int:
    p = C.c_void_p()
    call("VecCUDAGetArrayRead", v, C.byref(p))
    return p.value


def VecSet(v, a):
    call("VecSet", v, C.c_double(a))


def VecCopy(x, y):
    call("VecCopy", x, y)


def VecAXPY(y, a, x):
    call("VecAXPY", y, C.c_double(a), x)


def VecDot(x, y) -> float:
    d = C.c_double()
    call("VecDot", x, y, C.byref(d))
    return d.value


def VecNorm(x) -> float:
    d = C.c_double()
    call("VecNorm", x, C.c_int(1), C.byref(d))
    return d.value


def VecIsInvalidated(v) -> bool:
    f = C.c_int()
    call("VecIsInvalidated", v, C.byref(f))
    return bool(f.value)


# ---- IS / Mat -------------------------------------------------------------------------------------------
def ISCreateGeneral(idx, comm=None):
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    s = C.c_void_p()
    call("ISCreateGeneral", comm or world(), C.c_int(len(idx)), _iptr(idx), C.c_int(0), C.byref(s))
    return s


def ISDestroy(s):
    call("ISDestroy", C.byref(s))


def MatCreateAIJ(ia, ja, a, ncols_local=None, comm=None):
    """MatCreateMPIAIJWithArrays: local rows in CSR with GLOBAL column indices (copied to the device)."""
    ia = np.ascontiguousarray(ia, dtype=np.int32)
    ja = np.ascontiguousarray(ja, dtype=np.int32)
    a = np.ascontiguousarray(a, dtype=np.float64)
    m = len(ia) - 1
    n = m if ncols_local is None else ncols_local
    A = C.c_void_p()
    call("MatCreateMPIAIJWithArrays", comm or world(), C.c_int(m), C.c_int(n), C.c_int(DECIDE), C.c_int(DECIDE), _iptr(ia), _iptr(ja), _dptr(a), C.byref(A))
    return A


def MatCreateAIJFromDevicePointers(m, n, dia, dja, da, keep=None, comm=None):
    A = C.c_void_p()
    call("MatCreateSeqAIJCUSPARSEWithArrays", comm or world(), C.c_int(m), C.c_int(n), C.c_void_p(dia), C.c_void_p(dja), C.c_void_p(da), C.byref(A))
    if keep is not None:
        _keep(A, keep)
    return A


def MatCreateAIJFromDeviceTensors(ia, ja, a, ncols_local=None, comm=None):
    """MatB200CreateAIJWithDeviceArrays: local rows in CSR with GLOBAL column indices, as torch CUDA tensors (int32 / int32 / float64,
    contiguous) on the library's device.  The matrix is re-coded on the GPU into the form MatCreateAIJ builds; the tensors are not kept
    and may be freed or overwritten when the call returns."""
    import torch
    for t, dt, name in ((ia, torch.int32, "ia"), (ja, torch.int32, "ja"), (a, torch.float64, "a")):
        if not isinstance(t, torch.Tensor) or t.device.type != "cuda":
            raise TypeError(f"{name}: a torch CUDA tensor is required")
        if t.dtype != dt or not t.is_contiguous() or t.dim() != 1:
            raise TypeError(f"{name}: a contiguous 1-D {dt} tensor is required (got {t.dtype}, shape {tuple(t.shape)})")
    m = ia.numel() - 1
    n = m if ncols_local is None else ncols_local
    # the tensors were written on torch's current stream: the library reads them on its own stream
    torch.cuda.current_stream(ia.device).synchronize()
    A = C.c_void_p()
    call("MatB200CreateAIJWithDeviceArrays", comm or world(), C.c_int(m), C.c_int(n), C.c_int(DECIDE), C.c_int(DECIDE),
         C.c_void_p(ia.data_ptr()), C.c_void_p(ja.data_ptr() if ja.numel() else None), C.c_void_p(a.data_ptr() if a.numel() else None), C.byref(A))
    return A


def _colmajor_lda(shape, strides):
    """leading dimension (in elements) when a 2-D array with these element strides is column-major with lda >= m, else None"""
    m, n = shape
    if m > 1 and strides[0] != 1:
        return None
    lda = strides[1] if n > 1 else max(m, 1)
    return lda if lda >= max(m, 1) else None


def MatCreateDense(arr, comm=None):
    """MatCreateSeqDense (MatCreateDense on one rank): a 2-D float64 NumPy array in any order.  A column-major array (or a column-major view
    with a leading dimension, e.g. big[:m, :] of a Fortran-ordered big) is handed over as it is, anything else is copied column-major first.
    The library uploads it at the first use; the array is kept alive with the matrix."""
    arr = np.asarray(arr, dtype=np.float64)
    if arr.ndim != 2:
        raise ValueError(f"a 2-D array is required (got shape {arr.shape})")
    lda = _colmajor_lda(arr.shape, tuple(s // 8 for s in arr.strides)) if all(s % 8 == 0 and s >= 0 for s in arr.strides) else None
    if lda is None:
        arr = np.asfortranarray(arr)
        lda = max(arr.shape[0], 1)
    m, n = arr.shape
    A = C.c_void_p()
    call("MatCreateDense", comm or world(), C.c_int(m), C.c_int(n), C.c_int(DECIDE), C.c_int(DECIDE), C.c_void_p(arr.ctypes.data), C.byref(A))
    _keep(A, arr)
    if lda != max(m, 1):
        call("MatDenseSetLDA", A, C.c_int(lda))
    return A


def MatCreateDenseFromTensor(t, comm=None):
    """MatCreateSeqDenseCUDA from a 2-D torch CUDA float64 tensor on the library's device.  A column-major tensor (stride(0) == 1, stride(1)
    = lda >= m) is adopted without a copy when its base is 16-byte aligned and lda is even: every product reads the tensor, so in-place
    changes show in the next MatMult.  Otherwise one column-major device copy is made here and handed over instead.  A symmetric Hessian
    in row-major order is already its own column-major form: pass H.T (a view) to have it adopted.  The tensor is kept alive with the
    matrix."""
    import torch
    if not isinstance(t, torch.Tensor) or t.device.type != "cuda" or t.dtype != torch.float64 or t.dim() != 2:
        raise TypeError("a 2-D torch CUDA float64 tensor is required")
    lda = _colmajor_lda(tuple(t.shape), t.stride())
    if lda is None:
        t = t.t().contiguous().t()
        lda = max(t.shape[0], 1)
    m, n = t.shape
    # the tensor was written on torch's current stream: the library reads it on its own stream
    torch.cuda.current_stream(t.device).synchronize()
    A = C.c_void_p()
    call("MatCreateSeqDenseCUDA", comm or world(), C.c_int(m), C.c_int(n), C.c_void_p(t.data_ptr()), C.byref(A))
    _keep(A, t)
    if lda != max(m, 1):
        call("MatDenseSetLDA", A, C.c_int(lda))
    return A


def MatDenseGetLDA(A) -> int:
    lda = C.c_int()
    call("MatDenseGetLDA", A, C.byref(lda))
    return lda.value


def MatDenseGetInfo(A):
    """MatB200GetDenseInfo: leading dimension the kernels read with, whether the caller's device array is read in place, rows per CTA,
    column chunk of the split-column variant (0: one thread per row)"""
    lda, adopted, rpb, split = C.c_int64(), C.c_int(), C.c_int(), C.c_int()
    call("MatB200GetDenseInfo", A, C.byref(lda), C.byref(adopted), C.byref(rpb), C.byref(split))
    return dict(lda=lda.value, adopted=bool(adopted.value), rows_per_block=rpb.value, split_columns=split.value)


FORM_PARTS = {"scalars": 0, "st_masks": 1, "st_pid": 2, "st_pats": 3, "pk_blob": 4, "pk_off": 5, "csr_ia": 6, "csr_ja": 7, "csr_a": 8,
              "ell_val": 9, "ell_col": 10, "ell_len": 11, "ell_lt": 12, "ell_off": 13, "rows": 14}
FORM_OFFDIAG = 16
FORM_SCALARS = ("kind", "n", "ncols", "nnz", "st_npat", "st_nwin", "st_lmax", "st_dlo", "st_dhi", "pk_max", "pk_bytes", "pk_coded", "stages",
                "tile_cap", "W")


def MatGetStoredForm(A, offdiag=False):
    """MatB200GetStoredForm: every part of the stored form of the diagonal (or off-diagonal) block as bytes, plus the scalar fields"""
    out = {}
    for name, part in FORM_PARTS.items():
        part += FORM_OFFDIAG if offdiag else 0
        nb = C.c_size_t()
        call("MatB200GetStoredForm", A, C.c_int(part), None, C.byref(nb))
        buf = C.create_string_buffer(max(nb.value, 1))
        call("MatB200GetStoredForm", A, C.c_int(part), buf, C.byref(nb))
        out[name] = buf.raw[:nb.value]
    out["fields"] = dict(zip(FORM_SCALARS, np.frombuffer(out["scalars"], dtype=np.int64).tolist()))
    return out


def MatCreateOneRow(vec):
    A = C.c_void_p()
    call("MatCreateOneRow", vec, C.byref(A))
    return A


def MatCreateProd(mats, comm=None):
    arr = (C.c_void_p * len(mats))(*[m.value for m in mats])
    A = C.c_void_p()
    call("MatCreateProd", comm or world(), C.c_int(len(mats)), arr, C.byref(A))
    return A


def MatDestroy(A):
    _keepalive.pop(A.value, None)
    call("MatDestroy", C.byref(A))


def MatMult(A, x, y):
    call("MatMult", A, x, y)


def MatGetMaxEigenvalue(A, tol=DECIDE, maxits=DECIDE) -> float:
    lam = C.c_double()
    call("MatGetMaxEigenvalue", A, None, C.byref(lam), C.c_double(tol), C.c_int(maxits))
    return lam.value


def MatGetHaloInfo(A):
    ng, nn, nb = C.c_int(), C.c_int(), C.c_int()
    ga, nr, ro, so, si = (C.POINTER(C.c_int32)() for _ in range(5))
    call("MatB200GetHaloInfo", A, C.byref(ng), C.byref(ga), C.byref(nn), C.byref(nr), C.byref(ro), C.byref(so), C.byref(si), C.byref(nb))
    k = nn.value
    send_off = [so[i] for i in range(k + 1)] if k else [0]
    return dict(garray=[ga[i] for i in range(ng.value)], neigh=[nr[i] for i in range(k)],
                recv_off=[ro[i] for i in range(k + 1)] if k else [0], send_off=send_off,
                send_idx=[si[i] for i in range(send_off[-1])], nboundary=nb.value)


def MatGetHostSplit(A, m):
    """(dia, dja, da, oia, oja, oa, orow) of a row-partitioned matrix that has not been used on the device yet (copies)"""
    pi = lambda: C.POINTER(C.c_int32)()
    dia, dja, oia, oja, orow = pi(), pi(), pi(), pi(), pi()
    da, oa = C.POINTER(C.c_double)(), C.POINTER(C.c_double)()
    no = C.c_int()
    call("MatB200GetHostSplit", A, C.byref(dia), C.byref(dja), C.byref(da), C.byref(no), C.byref(oia), C.byref(oja), C.byref(oa), C.byref(orow))
    arr = lambda p, k, t: np.ctypeslib.as_array(p, shape=(k,)).astype(t).copy() if k else np.zeros(0, dtype=t)
    dia_ = arr(dia, m + 1, np.int64)
    oia_ = arr(oia, no.value + 1, np.int64)
    return (dia_, arr(dja, int(dia_[-1]), np.int64), arr(da, int(dia_[-1]), np.float64), oia_, arr(oja, int(oia_[-1]), np.int64),
            arr(oa, int(oia_[-1]), np.float64), arr(orow, no.value, np.int64))


def MatStorageInfo(A):
    """Device storage of an AIJ or dense matrix: kind (3 = packed dictionary-coded tiles, 6 = dense), matrix bytes streamed per SpMV, coded / all
    tiles (dense: row blocks)."""
    kind, coded, tiles = C.c_int(), C.c_int(), C.c_int()
    nbytes = C.c_double()
    call("MatB200GetStorageInfo", A, C.byref(kind), C.byref(nbytes), C.byref(coded), C.byref(tiles))
    return dict(kind=kind.value, stream_bytes=nbytes.value, coded_tiles=coded.value, tiles=tiles.value)


# ---- QPC ---------------------------------------------------------------------------------------------
def QPCCreateBox(is_, lb, ub, comm=None):
    q = C.c_void_p()
    call("QPCCreateBox", comm or world(), _h(is_), _h(lb), _h(ub), C.byref(q))
    return q


def QPCDestroy(q):
    call("QPCDestroy", C.byref(q))


def QPCProject(q, x, Px):
    call("QPCProject", q, x, Px)


def QPCGrads(q, x, g, gf, gc):
    call("QPCGrads", q, x, g, gf, gc)


def QPCGradReduced(q, x, gf, alpha, gr):
    call("QPCGradReduced", q, x, gf, C.c_double(alpha), gr)


def QPCFeas(q, x, d) -> float:
    a = C.c_double()
    call("QPCFeas", q, x, d, C.byref(a))
    return a.value


def QPCBoxGetMultipliers(q):
    a, b = C.c_void_p(), C.c_void_p()
    call("QPCBoxGetMultipliers", q, C.byref(a), C.byref(b))
    return (a if a.value else None), (b if b.value else None)


# ---- QP ----------------------------------------------------------------------------------------------
def QPCreate(comm=None):
    q = C.c_void_p()
    call("QPCreate", comm or world(), C.byref(q))
    return q


def QPDestroy(q):
    call("QPDestroy", C.byref(q))


def QPSetOperator(qp, A):
    call("QPSetOperator", qp, A)


def QPSetRhs(qp, b):
    call("QPSetRhs", qp, b)


def QPSetRhsPlus(qp, b):
    call("QPSetRhsPlus", qp, b)


def QPSetInitialVector(qp, x):
    call("QPSetInitialVector", qp, x)


def QPSetBox(qp, is_, lb, ub):
    call("QPSetBox", qp, _h(is_), _h(lb), _h(ub))


def QPSetEq(qp, B, c):
    call("QPSetEq", qp, _h(B), _h(c))


MAT_ORTH = dict(none=0, gs=1, gslingen=2, cholesky=3, implicit=4, inexact=5)


def QPTOrthonormalizeEq(qp, kind="gs", explicit=True):
    call("QPTOrthonormalizeEq", qp, C.c_int(MAT_ORTH[kind]), C.c_int(1 if explicit else 0))


def QPTEnforceEqByProjector(qp):
    call("QPTEnforceEqByProjector", qp)


def QPTHomogenizeEq(qp):
    call("QPTHomogenizeEq", qp)


def QPChainGetLast(qp):
    c = C.c_void_p()
    call("QPChainGetLast", qp, C.byref(c))
    return c


def QPSetOptionsPrefix(qp, prefix):
    call("QPSetOptionsPrefix", qp, prefix.encode())


def QPGetSolutionVector(qp):
    v = C.c_void_p()
    call("QPGetSolutionVector", qp, C.byref(v))
    return v


def QPGetQPC(qp):
    v = C.c_void_p()
    call("QPGetQPC", qp, C.byref(v))
    return v if v.value else None


def QPGetEqMultiplier(qp):
    a, b = C.c_void_p(), C.c_void_p()
    call("QPGetEqMultiplier", qp, C.byref(a), C.byref(b))
    return (a if a.value else None), (b if b.value else None)


def QPIsSolved(qp) -> bool:
    f = C.c_int()
    call("QPIsSolved", qp, C.byref(f))
    return bool(f.value)


def QPSetUp(qp):
    call("QPSetUp", qp)


def QPComputeObjective(qp, x) -> float:
    f = C.c_double()
    call("QPComputeObjective", qp, x, C.byref(f))
    return f.value


def QPChainViewKKT(qp, viewer=None):
    call("QPChainViewKKT", qp, _h(viewer))


# ---- QPS ---------------------------------------------------------------------------------------------
def QPSCreate(comm=None):
    q = C.c_void_p()
    call("QPSCreate", comm or world(), C.byref(q))
    return q


def QPSDestroy(q):
    call("QPSDestroy", C.byref(q))


def QPSSetType(qps, t):
    call("QPSSetType", qps, t.encode())


def QPSGetType(qps) -> str:
    t = C.c_char_p()
    call("QPSGetType", qps, C.byref(t))
    return t.value.decode()


def QPSSetQP(qps, qp):
    call("QPSSetQP", qps, qp)


def QPSSetFromOptions(qps):
    call("QPSSetFromOptions", qps)


def QPSSetOptionsPrefix(qps, prefix):
    call("QPSSetOptionsPrefix", qps, prefix.encode())


def QPSSetTolerances(qps, rtol=DEFAULT, atol=DEFAULT, dtol=DEFAULT, maxits=DEFAULT):
    call("QPSSetTolerances", qps, C.c_double(rtol), C.c_double(atol), C.c_double(dtol), C.c_int(maxits))


def QPSSetUp(qps):
    call("QPSSetUp", qps)


def QPSSolve(qps):
    call("QPSSolve", qps)


def QPSSetAutoPostSolve(qps, flg):
    call("QPSSetAutoPostSolve", qps, C.c_int(1 if flg else 0))


def QPSPostSolve(qps):
    call("QPSPostSolve", qps)


def QPSGetConvergedReason(qps) -> int:
    r = C.c_int()
    call("QPSGetConvergedReason", qps, C.byref(r))
    return r.value


def QPSGetIterationNumber(qps) -> int:
    r = C.c_int()
    call("QPSGetIterationNumber", qps, C.byref(r))
    return r.value


def QPSGetResidualNorm(qps) -> float:
    r = C.c_double()
    call("QPSGetResidualNorm", qps, C.byref(r))
    return r.value


def QPSViewConvergence(qps, viewer=None):
    call("QPSViewConvergence", qps, _h(viewer))


_MONITOR = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p)
_monitor_refs = []


def QPSMonitorSet(qps, fn):
    """fn(qps_handle, it, rnorm) -> None"""
    def tramp(q, it, rnorm, _ctx):
        fn(C.c_void_p(q), it, rnorm)
        return 0
    cb = _MONITOR(tramp)
    _monitor_refs.append(cb)
    call("QPSMonitorSet", qps, cb, None, None)


def QPSMonitorDefault():
    return C.cast(lib().QPSMonitorDefault, C.c_void_p)


def QPSMonitorSetDefault(qps, viewer=None):
    call("QPSMonitorSet", qps, C.cast(lib().QPSMonitorDefault, _MONITOR), _h(viewer), None)


def PetscViewerASCIIOpen(path, comm=None):
    v = C.c_void_p()
    call("PetscViewerASCIIOpen", comm or world(), path.encode(), C.byref(v))
    return v


def PetscViewerDestroy(v):
    call("PetscViewerDestroy", C.byref(v))


def QPSMPGPGetStepCounts(qps):
    a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    call("QPSMPGPGetStepCounts", qps, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    return dict(nmv=a.value, ncg=b.value, nexp=c.value, nprop=d.value)


def QPSMPGPGetCurrentStepType(qps) -> str:
    ch = C.c_char()
    call("QPSMPGPGetCurrentStepType", qps, C.byref(ch))
    return ch.value.decode()


def QPSMPGPGetAlpha(qps):
    a, t = C.c_double(), C.c_int()
    call("QPSMPGPGetAlpha", qps, C.byref(a), C.byref(t))
    return a.value, t.value


def QPSMPGPGetOperatorMaxEigenvalue(qps) -> float:
    a = C.c_double()
    call("QPSMPGPGetOperatorMaxEigenvalue", qps, C.byref(a))
    return a.value


def QPSMPGPSetOperatorMaxEigenvalue(qps, v):
    call("QPSMPGPSetOperatorMaxEigenvalue", qps, C.c_double(v))


def QPSSMALXEGetInnerQPS(qps):
    q = C.c_void_p()
    call("QPSSMALXEGetInnerQPS", qps, C.byref(q))
    return q


def QPSSMALXEGetStatistics(qps):
    v = [C.c_int() for _ in range(5)]
    call("QPSSMALXEGetStatistics", qps, *[C.byref(x) for x in v])
    return dict(inner_iter_accu=v[0].value, M1_hits=v[1].value, eta_hits=v[2].value, M1_updates=v[3].value, rho_updates=v[4].value)


# ---- convenience used by tests / bench ---------------------------------------------------------------------
class Solved:
    pass


def solve_problem(pr, qps_type=None, options: str = "", monitor=None, keep=False, device_arrays=None, device_input=None, dense=False):
    """Build QP + QPS for a permon_b200.problems.QPProblem through the C ABI, solve, return a result object.

    `options` is a PETSc-style option string ("-qps_rtol 1e-8 -qps_mpgp_expansion_type gf ...").
    `device_input`: "keep" builds the AIJ matrices from torch CUDA tensors (MatCreateAIJFromDeviceTensors), "zero" does the same and
    zeroes the tensors right after each constructor returns.
    `dense`: the Hessian (both factors of a product Hessian) is built as a dense matrix from the problem's CSR (MatCreateDense)."""
    if device_input:
        import torch

        def MatCreateAIJ(ia, ja, a, ncols_local=None):
            t = [torch.as_tensor(np.ascontiguousarray(v, dtype=dt)).cuda() for v, dt in ((ia, np.int32), (ja, np.int32), (a, np.float64))]
            M = MatCreateAIJFromDeviceTensors(*t, ncols_local=ncols_local)
            if device_input == "zero":
                for v in t:
                    v.zero_()
                torch.cuda.synchronize()
            return M
    else:
        MatCreateAIJ = globals()["MatCreateAIJ"]
    MatCreateH = MatCreateAIJ
    if dense:
        import scipy.sparse as sp

        def MatCreateH(ia, ja, a, ncols_local=None):
            return MatCreateDense(sp.csr_matrix((a, ja, ia), shape=(len(ia) - 1, ncols_local)).toarray(order="F"))
    options_clear()
    if options:
        call("PetscOptionsInsertString", None, options.encode())
    r = Solved()
    x_host = np.ascontiguousarray(pr.x0, dtype=np.float64).copy()
    b_host = np.ascontiguousarray(pr.b, dtype=np.float64)
    ncols = pr.n
    A1 = MatCreateH(pr.ia, pr.ja, pr.a, ncols_local=(pr.meta.get("d") if pr.second is not None else ncols))
    mats = [A1]
    A = A1
    if pr.second is not None:
        A2 = MatCreateH(pr.second[0], pr.second[1], pr.second[2], ncols_local=pr.n)
        A = MatCreateProd([A2, A1])   # product = mats[1]*mats[0] = A1 * A2
        mats += [A2, A]
    b = VecFromArray(b_host)
    x = VecFromArray(x_host)
    lb = VecFromArray(np.ascontiguousarray(pr.lb, dtype=np.float64)) if pr.lb is not None else None
    ub = VecFromArray(np.ascontiguousarray(pr.ub, dtype=np.float64)) if pr.ub is not None else None
    is_ = ISCreateGeneral(pr.is_) if pr.is_ is not None else None
    qp = QPCreate()
    QPSetOperator(qp, A)
    QPSetRhs(qp, b)
    QPSetInitialVector(qp, x)
    QPSetBox(qp, is_, lb, ub)
    extra = []
    if getattr(pr, "BE_local", None) is not None:
        # row-partitioned AIJ equality matrix, the way a PETSc user assembles B_E: this rank's rows in CSR with GLOBAL column indices
        # (pr.BE_local = (ia, ja, a)), pr.c = this rank's entries of c_E
        BE = MatCreateAIJ(pr.BE_local[0], pr.BE_local[1], pr.BE_local[2], ncols_local=pr.n)
        cE = VecFromArray(np.ascontiguousarray(pr.c, dtype=np.float64)) if pr.c is not None else None
        QPSetEq(qp, BE, cE)
        mats.append(BE)
        if cE is not None:
            extra.append(cE)
    elif pr.B is not None:
        Bm = np.ascontiguousarray(pr.B, dtype=np.float64)
        if Bm.shape[0] == 1:
            brow = VecFromArray(Bm[0].copy())
            BE = MatCreateOneRow(brow)
            extra += [brow]
        else:
            import scipy.sparse as sp
            S = sp.csr_matrix(Bm)
            BE = MatCreateAIJ(S.indptr, S.indices, S.data, ncols_local=pr.n)
        cE = VecFromArray(np.ascontiguousarray(pr.c, dtype=np.float64)) if pr.c is not None else None
        QPSetEq(qp, BE, cE)
        mats.append(BE)
        if cE is not None:
            extra.append(cE)
    for t in getattr(pr, "transforms", ()):     # QP transforms applied before the solver sees the chain (QPT*, qptransform.c)
        if t.startswith("orth_"):
            QPTOrthonormalizeEq(qp, t[len("orth_"):])
        elif t == "projector":
            QPTEnforceEqByProjector(qp)
        else:
            raise ValueError(t)
    qps = QPSCreate()
    if qps_type:
        QPSSetType(qps, qps_type)
    QPSSetQP(qps, qp)
    QPSSetFromOptions(qps)
    if monitor is not None:
        QPSMonitorSet(qps, monitor)
    QPSSolve(qps)
    r.x = VecGetArray(x)
    r.its = QPSGetIterationNumber(qps)
    r.reason = QPSGetConvergedReason(qps)
    r.rnorm = QPSGetResidualNorm(qps)
    r.solved = QPIsSolved(qp)
    r.objective = QPComputeObjective(qp, x)
    qpc = QPGetQPC(qp)
    llb, lub = QPCBoxGetMultipliers(qpc)
    r.llb = VecGetArray(llb) if (llb is not None and not VecIsInvalidated(llb)) else None
    r.lub = VecGetArray(lub) if (lub is not None and not VecIsInvalidated(lub)) else None
    if pr.B is None and getattr(pr, "BE_local", None) is None:
        r.counts = QPSMPGPGetStepCounts(qps)
        r.alpha_user, _ = QPSMPGPGetAlpha(qps)
        r.maxeig = QPSMPGPGetOperatorMaxEigenvalue(qps)
        r.step = QPSMPGPGetCurrentStepType(qps)
    else:
        inner = QPSSMALXEGetInnerQPS(qps)
        r.counts = QPSMPGPGetStepCounts(inner)
        r.stats = QPSSMALXEGetStatistics(qps)
        r.inner_reason = QPSGetConvergedReason(inner)
        r.maxeig_inner = QPSMPGPGetOperatorMaxEigenvalue(inner)
        lamE, Btl = QPGetEqMultiplier(qp)
        r.Bt_lambda = VecGetArray(Btl) if (Btl is not None and not VecIsInvalidated(Btl)) else None
    if keep:
        r.handles = dict(qps=qps, qp=qp, x=x, b=b, lb=lb, ub=ub, mats=mats, extra=extra)
        return r
    QPSDestroy(qps)
    QPDestroy(qp)
    for v in [x, b, lb, ub] + extra:
        if v is not None:
            VecDestroy(v)
    if is_ is not None:
        ISDestroy(is_)
    for m in reversed(mats):
        MatDestroy(m)
    return r
