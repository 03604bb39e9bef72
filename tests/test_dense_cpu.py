"""CPU-side checks of the dense-matrix interface (MatCreateSeqDense / MatCreateSeqDenseCUDA / MatCreateDense, MatDenseSetLDA /
MatDenseGetLDA, MatB200GetDenseInfo): the symbols are declared and exported, argument errors come back with PETSc's codes before any
device work, and a dense matrix on more than one rank is refused."""
import ctypes as C
import os
import re
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "permon_b200.h")
DENSE_SYMBOLS = ("MatCreateSeqDense", "MatCreateSeqDenseCUDA", "MatCreateDense", "MatDenseSetLDA", "MatDenseGetLDA", "MatB200GetDenseInfo")
ERR_SUP, ERR_ARG_WRONG, ERR_OUTOFRANGE, ERR_ARG_NULL = 56, 62, 63, 85


@pytest.fixture(scope="module")
def P():
    from permon_b200 import build
    build.build()
    from permon_b200 import api
    api.lib()
    api.initialize()
    return api


def _code(P, name, *args):
    f = getattr(P.lib(), name)
    f.restype = C.c_int
    return f(*args)


def test_dense_symbols_declared_and_exported(P):
    text = open(HEADER).read()
    for name in DENSE_SYMBOLS:
        assert re.search(r"^PERMON_EXTERN PetscErrorCode " + name + r"\(", text, flags=re.M), name
        assert hasattr(P.lib(), name), name


def test_argument_errors(P):
    A = C.c_void_p()
    w = P.world()
    data = np.zeros((4, 3), order="F")
    ptr = C.c_void_p(data.ctypes.data)
    assert _code(P, "MatCreateSeqDense", w, C.c_int(4), C.c_int(3), C.c_void_p(None), C.byref(A)) == ERR_ARG_NULL
    assert _code(P, "MatCreateSeqDenseCUDA", w, C.c_int(4), C.c_int(3), C.c_void_p(None), C.byref(A)) == ERR_ARG_NULL
    assert _code(P, "MatCreateSeqDense", w, C.c_int(-1), C.c_int(3), ptr, C.byref(A)) == ERR_OUTOFRANGE
    assert _code(P, "MatCreateSeqDense", w, C.c_int(4), C.c_int(-3), ptr, C.byref(A)) == ERR_OUTOFRANGE
    assert _code(P, "MatCreateDense", w, C.c_int(4), C.c_int(3), C.c_int(P.DECIDE), C.c_int(P.DECIDE), ptr, C.byref(A)) == 0
    assert P.MatDenseGetLDA(A) == 4
    assert _code(P, "MatDenseSetLDA", A, C.c_int(3)) == ERR_OUTOFRANGE
    assert _code(P, "MatDenseSetLDA", A, C.c_int(6)) == 0
    assert P.MatDenseGetLDA(A) == 6
    P.MatDestroy(A)
    # the dense-only calls refuse other matrices
    vrow = P.VecFromArray(np.ones(3))
    R = P.MatCreateOneRow(vrow)
    assert _code(P, "MatDenseSetLDA", R, C.c_int(3)) == ERR_ARG_WRONG
    assert _code(P, "MatB200GetDenseInfo", R, None, None, None, None) == ERR_ARG_WRONG
    P.MatDestroy(R)
    P.VecDestroy(vrow)


def test_python_wrapper_passes_layout(P):
    """MatCreateDense hands a column-major view over as it is (lda = its column stride) and copies anything else column-major"""
    big = np.asfortranarray(np.arange(7.0 * 5).reshape(7, 5))
    A = P.MatCreateDense(big[:4, :])
    assert P.MatDenseGetLDA(A) == 7
    P.MatDestroy(A)
    A = P.MatCreateDense(np.arange(12.0).reshape(4, 3))      # row-major: copied
    assert P.MatDenseGetLDA(A) == 4
    P.MatDestroy(A)
    with pytest.raises(ValueError):
        P.MatCreateDense(np.zeros(5))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, size, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    from permon_b200 import api as P

    def agi(v):
        out = [None] * size
        dist.all_gather_object(out, int(v))
        return out

    def agv(data):
        out = [None] * size
        dist.all_gather_object(out, bytes(data))
        return out

    P.initialize()
    P.comm_set_host_exchange(size, rank, agi, agv)
    data = np.ones((3, 8), order="F")
    A = C.c_void_p()
    code = _code(P, "MatCreateDense", P.world(), C.c_int(3), C.c_int(8), C.c_int(P.DECIDE), C.c_int(P.DECIDE), C.c_void_p(data.ctypes.data), C.byref(A))
    msg = P.lib().PermonB200GetLastErrorMessage().decode()
    code_seq = _code(P, "MatCreateSeqDense", P.world(), C.c_int(3), C.c_int(8), C.c_void_p(data.ctypes.data), C.byref(A))
    dist.barrier()
    dist.destroy_process_group()
    ret[rank] = (code, code_seq, msg)


def test_dense_on_two_ranks_is_refused():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    mgr = ctx.Manager()
    ret = mgr.dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=240)
    for p in procs:
        if p.is_alive():
            p.kill()
            pytest.fail("worker hung")
        assert p.exitcode == 0
    for r in range(2):
        code, code_seq, msg = ret[r]
        assert code == ERR_SUP and code_seq == ERR_SUP, (code, code_seq)
        assert "one rank" in msg
