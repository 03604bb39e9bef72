"""MatB200CreateAIJWithDeviceArrays: a CSR that already lives on the GPU, re-coded on the GPU (recode.cu).

The host constructor's stored forms are pinned by test_pack_cpu.py and the parity suites, so the device constructor is held to
BYTE equality with it: every part of MatB200GetStoredForm, MatB200GetStorageInfo, MatMult bit for bit, and whole solves with identical
iteration counts and bit-identical iterates."""
import dataclasses
import os
import socket
import sys

import ctypes as C
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

ENVS = {
    "default": {},
    "no_pack_stencil": {"PERMON_B200_PACK_STENCIL": "0"},
    "no_st_windows": {"PERMON_B200_ST_WINDOWS": "0"},
    "spmv_tma": {"PERMON_B200_SPMV": "tma"},
    "noell": {"PERMON_B200_NOELL": "1"},
}


@pytest.fixture(scope="module")
def P():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from permon_b200 import api
    api.initialize()
    return api


def _csr(rows, ncols=None):
    """rows: list of (cols, vals) -> ia, ja, a"""
    ia = np.zeros(len(rows) + 1, np.int64)
    for r, (c, _) in enumerate(rows):
        ia[r + 1] = ia[r] + len(c)
    ja = np.concatenate([np.asarray(c, np.int64) for c, _ in rows]) if ia[-1] else np.zeros(0, np.int64)
    a = np.concatenate([np.asarray(v, np.float64) for _, v in rows]) if ia[-1] else np.zeros(0)
    return ia, ja, a


def lap2d(N):
    from permon_b200 import problems as PR
    pr = PR.obstacle2d(N)
    return pr.ia, pr.ja, pr.a, None


def lap3d(N):
    from permon_b200 import problems as PR
    pr = PR.obstacle3d(N)
    return pr.ia, pr.ja, pr.a, None


def varcoef(N):
    from permon_b200 import problems as PR
    pr = PR.varcoef3d(N)
    return pr.ia, pr.ja, pr.a, None


def raw_tile():
    """5-point Laplacian of 64 x 64 whose tile 3 carries distinct values: more than 256 (delta, value) pairs -> a raw tile in the blob"""
    ia, ja, a, _ = lap2d(64)
    a = a.copy()
    k0, k1 = ia[3 * 256], ia[4 * 256]
    a[k0:k1] = 1.0 + np.arange(k1 - k0) * 1e-3
    return ia, ja, a, None


def ragged(n, lens, span, nval, seed):
    rng = np.random.default_rng(seed)
    rows = []
    for r in range(n):
        L = int(rng.choice(lens))
        cand = np.arange(max(0, r - span), min(n, r + span + 1))
        c = np.sort(rng.choice(cand, size=min(L, len(cand)), replace=False))
        rows.append((c, rng.integers(1, nval + 1, size=len(c)).astype(np.float64)))
    return (*_csr(rows), None)


def empty_rows():
    """2-D Laplacian with scattered empty rows and one whole empty tile"""
    ia, ja, a, _ = lap2d(40)
    n = len(ia) - 1
    rows = [(ja[ia[r]:ia[r + 1]], a[ia[r]:ia[r + 1]]) for r in range(n)]
    for r in list(range(0, n, 37)) + list(range(512, 768)):
        rows[r] = ([], [])
    return (*_csr(rows), None)


def unsorted():
    ia, ja, a, _ = lap2d(40)
    ja = ja.copy()
    for r in (5, 300, 1000):
        ja[ia[r]:ia[r + 1]] = ja[ia[r]:ia[r + 1]][::-1]
    return ia, ja, a, None


def dad():
    from permon_b200 import problems as PR
    pr = PR.obstacle2d(64, scaled=True)
    return pr.ia, pr.ja, pr.a, None


def long_rows(n, L, seed):
    """n rows of L > 64 distinct values; column k of row r is r + 3k + (0, 1 or 2): strictly increasing"""
    rng = np.random.default_rng(seed)
    ja = np.arange(n)[:, None] + 3 * np.arange(L)[None, :] + rng.integers(0, 3, size=(n, L))
    ia = np.arange(n + 1, dtype=np.int64) * L
    return ia, ja.ravel(), rng.standard_normal(n * L), n + 3 * L


def rect():
    """1000 x 1500: a 5-point-like band plus a wide coupling column block"""
    ia, ja, a, _ = lap2d(32)
    n = 1000
    rows = [(np.append(ja[ia[r]:ia[r + 1]], [1100 + r % 400]), np.append(a[ia[r]:ia[r + 1]], [0.5])) for r in range(n)]
    rows = [(c[c < 1500], v[c < 1500]) for c, v in rows]
    return (*_csr(rows), 1500)


CASES = {
    "lap5_n40": lambda: lap2d(40),            # n = 1600, not a multiple of 256
    "lap5_n7": lambda: lap2d(7),              # n = 49 < 64
    "lap5_n32": lambda: lap2d(32),            # n = 1024
    "lap7_n12": lambda: lap3d(12),
    "varcoef16": lambda: varcoef(16),         # two-bound C5-like operator: packed tiles
    "raw_tile": raw_tile,
    "ragged_short": lambda: ragged(3000, [4, 5], 20, 3, 1),    # padded short rows
    "ragged_long": lambda: ragged(3000, range(1, 30), 40, 2, 2),   # 16-bit row offsets
    "empty_rows": empty_rows,
    "unsorted": unsorted,
    "dad": dad,                               # every value distinct: CSR ring
    "long_rows_ell": lambda: long_rows(16384, 72, 3),   # nnz >= 2^20: tile-ELL
    "long_rows_vector": lambda: long_rows(2000, 80, 4),
    "rect": rect,
}


def _tensors(ia, ja, a):
    import torch
    return (torch.as_tensor(np.ascontiguousarray(ia, np.int32)).cuda(), torch.as_tensor(np.ascontiguousarray(ja, np.int32)).cuda(),
            torch.as_tensor(np.ascontiguousarray(a, np.float64)).cuda())


def _mult(P, A, ncols, nrows, seed=0):
    x = np.random.default_rng(seed).standard_normal(ncols)
    y = np.zeros(nrows)
    vx, vy = P.VecFromArray(x), P.VecFromArray(y)
    P.MatMult(A, vx, vy)
    out = P.VecGetArray(vy)
    P.VecDestroy(vx)
    P.VecDestroy(vy)
    return out


@pytest.mark.parametrize("env", list(ENVS))
@pytest.mark.parametrize("case", list(CASES))
def test_stored_form_and_product_match_host(P, case, env, monkeypatch):
    for k, v in ENVS[env].items():
        monkeypatch.setenv(k, v)
    ia, ja, a, ncols = CASES[case]()
    n = len(ia) - 1
    ncols = n if ncols is None else ncols
    Ah = P.MatCreateAIJ(ia, ja, a, ncols_local=ncols)
    Ad = P.MatCreateAIJFromDeviceTensors(*_tensors(ia, ja, a), ncols_local=ncols)
    fh, fd = P.MatGetStoredForm(Ah), P.MatGetStoredForm(Ad)
    assert fh["fields"] == fd["fields"]
    for part in P.FORM_PARTS:
        assert fh[part] == fd[part], part
    assert P.MatStorageInfo(Ah) == P.MatStorageInfo(Ad)
    if env == "default":
        expect = {"lap5_n40": 4, "lap5_n7": 2, "varcoef16": 3, "raw_tile": 3, "ragged_short": 3, "ragged_long": 3, "unsorted": 3, "dad": 2,
                  "long_rows_ell": 5, "long_rows_vector": 1}
        if case in expect:
            assert fd["fields"]["kind"] == expect[case], (case, fd["fields"])
    yh, yd = _mult(P, Ah, ncols, n), _mult(P, Ad, ncols, n)
    assert yh.tobytes() == yd.tobytes()
    P.MatDestroy(Ah)
    P.MatDestroy(Ad)


def test_packed_blob_kinds_are_exercised(P):
    """the cases above reach raw tiles, padded ragged rows and row offsets inside the blob"""
    def kinds(ia, ja, a):
        Ad = P.MatCreateAIJFromDeviceTensors(*_tensors(ia, ja, a))
        f = P.MatGetStoredForm(Ad)
        blob, off = f["pk_blob"], np.frombuffer(f["pk_off"], np.uint32)
        hdr = [np.frombuffer(blob[o * 16:o * 16 + 16], dtype=np.dtype([("kind", "<u2"), ("ndict", "<u2"), ("nnz", "<u4"), ("ulen", "<u2"),
                                                                            ("nrows", "<u2"), ("pad", "<u4")]))[0] for o in off[:-1]]
        P.MatDestroy(Ad)
        return hdr
    h = kinds(*raw_tile()[:3])
    assert h[3]["kind"] == 0 and all(x["kind"] == 2 for i, x in enumerate(h) if i != 3)
    h = kinds(*ragged(3000, [4, 5], 20, 3, 1)[:3])
    assert any(x["kind"] == 1 and x["pad"] > 0 for x in h)
    h = kinds(*ragged(3000, range(1, 30), 40, 2, 2)[:3])
    assert any(x["kind"] == 1 and x["ulen"] == 0xFFFF for x in h)


def _same_solve(rh, rd):
    assert rh.reason == rd.reason
    assert rh.its == rd.its
    assert rh.counts == rd.counts
    assert rh.x.tobytes() == rd.x.tobytes()


@pytest.mark.parametrize("mode", ["keep", "zero"])
def test_mpgp_solve_bit_identical(P, mode):
    from permon_b200 import problems as PR
    pr = PR.obstacle2d(48, -100.0)
    rh = P.solve_problem(pr, "mpgp", "-qps_rtol 1e-8")
    rd = P.solve_problem(pr, "mpgp", "-qps_rtol 1e-8", device_input=mode)
    assert rh.reason == 2
    _same_solve(rh, rd)


def test_mpgp_solve_varcoef_bit_identical(P):
    from permon_b200 import problems as PR
    pr = PR.varcoef3d(16)
    rh = P.solve_problem(pr, "mpgp", "-qps_rtol 1e-8")
    rd = P.solve_problem(pr, "mpgp", "-qps_rtol 1e-8", device_input="zero")
    _same_solve(rh, rd)


def test_smalxe_one_equality_row_bit_identical(P):
    from permon_b200 import problems as PR
    pr = PR.obstacle2d(32)
    n = pr.n
    pr = dataclasses.replace(pr, B=np.ones((1, n)), c=np.array([float(np.sum(pr.lb)) + 0.1 * n]))
    rh = P.solve_problem(pr, "smalxe", "-qps_rtol 1e-8")
    rd = P.solve_problem(pr, "smalxe", "-qps_rtol 1e-8", device_input="zero")
    _same_solve(rh, rd)


def _ksp_solve(P, A, b):
    P.options_clear()
    P.call("PetscOptionsInsertString", None, b"-qps_rtol 1e-10")
    vb, vx = P.VecFromArray(b.copy()), P.VecFromArray(np.zeros_like(b))
    qp = P.QPCreate()
    P.QPSetOperator(qp, A), P.QPSetRhs(qp, vb), P.QPSetInitialVector(qp, vx)
    qps = P.QPSCreate()
    P.QPSSetType(qps, "ksp")
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    P.QPSSolve(qps)
    out = (P.VecGetArray(vx).copy(), P.QPSGetIterationNumber(qps), P.QPSGetConvergedReason(qps))
    P.QPSDestroy(qps), P.QPDestroy(qp), P.VecDestroy(vb), P.VecDestroy(vx), P.MatDestroy(A)
    P.options_clear()
    return out


def test_ksp_bit_identical(P):
    from permon_b200 import problems as PR
    pr = PR.obstacle2d(48)
    t = _tensors(pr.ia, pr.ja, pr.a)
    Ad = P.MatCreateAIJFromDeviceTensors(*t)
    for v in t:
        v.zero_()
    xh, ih, rh = _ksp_solve(P, P.MatCreateAIJ(pr.ia, pr.ja, pr.a), pr.b)
    xd, id_, rd = _ksp_solve(P, Ad, pr.b)
    assert rh == rd and rh > 0 and ih == id_
    assert xh.tobytes() == xd.tobytes()


def test_error_codes(P):
    import torch
    ia, ja, a, _ = lap2d(16)
    t = _tensors(ia, ja, a)
    n = len(ia) - 1

    def create(pi, pj, pa):
        A = C.c_void_p()
        f = P.lib().MatB200CreateAIJWithDeviceArrays
        f.restype = C.c_int
        return f(P.world(), C.c_int(n), C.c_int(n), C.c_int(P.DECIDE), C.c_int(P.DECIDE), C.c_void_p(pi), C.c_void_p(pj), C.c_void_p(pa), C.byref(A))

    assert create(None, t[1].data_ptr(), t[2].data_ptr()) == 85          # PETSC_ERR_ARG_NULL
    assert create(t[0].data_ptr(), None, t[2].data_ptr()) == 85
    assert create(t[0].data_ptr(), t[1].data_ptr(), None) == 85
    hia = np.ascontiguousarray(ia, np.int32)
    assert create(hia.ctypes.data, t[1].data_ptr(), t[2].data_ptr()) == 62   # PETSC_ERR_ARG_WRONG: pageable host memory
    pinned = torch.as_tensor(np.ascontiguousarray(a, np.float64)).pin_memory()
    assert create(t[0].data_ptr(), t[1].data_ptr(), pinned.data_ptr()) == 62   # pinned host memory
    with pytest.raises(TypeError):
        P.MatCreateAIJFromDeviceTensors(t[0].long(), t[1], t[2])
    with pytest.raises(TypeError):
        P.MatCreateAIJFromDeviceTensors(t[0].cpu(), t[1], t[2])


# ---- several ranks on one GPU (gloo host exchange) ---------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _mr_worker(rank, size, port, kind, ret):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    from permon_b200 import api as P
    from permon_b200 import problems as PR

    def agi(v):
        out = [None] * size
        dist.all_gather_object(out, int(v))
        return out

    def agv(data):
        out = [None] * size
        dist.all_gather_object(out, bytes(data))
        return out

    try:
        P.initialize()
        P.comm_set_host_exchange(size, rank, agi, agv)
        if kind == "2d":
            N = 64
            starts = PR.row_partition(N * N, size, align=N)
            pr = PR.obstacle2d(N, rows=(starts[rank], starts[rank + 1]))
            ia, ja, a, ncols = pr.ia, pr.ja, pr.a, pr.n
        elif kind == "var":
            N = 12
            starts = PR.row_partition(N ** 3, size, align=N * N)
            pr = PR.varcoef3d(N, rows=(starts[rank], starts[rank + 1]))
            ia, ja, a, ncols = pr.ia, pr.ja, pr.a, pr.n
        else:   # equality rows: 3 rows over 600 columns, the rows split over the ranks
            nglob = 600
            cstarts = PR.row_partition(nglob, size)
            rstarts = PR.row_partition(3, size)
            rows = [(np.arange(q, nglob, 7), np.full(len(range(q, nglob, 7)), 1.0 + q)) for q in range(rstarts[rank], rstarts[rank + 1])]
            ia, ja, a = _csr(rows) if rows else (np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0))
            ncols = cstarts[rank + 1] - cstarts[rank]
        Ah = P.MatCreateAIJ(ia, ja, a, ncols_local=ncols)
        hi = P.MatGetHaloInfo(Ah)
        Ad = P.MatCreateAIJFromDeviceTensors(*_tensors(ia, ja, a), ncols_local=ncols)
        di = P.MatGetHaloInfo(Ad)
        assert hi == di, (hi, di)
        for off in (False, True):
            fh, fd = P.MatGetStoredForm(Ah, offdiag=off), P.MatGetStoredForm(Ad, offdiag=off)
            assert fh["fields"] == fd["fields"], (off, fh["fields"], fd["fields"])
            for part in P.FORM_PARTS:
                assert fh[part] == fd[part], (off, part)
        if kind == "2d":
            assert P.MatGetStoredForm(Ad)["fields"]["kind"] == 4
        try:
            P.MatGetHostSplit(Ad, len(ia) - 1)
            raise AssertionError("a device-built matrix has no host split")
        except P.PermonError as e:
            assert e.code == 73
        ret[rank] = True
    except Exception:
        import traceback
        traceback.print_exc()
        ret[rank] = False
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("size", [2, 3])
@pytest.mark.parametrize("kind", ["2d", "var", "eq"])
def test_multirank_one_gpu_matches_host(P, size, kind):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    mgr = ctx.Manager()
    ret = mgr.dict()
    port = _free_port()
    procs = [ctx.Process(target=_mr_worker, args=(r, size, port, kind, ret)) for r in range(size)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert all(ret.get(r) for r in range(size)), dict(ret)


# ---- several GPUs (torchrun) --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_multi_gpu_device_input_solves_bit_identical(nproc):
    import json
    import subprocess
    from permon_b200 import api
    if api.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1", "--master-port",
           str(_free_port()), os.path.join(ROOT, "tests", "device_input_mgpu_worker.py"), "obstacle2d,obstacle3d,varcoef3d,smalxe_aij2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("DEVICE_INPUT_RESULT ")][-1]
    res = json.loads(line[len("DEVICE_INPUT_RESULT "):])
    for kind, r in res.items():
        assert r["identical"], (kind, r)
