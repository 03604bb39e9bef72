"""Dense Hessians (MatCreateSeqDense / MatCreateSeqDenseCUDA, stored form kind 6) on the GPU: MatMult against the full-CSR AIJ form of
the same matrix bit for bit, layouts (lda, host / device, adopted / copied), the split-column variant of wide matrices, and the solvers
(fused and generic MPGP, SMALXE, CG, PCPG, power method) on dense Hessians against the AIJ form and the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import oracle_py as O
from permon_b200 import problems as PR

EPS = 2.220446049250313e-16


@pytest.fixture(scope="module")
def P():
    from permon_b200 import api
    if api.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    api.initialize()
    yield api
    api.options_clear()


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def mult(P, A, x, m):
    vx, vy = P.VecFromArray(np.ascontiguousarray(x, dtype=np.float64).copy()), P.VecCreate(m)
    P.MatMult(A, vx, vy)
    y = P.VecGetArray(vy).copy()
    P.VecDestroy(vx), P.VecDestroy(vy)
    return y


def full_csr_aij(P, torch, Ad):
    """AIJ matrix that stores every entry of the (m x n) device tensor Ad, built on the device"""
    m, n = Ad.shape
    ia = torch.arange(0, (m + 1) * n, n, dtype=torch.int32, device=Ad.device)
    ja = torch.arange(n, dtype=torch.int32, device=Ad.device).repeat(m)
    a = Ad.contiguous().reshape(-1)
    A = P.MatCreateAIJFromDeviceTensors(ia, ja, a, ncols_local=n)
    del ia, ja, a
    return A


def with_lda(torch, Ad, lda, offset=0):
    """column-major copy of Ad with leading dimension lda, its first element `offset` doubles into the allocation"""
    m, n = Ad.shape
    buf = torch.zeros(n * lda + offset, dtype=torch.float64, device=Ad.device)
    v = buf[offset:].as_strided((m, n), (1, lda))
    v.copy_(Ad)
    return v


def tol_check(y, A, x):
    scale = np.abs(A) @ np.abs(x)
    n = A.shape[1]
    assert np.all(np.abs(y - A @ x) <= 4 * n * EPS * scale + 1e-300), np.max(np.abs(y - A @ x) / (scale + 1e-300))


@pytest.mark.parametrize("n", [1024, 1025, 4095, 4736, 4737, 20000])
def test_matmult_bit_identical_to_full_csr(P, torch, n):
    """every layout of the same matrix gives the bits of the full-CSR AIJ matrix (tile-ELL, products added in storage order)"""
    g = torch.Generator(device="cuda").manual_seed(n)
    Ad = torch.randn(n, n, generator=g, dtype=torch.float64, device="cuda").t()      # column-major view
    x = np.random.default_rng(n).standard_normal(n)
    Aij = full_csr_aij(P, torch, Ad)
    assert P.MatStorageInfo(Aij)["kind"] == 5
    y_ref = mult(P, Aij, x, n)
    P.MatDestroy(Aij)
    odd = n + 1 if n % 2 == 0 else n + 2
    variants = [("device", Ad, n % 2 == 0), ("device lda m+7", with_lda(torch, Ad, n + 7), (n + 7) % 2 == 0),
                ("device odd lda", with_lda(torch, Ad, odd), False), ("device offset 8 bytes", with_lda(torch, Ad, n + (n % 2), offset=1), False)]
    for name, t, adopt in variants:
        A = P.MatCreateDenseFromTensor(t)
        info = P.MatDenseGetInfo(A)
        assert info["adopted"] == adopt, (name, info)
        assert info["split_columns"] == 0 and info["lda"] % 2 == 0
        st = P.MatStorageInfo(A)
        assert st["kind"] == 6 and st["stream_bytes"] == 8.0 * n * n
        y = mult(P, A, x, n)
        assert np.array_equal(y, y_ref), name
        P.MatDestroy(A)
    # host arrays: lda = m at every size; odd lda and lda = m + 7 up to n = 4737 (at n = 20000 each is another 3.2 GB host copy)
    Ah = Ad.cpu().numpy()
    for lda in ((n, odd, n + 7) if n <= 4737 else (n,)):
        big = np.zeros((lda, n), order="F")
        big[:n, :] = Ah
        A = P.MatCreateDense(big[:n, :])
        assert P.MatDenseGetLDA(A) == lda
        info = P.MatDenseGetInfo(A)
        assert not info["adopted"] and info["lda"] % 2 == 0
        assert np.array_equal(mult(P, A, x, n), y_ref), lda
        P.MatDestroy(A)


@pytest.mark.parametrize("shape", [(1, 1), (31, 31), (100, 100), (513, 513), (3000, 40), (777, 5), (40, 5000), (3, 20000), (64, 4096)])
def test_matmult_small_and_rectangular(P, torch, shape):
    """n < 1024 and rectangular shapes against NumPy; wide matrices (n > 64 m) take the split-column variant, bit-reproducible"""
    m, n = shape
    rng = np.random.default_rng(m * 7 + n)
    A = rng.standard_normal((m, n))
    x = rng.standard_normal(n)
    M = P.MatCreateDense(A)
    info = P.MatDenseGetInfo(M)
    assert (info["split_columns"] > 0) == (n > 64 * m), info
    y1 = mult(P, M, x, m)
    y2 = mult(P, M, x, m)
    tol_check(y1, A, x)
    assert np.array_equal(y1, y2)
    P.MatDestroy(M)
    # the same from a device tensor (column-major; adopted when lda is even, copied otherwise)
    t = torch.tensor(A, device="cuda").t().contiguous().t()
    Md = P.MatCreateDenseFromTensor(t)
    assert np.array_equal(mult(P, Md, x, m), y1)
    P.MatDestroy(Md)


def test_adopted_tensor_is_read_in_place(P, torch):
    g = torch.Generator(device="cuda").manual_seed(3)
    t = torch.randn(600, 600, generator=g, dtype=torch.float64, device="cuda").t()
    A = P.MatCreateDenseFromTensor(t)
    assert P.MatDenseGetInfo(A)["adopted"]
    x = np.random.default_rng(3).standard_normal(600)
    y1 = mult(P, A, x, 600)
    t.mul_(2.0)
    torch.cuda.synchronize()
    y2 = mult(P, A, x, 600)
    assert np.array_equal(y2, 2.0 * y1)
    P.MatDestroy(A)
    # set-up state: the leading dimension cannot change after the first use
    import ctypes as C
    B = P.MatCreateDense(np.eye(4))
    P.MatDenseGetInfo(B)
    with pytest.raises(P.PermonError) as e:
        P.call("MatDenseSetLDA", B, C.c_int(6))
    assert e.value.code == 73
    P.MatDestroy(B)
    # host memory handed to the CUDA constructor
    h = np.zeros((4, 4), order="F")
    M = C.c_void_p()
    with pytest.raises(P.PermonError) as e:
        P.call("MatCreateSeqDenseCUDA", P.world(), C.c_int(4), C.c_int(4), C.c_void_p(h.ctypes.data), C.byref(M))
    assert e.value.code == 62


def test_power_method_dense_vs_aij(P, torch):
    pr = PR.tutorial_ex3_dual(100)
    rng = np.random.default_rng(9)
    G = rng.standard_normal((2000, 2000))
    for A in (pr.a.reshape(pr.n, pr.n), G @ G.T / 2000 + np.eye(2000)):
        n = A.shape[0]
        import scipy.sparse as sp
        S = sp.csr_matrix(A)
        Ma, Md = P.MatCreateAIJ(S.indptr, S.indices, S.data), P.MatCreateDense(A)
        la, ld = P.MatGetMaxEigenvalue(Ma), P.MatGetMaxEigenvalue(Md)
        assert ld == pytest.approx(la, rel=1e-14), (n, la, ld)
        P.MatDestroy(Ma), P.MatDestroy(Md)


# ------------------------------------------------------------------------------------------------------
# golden problems through the dense form
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("driver", ["fused", "generic"])
def test_ex3_dual_golden_counts_dense(P, golden, driver):
    g = golden["ex3_1"]
    pr = PR.tutorial_ex3_dual(g["n"])
    r = P.solve_problem(pr, "mpgp", f"-qps_mpgp_b200_driver {driver}", dense=True)
    c = r.counts
    assert (r.its, c["nmv"], c["ncg"], c["nexp"], c["nprop"], r.reason) == (g["its"], g["nmv"], g["ncg"], g["nexp"], g["nprop"], g["reason"])
    op = O.Operator(pr.ia, pr.ja, pr.a)
    xr, ro = O.mpgp_solve(op, pr.b, O.BoxC(pr.n, pr.lb, None), pr.x0, O.mpgp_opts())
    assert np.linalg.norm(r.x - xr) <= 1e-9 * np.linalg.norm(xr)


def test_ex3_nullspace_smalxe_golden_dense(P, golden):
    g = golden["ex3_nullspace"]
    pr = PR.tutorial_ex3_dual(g["n"])
    P.options_clear()
    A = P.MatCreateDense(pr.a.reshape(pr.n, pr.n))
    vb, vx, vl = P.VecFromArray(pr.b.copy()), P.VecFromArray(np.zeros(pr.n)), P.VecFromArray(np.zeros(pr.n))
    BE = P.MatCreateAIJ(np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0), ncols_local=pr.n)
    qp = P.QPCreate()
    P.QPSetOperator(qp, A), P.QPSetRhs(qp, vb), P.QPSetInitialVector(qp, vx), P.QPSetBox(qp, None, vl, None), P.QPSetEq(qp, BE, None)
    qps = P.QPSCreate()
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    P.QPSSolve(qps)
    inner = P.QPSSMALXEGetInnerQPS(qps)
    c = P.QPSMPGPGetStepCounts(inner)
    st = P.QPSSMALXEGetStatistics(qps)
    assert (P.QPSGetIterationNumber(qps), P.QPSGetConvergedReason(qps)) == (g["outer_its"], g["outer_reason"])
    assert (st["inner_iter_accu"], P.QPSGetConvergedReason(inner)) == (g["total_inner"], g["inner_reason"])
    assert (c["nmv"], c["ncg"], c["nexp"], c["nprop"]) == (g["nmv"], g["ncg"], g["nexp"], g["nprop"])
    P.QPSDestroy(qps), P.QPDestroy(qp)
    for v in (vb, vx, vl):
        P.VecDestroy(v)
    P.MatDestroy(A), P.MatDestroy(BE)


# ------------------------------------------------------------------------------------------------------
# MPGP: dense against AIJ, step by step
# ------------------------------------------------------------------------------------------------------
def dense_box_qp(n, two_sided, seed=5):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((n, n)) / np.sqrt(n)
    A = G @ G.T + 0.05 * np.eye(n)
    A = 0.5 * (A + A.T)
    b = rng.standard_normal(n) * 2.0
    lb = -0.3 * np.abs(rng.standard_normal(n))
    ub = 0.3 + 0.3 * np.abs(rng.standard_normal(n)) if two_sided else None
    ia = (np.arange(n + 1) * n).astype(np.int32)
    ja = np.tile(np.arange(n, dtype=np.int32), n)
    return PR.QPProblem(f"densebox{n}", n, 0, n, ia, ja, np.ascontiguousarray(A).ravel(), b, lb, ub, np.zeros(n))


def product_qp(n, d, seed=6):
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    Z = rng.standard_normal((n, d)) / np.sqrt(d)
    S, St = sp.csr_matrix(Z), sp.csr_matrix(Z.T)
    b = Z @ rng.standard_normal(d)   # in the range of Z: the objective is bounded below on x >= 0
    return PR.QPProblem(f"zzt{n}x{d}", n, 0, n, S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data, b, np.zeros(n), None, np.zeros(n),
                        second=(St.indptr.astype(np.int32), St.indices.astype(np.int32), St.data), meta=dict(d=d))


def traced(P, pr, dense, its):
    steps = []
    r = P.solve_problem(pr, "mpgp", f"-qps_max_it {its} -qps_rtol 1e-14 -qps_mpgp_b200_driver fused",
                        monitor=lambda q, it, rn: steps.append(P.QPSMPGPGetCurrentStepType(q)), dense=dense)
    return r, "".join(steps)


@pytest.mark.parametrize("kind", ["lower", "two_sided", "product"])
def test_mpgp_dense_against_aij(P, kind):
    pr = product_qp(4096, 64) if kind == "product" else dense_box_qp(2000, kind == "two_sided")
    for its in (50, 200):   # checkpoints
        ra, sa = traced(P, pr, False, its)
        rd, sd = traced(P, pr, True, its)
        assert sd == sa and len(sd) >= min(its, ra.its), (its, sd[:80], sa[:80])
        assert rd.counts == ra.counts
        assert np.linalg.norm(rd.x - ra.x) <= 1e-12 * np.linalg.norm(ra.x)
    if kind != "product":
        # against the oracle at a checkpoint, with the checkpoint tolerances of the lockstep tests (iterate and objective)
        import test_gpu_lockstep as LS
        op = O.Operator(pr.ia, pr.ja, pr.a)
        xr, ro = O.mpgp_solve(op, pr.b, O.BoxC(pr.n, pr.lb, pr.ub), pr.x0, O.mpgp_opts(rtol=1e-14, max_it=50))
        r50, _ = traced(P, pr, True, 50)
        assert (ro["its"], ro["ncg"], ro["nexp"], ro["nprop"]) == (r50.its, r50.counts["ncg"], r50.counts["nexp"], r50.counts["nprop"])
        assert np.linalg.norm(r50.x - xr) <= LS.X_TOL * np.linalg.norm(xr)
        fr = O.objective(op, pr.b, xr)
        assert abs(O.objective(op, pr.b, r50.x) - fr) <= LS.F_TOL * abs(fr)


# ------------------------------------------------------------------------------------------------------
# SMALXE, CG, PCPG
# ------------------------------------------------------------------------------------------------------
def svm_kernel_qp(n, seed=8, C=1.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 8))
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    sq = (X * X).sum(1)
    K = np.exp(-0.125 * np.maximum(sq[:, None] + sq[None, :] - 2 * X @ X.T, 0.0))
    H = (y[:, None] * K) * y[None, :]
    H = 0.5 * (H + H.T)
    ia = (np.arange(n + 1) * n).astype(np.int32)
    ja = np.tile(np.arange(n, dtype=np.int32), n)
    return PR.QPProblem(f"ksvm{n}", n, 0, n, ia, ja, np.ascontiguousarray(H).ravel(), np.ones(n), np.zeros(n), np.full(n, C), np.zeros(n),
                        B=y.reshape(1, n).copy(), c=None, meta=dict(y=y))


def smalxe_svm(P, pr, be):
    n = pr.n
    P.options_clear()
    P.call("PetscOptionsInsertString", None, b"-qps_rtol 1e-9")
    A = P.MatCreateDense(pr.a.reshape(n, n))
    vb, vx = P.VecFromArray(pr.b.copy()), P.VecFromArray(pr.x0.copy())
    vl, vu = P.VecFromArray(pr.lb.copy()), P.VecFromArray(pr.ub.copy())
    if be == "onerow":
        brow = P.VecFromArray(pr.B[0].copy())
        BE = P.MatCreateOneRow(brow)
    else:
        brow = None
        BE = P.MatCreateDense(pr.B)
    qp = P.QPCreate()
    P.QPSetOperator(qp, A), P.QPSetRhs(qp, vb), P.QPSetInitialVector(qp, vx), P.QPSetBox(qp, None, vl, vu), P.QPSetEq(qp, BE, None)
    qps = P.QPSCreate()
    P.QPSSetType(qps, "smalxe")
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    P.QPSSolve(qps)
    x = P.VecGetArray(vx).copy()
    P.QPSDestroy(qps), P.QPDestroy(qp)
    for v in (vb, vx, vl, vu, brow):
        if v is not None:
            P.VecDestroy(v)
    P.MatDestroy(A), P.MatDestroy(BE)
    return x


def test_smalxe_kernel_svm_dense(P):
    """one equality row y^T a = 0 given as MatCreateOneRow and as a 1 x n dense B_E: the same iterates bit for bit; against the oracle the
    solution agrees to 5.6e-9 relative at rtol 1e-9 (the reference's own solution moves by ~rtol * cond with the summation order of its
    dot products, DESIGN.md section 5)"""
    pr = svm_kernel_qp(2000)
    x1, x2 = smalxe_svm(P, pr, "onerow"), smalxe_svm(P, pr, "dense")
    assert np.array_equal(x1, x2)
    op = O.Operator(pr.ia, pr.ja, pr.a)
    xr, ro = O.smalxe_solve(op, pr.b, O.BoxC(pr.n, pr.lb, pr.ub), pr.B, pr.c, pr.x0, O.smalxe_opts(rtol=1e-9))
    assert np.linalg.norm(x1 - xr) <= 1e-8 * np.linalg.norm(xr)
    assert abs(pr.meta["y"] @ x1) <= 1e-6 * np.linalg.norm(x1)


def linear_solve(P, A_np, b, x0, qps_type=None, G=None, options="-qps_rtol 1e-9"):
    P.options_clear()
    P.call("PetscOptionsInsertString", None, options.encode())
    A = P.MatCreateDense(A_np)
    vb, vx = P.VecFromArray(b.copy()), P.VecFromArray(x0.copy())
    qp = P.QPCreate()
    P.QPSetOperator(qp, A), P.QPSetRhs(qp, vb), P.QPSetInitialVector(qp, vx)
    BE = None
    if G is not None:
        BE = P.MatCreateDense(G)
        P.QPSetEq(qp, BE, None)
    qps = P.QPSCreate()
    if qps_type:
        P.QPSSetType(qps, qps_type)
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    P.QPSSolve(qps)
    out = dict(x=P.VecGetArray(vx).copy(), its=P.QPSGetIterationNumber(qps), reason=P.QPSGetConvergedReason(qps), type=P.QPSGetType(qps))
    P.QPSDestroy(qps), P.QPDestroy(qp), P.VecDestroy(vb), P.VecDestroy(vx), P.MatDestroy(A)
    if BE is not None:
        P.MatDestroy(BE)
    return out


@pytest.mark.parametrize("driver", ["auto", "generic"])
def test_cg_on_dense(P, driver):
    """auto: the fused CG takes the dense Hessian (3 launches per iteration: direction update, SpMV + p.Ap, x / r update + r.r);
    generic: one launch per KSPCG call (7 per iteration)"""
    pr = dense_box_qp(1500, False, seed=11)
    A = pr.a.reshape(pr.n, pr.n)
    rng = np.random.default_rng(12)
    b, x0 = rng.standard_normal(pr.n), rng.standard_normal(pr.n)
    l0 = P.launch_count()
    r = linear_solve(P, A, b, x0, options=f"-qps_rtol 1e-9 -qps_ksp_b200_driver {driver}")
    per_it = (P.launch_count() - l0) / r["its"]
    assert r["type"] == "ksp" and r["reason"] > 0 and r["its"] >= 20
    assert (per_it < 4.0) if driver == "auto" else (per_it > 6.0), per_it
    xr, ro = O.cg_solve(O.Operator(pr.ia, pr.ja, pr.a), b, x0, O.lin_opts(rtol=1e-9))
    assert abs(r["its"] - ro["its"]) <= 2, (r["its"], ro["its"])
    assert np.linalg.norm(r["x"] - xr) <= 1e-7 * np.linalg.norm(xr)


def test_pcpg_with_dense_equality_rows(P):
    pr = dense_box_qp(1200, False, seed=13)
    A = pr.a.reshape(pr.n, pr.n)
    rng = np.random.default_rng(14)
    G = rng.standard_normal((3, pr.n))
    b = rng.standard_normal(pr.n)
    r = linear_solve(P, A, b, np.zeros(pr.n), "pcpg", G=G, options="-qps_rtol 1e-10")
    assert r["reason"] > 0
    xr, ro = O.pcpg_solve(O.Operator(pr.ia, pr.ja, pr.a), b, G, None, np.zeros(pr.n), O.lin_opts(rtol=1e-10))
    assert abs(r["its"] - ro["its"]) <= 2, (r["its"], ro["its"])
    assert np.linalg.norm(r["x"] - xr) <= 1e-8 * np.linalg.norm(xr)
    assert np.abs(G @ r["x"]).max() <= 1e-9 * np.linalg.norm(xr)


def test_matmult_beyond_the_aij_ceiling(P, torch):
    """n = 50 000: n^2 > 2^31 entries, which an AIJ matrix with int32 row pointers cannot hold"""
    n = 50000
    g = torch.Generator(device="cuda").manual_seed(50)
    A = torch.randn(n, n, generator=g, dtype=torch.float64, device="cuda").t()
    xt = torch.randn(n, generator=g, dtype=torch.float64, device="cuda")
    ref = (A @ xt).cpu().numpy()
    scale = (A.abs() @ xt.abs()).cpu().numpy()
    M = P.MatCreateDenseFromTensor(A)
    assert P.MatDenseGetInfo(M)["adopted"]
    y = mult(P, M, xt.cpu().numpy(), n)
    P.MatDestroy(M)
    del A
    torch.cuda.empty_cache()
    assert np.all(np.abs(y - ref) <= 4 * n * EPS * scale)
