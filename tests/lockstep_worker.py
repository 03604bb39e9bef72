"""Cases and GPU runs of tests/test_gpu_lockstep.py.

Every case is a small QP whose data picks one variant of the fused MPGP kernels (SpMV form, box, vector layout, equality rows).  `gpu_runs`
solves it through the C ABI in the two schedules the library has: host-sync (a monitor is set: one trace record per iteration) and the
folded device-driven one (`-qps_max_it k` for a list of checkpoints, tolerances disabled).

Run as a script (`python tests/lockstep_worker.py CASE OUT.npz [OPTIONS]`) it does the same in a fresh process: several PERMON_B200_*
switches are read once per process into statics, so an A/B variant needs a process of its own.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from permon_b200 import problems as PR  # noqa: E402

CHECKPOINTS = (0, 1, 2, 3, 5, 8, 13, 21, 34)
TRACE_ITS = 50
NOTOL = "-qps_rtol 1e-30 -qps_atol 1e-300"
INF = PR.PETSC_INFINITY


class Case:
    """pr: the QP (PR.QPProblem; pr.B unused).  B / rho: equality rows enforced by the penalty rho B'B (QPTEnforceEqByPenalty, direct rho),
    eq_form "onerow" (MatCreateOneRow, m = 1) or "aij".  kind: expected MatStorageInfo kind of the Hessian (None: not asserted), W: the
    lanes-per-row bucket of kind 1.  devvec: b, x and the bounds handed over as device pointers 8 bytes into an allocation."""

    def __init__(self, pr, kind=None, W=None, B=None, rho=0.0, eq_form="aij", driver="fused", devvec=False, alpha=None, rtol=1e-30):
        self.pr, self.kind, self.W, self.B, self.rho, self.eq_form, self.driver, self.devvec = pr, kind, W, B, rho, eq_form, driver, devvec
        self.alpha = alpha   # -qps_mpgp_alpha (multiple of 1/maxeig); None: the default 2
        self.rtol = rtol     # 1e-30: never converges; fast-converging cases stop at a real tolerance instead of at rounding level


# ---- matrices -------------------------------------------------------------------------------------------
def _csr(S):
    import scipy.sparse as sp
    S = sp.csr_matrix(S)
    S.sort_indices()
    return S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data.astype(np.float64)


def lap1d(n, diag=2.05):
    import scipy.sparse as sp
    return sp.diags([-np.ones(n - 1), diag * np.ones(n), -np.ones(n - 1)], [-1, 0, 1], format="csr")


def lap2d(nx, ny, diag=4.0):
    import scipy.sparse as sp
    return (sp.kron(sp.identity(ny), lap1d(nx, 0.0)) + sp.kron(lap1d(ny, 0.0), sp.identity(nx)) + diag * sp.identity(nx * ny)).tocsr()


def band_plus_rank_one(n, k, support=100, seed=3):
    """SPD: a symmetric band of half-width k (constant diagonals, diagonally dominant) plus u u' on `support` rows spread over the
    matrix.  Those rows have about `support` entries (> 64), which sends the whole Hessian to the lanes-per-row kernel."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    offs = list(range(-k, k + 1))
    margin = 10.0 ** (-3.0 * rng.random(n))           # diagonal dominance between 1e-3 and 1: a spread-out spectrum
    diags = [(-0.5 / (abs(d) + 1)) * np.ones(n - abs(d)) if d else margin + sum(1.0 / (abs(e) + 1) for e in offs if e) for d in offs]
    A = sp.diags(diags, offs, format="csr")
    idx = np.linspace(0, n - 1, support).astype(np.int64)
    u = 0.05 * (0.5 + rng.random(support))
    U = sp.csr_matrix((np.outer(u, u).ravel(), (np.repeat(idx, support), np.tile(idx, support))), shape=(n, n))
    return (A + U).tocsr()


# ---- loads and boxes ------------------------------------------------------------------------------------
def _problem(name, S, b, lb=None, ub=None, x0=None, is_=None):
    n = len(b)
    ia, ja, a = _csr(S)
    return PR.QPProblem(name, n, 0, n, ia, ja, a, np.ascontiguousarray(b, dtype=np.float64), lb, ub,
                        np.zeros(n) if x0 is None else np.ascontiguousarray(x0, dtype=np.float64), is_=is_)


def _wave(n, f=7.0, ph=0.3):
    t = np.linspace(0.0, 1.0, n)
    return np.sin(f * np.pi * t + ph)


def lower_case(S, name, scale=1.0, depth=0.2):
    """x0 sits on a wavy lower obstacle over half of the domain; b changes sign: proportioning releases the active dofs that b pulls up,
    CG steps run on the free ones and expansions follow when b pushes them down onto the obstacle"""
    n = S.shape[0]
    lb = -depth * (1.0 + 0.5 * _wave(n, 11.0, 1.1))
    x0 = np.where(_wave(n, 3.0, 0.5) > 0, lb, 0.0)
    return _problem(name, S, scale * _wave(n, 7.0), lb=lb, x0=x0)


def case_st1d(n=4099, box="both"):
    """1-D chain (all-stencil, LMAX 3); x0 on a bound over half of the domain, a load of both signs"""
    S = lap1d(n)
    b = 0.02 * _wave(n, 5.0)
    lb = -0.05 - 0.02 * _wave(n, 9.0) ** 2
    ub = 0.05 + 0.02 * _wave(n, 13.0, 0.7) ** 2
    half = _wave(n, 3.0, 0.5) > 0
    if box == "lower":
        return Case(_problem(f"st1d_{n}_lb", S, b, lb=lb, x0=np.where(half, lb, 0.0)), kind=4)
    if box == "upper":
        return Case(_problem(f"st1d_{n}_ub", S, b, ub=ub, x0=np.where(half, ub, 0.0)), kind=4)
    if box == "inf":
        lb[::3] = PR.PETSC_NINFINITY
        ub[1::3] = INF
    if box == "is":   # bounds on every other dof of the first half only
        is_ = np.arange(0, n // 2, 2, dtype=np.int32)
        return Case(_problem(f"st1d_{n}_is", S, b, lb=lb[is_].copy(), is_=is_, x0=np.where(half, lb, 0.0)), kind=4)
    if box == "infeasible":   # x0 outside the box on both sides: projected at iteration 0
        x0 = np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
        return Case(_problem(f"st1d_{n}_x0out", S, b, lb=lb, ub=ub, x0=x0), kind=4)
    x0 = np.where(half, np.where(np.arange(n) % 2 == 0, lb, ub), 0.0)
    return Case(_problem(f"st1d_{n}_{box}", S, b, lb=lb, ub=ub, x0=np.where(np.abs(x0) < INF, x0, 0.0)), kind=4)


def case_st2d(N=128):
    return Case(PR.obstacle2d(N, -100.0), kind=4)


def case_st3d(N=32):
    return Case(PR.obstacle3d(N), kind=4)


def case_mix():
    """block diagonal: a 1-D chain (3-entry tiles) and a 2-D grid (5-entry tiles) in one all-stencil matrix (LMAX 5)"""
    import scipy.sparse as sp
    S = sp.block_diag([lap1d(3072, 4.0), lap2d(64, 64)], format="csr")   # the blocks meet at a tile boundary, same diagonal value
    return Case(lower_case(S, "mix_1d_2d", scale=0.02), kind=4)


def case_packed():
    return Case(PR.varcoef3d(24), kind=3)       # dictionary-coded tiles, both bounds, +-inf entries


def case_csr_ring():
    return Case(PR.obstacle2d(96, -100.0, scaled=True), kind=2)   # D A D: every value distinct -> plain CSR through the TMA ring


W_BANDS = {2: 0, 4: 1, 8: 3, 16: 7, 32: 13}


def case_vector(W):
    S = band_plus_rank_one(20000, W_BANDS[W])
    return Case(lower_case(S, f"vector_W{W}", scale=0.2, depth=0.05), kind=1, W=W, rtol=1e-10)


def case_ell():
    """> 2^20 non-zeros in rows of ~350 entries, 3100 rows (a partial last 256-row tile): tile-ELL"""
    import scipy.sparse as sp
    n = 3100
    R = sp.random(n, n, density=0.06, random_state=7, format="csr")
    R = abs(R + R.T)
    R.setdiag(0.0)
    R.eliminate_zeros()
    S = (-R + sp.diags(np.asarray(R.sum(axis=1)).ravel() + 1.0)).tocsr()
    return Case(lower_case(S, "ell", scale=2.0, depth=0.05), kind=5, rtol=1e-10)


def case_prod():
    pr = PR.svm_dual(3000, 400, nnz_per_row=8)
    pr.B = None
    pr.b = 0.01 * pr.b   # a proportioning step is not clipped to the box: with b = 1 the first one leaves [0, 1] far behind
    return Case(pr)


def case_small():
    return case_st1d(1001, "lower")           # 4 tiles: less than one wave


def case_large():
    return Case(PR.obstacle2d(512, -100.0), kind=4)   # 262144 rows: several waves


def case_unaligned(form):
    pr = PR.varcoef3d(20) if form == "packed" else PR.obstacle2d(80, -100.0)
    return Case(pr, kind=3 if form == "packed" else 4, devvec=True)


def eq_rows(n, m):
    t = np.arange(n) / n
    B = np.vstack([np.full(n, 1.0 / np.sqrt(n))] + [np.sin((j + 1) * np.pi * t + 0.2 * j) * np.sqrt(2.0 / n) for j in range(1, m)])
    return B


def case_eq(m, n_odd, form="aij"):
    nx, ny = (45, 47) if n_odd else (48, 48)
    S = lap2d(nx, ny)
    n = nx * ny
    pr = lower_case(S, f"eq{m}_{n}_{form}", scale=0.05, depth=0.3)
    return Case(pr, kind=4, B=eq_rows(n, m), rho=5.0, eq_form=form, driver="fused" if m <= 4 else "generic")


CASES = {
    "st1d_both": lambda: case_st1d(4099, "both"),
    "st1d_lower_even": lambda: case_st1d(4096, "lower"),
    "st1d_upper": lambda: case_st1d(4097, "upper"),
    "st1d_inf": lambda: case_st1d(3001, "inf"),
    "st1d_is": lambda: case_st1d(3000, "is"),
    "st1d_infeasible": lambda: case_st1d(3001, "infeasible"),
    "st2d": case_st2d,
    "st3d": case_st3d,
    "mix": case_mix,
    "packed": case_packed,
    "csr_ring": case_csr_ring,
    "ell": case_ell,
    "prod": case_prod,
    "small": case_small,
    "large": case_large,
    "unaligned_packed": lambda: case_unaligned("packed"),
    "unaligned_stencil": lambda: case_unaligned("stencil"),
    **{f"vector_W{W}": (lambda W=W: case_vector(W)) for W in W_BANDS},
    "eq1_onerow_odd": lambda: case_eq(1, True, "onerow"),
    "eq1_onerow_even": lambda: case_eq(1, False, "onerow"),
    "eq1_aij_odd": lambda: case_eq(1, True),
    **{f"eq{m}_{p}": (lambda m=m, p=p: case_eq(m, p == "odd")) for m in (2, 3, 4) for p in ("odd", "even")},
    **{f"eq{m}_odd": (lambda m=m: case_eq(m, True)) for m in (5, 8, 9)},
}


# ---- GPU runs -------------------------------------------------------------------------------------------
def _devvec(P, arr, keep):
    import torch
    t = torch.empty(arr.size + 2, dtype=torch.float64, device="cuda")
    v = t[1:1 + arr.size]
    v.copy_(torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float64)))
    assert v.data_ptr() % 16 == 8
    keep.append(t)
    return P.VecFromDevicePointer(v.data_ptr(), arr.size), v


def gpu_solve(P, case, options, monitor=None):
    """one MPGP solve of `case` with `options` (PETSc option string); returns a dict of the results"""
    pr = case.pr
    P.options_clear()
    P.call("PetscOptionsInsertString", None, options.encode())
    mats, vecs, keep = [], [], []
    A = P.MatCreateAIJ(pr.ia, pr.ja, pr.a, ncols_local=(pr.meta.get("d") if pr.second is not None else pr.n))
    mats.append(A)
    storage = P.MatStorageInfo(A)
    if pr.second is not None:
        A2 = P.MatCreateAIJ(pr.second[0], pr.second[1], pr.second[2], ncols_local=pr.n)
        A = P.MatCreateProd([A2, A])
        mats += [A2, A]
    xv = None
    if case.devvec:
        P.synchronize()
        b, _ = _devvec(P, pr.b, keep)
        x, xv = _devvec(P, pr.x0, keep)
        lb = _devvec(P, pr.lb, keep)[0] if pr.lb is not None else None
        ub = _devvec(P, pr.ub, keep)[0] if pr.ub is not None else None
        import torch
        torch.cuda.synchronize()
    else:
        b = P.VecFromArray(pr.b.copy())
        x = P.VecFromArray(pr.x0.copy())
        lb = P.VecFromArray(pr.lb.copy()) if pr.lb is not None else None
        ub = P.VecFromArray(pr.ub.copy()) if pr.ub is not None else None
    vecs += [b, x, lb, ub]
    is_ = P.ISCreateGeneral(pr.is_) if pr.is_ is not None else None
    qp = P.QPCreate()
    P.QPSetOperator(qp, A)
    P.QPSetRhs(qp, b)
    P.QPSetInitialVector(qp, x)
    P.QPSetBox(qp, is_, lb, ub)
    if case.B is not None:
        if case.eq_form == "onerow":
            brow = P.VecFromArray(np.ascontiguousarray(case.B[0]).copy())
            BE = P.MatCreateOneRow(brow)
            vecs.append(brow)
        else:
            BE = P.MatCreateAIJ(*_csr(case.B), ncols_local=pr.n)
        mats.append(BE)
        P.QPSetEq(qp, BE, None)
        P.call("QPTEnforceEqByPenalty", qp, C.c_double(case.rho), C.c_int(1))
    qps = P.QPSCreate()
    P.QPSSetType(qps, "mpgp")
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    if monitor is not None:
        P.QPSMonitorSet(qps, monitor)
    try:
        P.QPSSolve(qps)
        r = dict(its=P.QPSGetIterationNumber(qps), reason=P.QPSGetConvergedReason(qps), rnorm=P.QPSGetResidualNorm(qps),
                 counts=P.QPSMPGPGetStepCounts(qps), maxeig=P.QPSMPGPGetOperatorMaxEigenvalue(qps), alpha_user=P.QPSMPGPGetAlpha(qps)[0],
                 objective=P.QPComputeObjective(qp, x), storage=storage)
        if xv is not None:
            P.synchronize()
            r["x"] = xv.cpu().numpy().copy()
        else:
            r["x"] = P.VecGetArray(x)
    finally:
        P.QPSDestroy(qps)
        P.QPDestroy(qp)
        for v in vecs:
            if v is not None:
                P.VecDestroy(v)
        if is_ is not None:
            P.ISDestroy(is_)
        for m in reversed(mats):
            P.MatDestroy(m)
    return r


def gpu_runs(P, case, extra="", checkpoints=CHECKPOINTS, trace=True, maxeig=None):
    """the host-sync trace (TRACE_ITS iterations) and the folded checkpoint runs; the first run computes the largest eigenvalue, the
    later ones are handed its value"""
    drv = f"-qps_mpgp_b200_driver {case.driver} -qps_rtol {case.rtol!r} -qps_atol 1e-300 {extra}" + (f" -qps_mpgp_alpha {case.alpha!r}" if case.alpha else "")
    out = dict(trace=[], ck={})
    if trace:
        seen = []

        def mon(q, it, rnorm):
            seen.append((it, P.QPSMPGPGetCurrentStepType(q), rnorm))

        opt = f"{drv} -qps_max_it {TRACE_ITS - 1}" + (f" -qps_mpgp_maxeig {maxeig!r}" if maxeig else "")
        r = gpu_solve(P, case, opt, monitor=mon)
        out["trace"] = seen
        out["trace_run"] = r
        maxeig = maxeig or r["maxeig"]
    for k in checkpoints:
        opt = f"{drv} -qps_max_it {k}" + (f" -qps_mpgp_maxeig {maxeig!r}" if maxeig else "")
        r = gpu_solve(P, case, opt)
        maxeig = maxeig or r["maxeig"]
        out["ck"][k] = r
    out["maxeig"] = maxeig
    return out


def pack(out):
    """results -> flat dict of numpy arrays (npz)"""
    d = {"maxeig": np.array(out["maxeig"])}
    if out["trace"]:
        d["trace_it"] = np.array([t[0] for t in out["trace"]])
        d["trace_step"] = np.array([t[1] for t in out["trace"]])
        d["trace_rnorm"] = np.array([t[2] for t in out["trace"]])
        tr = out["trace_run"]
        d["trace_meta"] = np.array([tr["its"], tr["reason"], tr["alpha_user"], tr["maxeig"]], dtype=np.float64)
    for k, r in out["ck"].items():
        c = r["counts"]
        d[f"ck{k}_x"] = r["x"]
        d[f"ck{k}_int"] = np.array([r["its"], r["reason"], c["nmv"], c["ncg"], c["nexp"], c["nprop"], r["storage"]["kind"]])
        d[f"ck{k}_real"] = np.array([r["rnorm"], r["objective"], r["maxeig"]])
    return d


def unpack(d):
    out = dict(maxeig=float(d["maxeig"]), trace=[], ck={})
    if "trace_it" in d:
        out["trace"] = list(zip(d["trace_it"].tolist(), d["trace_step"].tolist(), d["trace_rnorm"].tolist()))
        m = d["trace_meta"]
        out["trace_run"] = dict(its=int(m[0]), reason=int(m[1]), alpha_user=float(m[2]), maxeig=float(m[3]))
    for key in d:
        if key.startswith("ck") and key.endswith("_x"):
            k = int(key[2:-2])
            iv, rv = d[f"ck{k}_int"], d[f"ck{k}_real"]
            out["ck"][k] = dict(x=d[key], its=int(iv[0]), reason=int(iv[1]), counts=dict(nmv=int(iv[2]), ncg=int(iv[3]), nexp=int(iv[4]), nprop=int(iv[5])),
                                storage=dict(kind=int(iv[6])), rnorm=float(rv[0]), objective=float(rv[1]), maxeig=float(rv[2]))
    return out


def main(argv):
    """CASE OUT.npz [--no-trace] [--checkpoints 0,1,...] [--maxeig V] [--options '...']"""
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("case")
    ap.add_argument("out")
    ap.add_argument("--no-trace", action="store_true")
    ap.add_argument("--checkpoints", default=",".join(map(str, CHECKPOINTS)))
    ap.add_argument("--maxeig", type=float, default=None)
    ap.add_argument("--options", default="")
    a = ap.parse_args(argv)
    from permon_b200 import api as P
    P.initialize()
    out = gpu_runs(P, CASES[a.case](), extra=a.options, checkpoints=[int(k) for k in a.checkpoints.split(",") if k], trace=not a.no_trace,
                   maxeig=a.maxeig)
    np.savez(a.out, **pack(out))
    P.options_clear()


if __name__ == "__main__":
    main(sys.argv[1:])
