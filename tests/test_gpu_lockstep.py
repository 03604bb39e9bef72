"""Lockstep tests: the fused MPGP kernels against the oracle along the iteration, not only at the converged solution.

MPGP corrects its own errors, so a kernel bug that changes the path (a wrong feasible step, a dropped equality row, a bound read from the
wrong element) still converges to the right x and passes a converged-solution parity test.  Here every variant that the input data selects
(SpMV form, box, vector layout, equality rows through the fused rank-m update) is compared with the oracle (nthreads = 1)

* per iteration in the host-sync schedule (a monitor is set): step kind, ||gP|| and alpha, for TRACE_ITS iterations;
* at checkpoints k of the folded device-driven schedule (`-qps_max_it k`, tolerances off): iteration count, reason and step counts
  exactly, the iterate, ||gP|| and the objective to a relative tolerance.

Every case forces its driver (`-qps_mpgp_b200_driver fused`, which errors when the case is not eligible, or `generic`) and asserts the
storage kind of its Hessian, so that a test cannot silently run another kernel than the one it is about.

Past some iteration the oracle itself no longer reproduces its own path when only its summation order changes (thread counts 2, 3, 5,
8): an active-set decision turns on the last bits.  `oracle_trace_band` measures that spread per iteration; a deviation above the base
tolerance is accepted up to 10x the spread at that iteration, and the comparison ends at the first iteration where that would exceed
MAX_TOL = 1e-9 or where the oracle's step kinds flip (the horizon, at least MIN_HORIZON iterations unless the solve converges first).

Measured on one B200 (1000 W power limit), the largest deviations over the whole file:
  x at a checkpoint          3.7e-12  (prod; 2.8e-12 large, 2.5e-12 small, all others <= 6.0e-13)      X_TOL  = 5e-11
  ||gP|| at a checkpoint     1.4e-11  (ell, within 10x the oracle's spread; all others <= 8.7e-12)      RN_TOL = 1e-10
  ||gP|| along a trace       1.3e-10  (eq2_odd at its horizon, within 10x the oracle's spread; 8.9e-11 small, 5.7e-11 eq5_odd,
                                       3.8e-11 csr_ring, all others <= 2.0e-11)
  objective                  3.9e-12  (prod; all others <= 2.8e-13)                                      F_TOL  = 5e-11
  one iteration vs. the extended-precision reference: 0.15 eps * sum|terms| (eq2-p)                     STEP_ULPS = 8
Horizons: 51 (the whole trace) except st1d_is 33, st3d 32, prod 30, eq5_odd 38, eq2_odd 40, small 41, large 45; vector_W4..W32 and
ell converge (rtol 1e-10) after 16-27 iterations.

Kernel instantiation per case (lockstep_worker.CASES): st1d_* / small: all-stencil LMAX 3 (odd n: scalar K_B / K_C, even n: double2);
st2d / large / unaligned_stencil / eq*: all-stencil LMAX 5; st3d: LMAX 7; mix: LMAX 5 with 3-entry tiles; packed / unaligned_packed:
dictionary-coded tiles (kind 3); csr_ring: CSR through the TMA ring (kind 2); vector_W*: k_spmv_vector<W>; ell: tile-ELL (kind 5);
prod: two CSR factors (M1 M2); unaligned_*: caller vectors only 8-byte aligned (plain loads instead of TMA); eq1..eq4: the fused rank-m update
(EQ = true); eq5 / eq8 / eq9: the generic driver with dense equality rows.  The A/B switches (test_ab_switch_lockstep) reach
SD_PAIRS / ST_KERNEL=windows (stencil kernels), NOVEC (scalar K_B / K_C), STAGES / PK_OCC (TMA ring and packed tiles), SPMV=stream
(kind 0) / vector (kind 1, W = 4) / tma (kind 2) and NOELL (k_spmv_vector<32> instead of tile-ELL).

The extended-precision one-iteration reference at the end (`one_step_reference`) is a NumPy restatement of one MPGP iteration that does not
share code with the oracle; its CPU test checks the oracle's first iterate, its GPU test the library's.
"""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import lockstep_worker as L
from oracle import oracle_py as O

HERE = os.path.dirname(os.path.abspath(__file__))
EPS = np.finfo(np.float64).eps
X_TOL = 5e-11      # || x_gpu - x_oracle || / || x_oracle || at a checkpoint
RN_TOL = 1e-10     # | rnorm_gpu - rnorm_oracle | / rnorm_oracle, per iteration and at a checkpoint
F_TOL = 5e-11      # objective, relative
MAX_TOL = 1e-9     # never looser than this: past the iteration where the oracle's own spread needs more, the comparison stops
MIN_HORIZON = 30   # ... and that must not happen before this iteration
BAND_THREADS = (2, 3, 5, 8)
STEP_ULPS = 8      # one iteration against the extended-precision reference, in units of eps * (sum of |terms|)

# largest deviations seen, per case (written to $PERMON_LOCKSTEP_REPORT at the end of the module when set)
REPORT = {}


@pytest.fixture(scope="module")
def P():
    from permon_b200 import api
    if api.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    api.initialize()
    yield api
    api.options_clear()
    path = os.environ.get("PERMON_LOCKSTEP_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)


# ---- oracle side ----------------------------------------------------------------------------------------
def oracle_op(case, penalty=True):
    pr = case.pr
    op = O.Operator(pr.ia, pr.ja, pr.a, second=pr.second)
    if penalty and case.B is not None:
        op.set_penalty(case.B, case.rho)
    return op


def oracle_run(case, max_it, maxeig, trace_cap=0, nthreads=1):
    pr = case.pr
    op = oracle_op(case)
    kw = dict(max_it=max_it, rtol=case.rtol, atol=1e-300, maxeig=maxeig, nthreads=nthreads)
    if case.alpha:
        kw["alpha_user"] = case.alpha
    x, r = O.mpgp_solve(op, pr.b, O.BoxC(pr.n, pr.lb, pr.ub, pr.is_), pr.x0, O.mpgp_opts(**kw), trace_cap=trace_cap)
    r["objective"] = O.objective(oracle_op(case, penalty=False), pr.b, x)
    return x, r


def vector_bucket(pr):
    """lanes per row of k_spmv_vector for this matrix (kernels.cu: spmv_config)"""
    avg = len(pr.a) / pr.n
    return 2 if avg <= 3 else 4 if avg <= 6 else 8 if avg <= 12 else 16 if avg <= 24 else 32


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


def oracle_trace_band(case, me):
    """the oracle's own spread along the trace over thread counts (= summation orders): relative spread of ||gP|| per iteration and the
    horizon, the first iteration at which the spread reaches MAX_TOL / 10 or a step kind flips.  Past the horizon the iteration is
    decided by rounding, and no implementation can be held to the oracle's path."""
    _, r1 = oracle_run(case, L.TRACE_ITS - 1, me, trace_cap=L.TRACE_ITS + 1)
    t1 = r1["trace"]
    band = np.zeros(len(t1["rnorm"]))
    horizon = len(band)
    for nt in BAND_THREADS:
        _, r = oracle_run(case, L.TRACE_ITS - 1, me, trace_cap=L.TRACE_ITS + 1, nthreads=nt)
        t = r["trace"]
        k = min(len(t["rnorm"]), len(band))
        band[:k] = np.maximum(band[:k], np.abs(t["rnorm"][:k] - t1["rnorm"][:k]) / np.maximum(t1["rnorm"][:k], 1e-300))
        flip = next((i for i, (a, b) in enumerate(zip(t["step"], t1["step"])) if a != b), min(len(t["step"]), len(t1["step"])))
        horizon = min(horizon, flip, k)
    wild = np.nonzero(10 * band > MAX_TOL)[0]
    if len(wild):
        horizon = min(horizon, int(wild[0]))
    return band, horizon


def check_lockstep(name, case, res, kind=None):
    """res: L.gpu_runs output.  Compares with the oracle at every traced iteration and every checkpoint up to the horizon of the oracle's
    own reproducibility (oracle_trace_band); a deviation above the base tolerance is accepted up to 10x the oracle's spread there."""
    me = res["maxeig"]
    rep = REPORT.setdefault(name, dict(x=0.0, rnorm_trace=0.0, rnorm_ck=0.0, objective=0.0, horizon=None, band_used=0))
    kind = case.kind if kind is None else kind
    for k, r in res["ck"].items():
        if kind is not None:
            assert r["storage"]["kind"] == kind, (k, r["storage"])
    band, horizon = oracle_trace_band(case, me)
    rep["horizon"] = horizon
    assert horizon >= MIN_HORIZON or horizon == len(band), horizon
    if res["trace"]:
        xo, ro = oracle_run(case, L.TRACE_ITS - 1, me, trace_cap=L.TRACE_ITS + 1)
        t = ro["trace"]
        tr = res["trace_run"]
        if horizon == len(band):
            assert (tr["its"], tr["reason"]) == (ro["its"], ro["reason"])
            assert len(res["trace"]) == len(t["step"])
        steps = "".join(s for _, s, _ in res["trace"])[:horizon]
        assert steps == t["step"][:horizon], f"step kinds differ at iteration {next(i for i, (a, b) in enumerate(zip(steps, t['step'])) if a != b)}: {steps} vs {t['step']}"
        assert [s[0] for s in res["trace"]] == list(range(len(res["trace"])))
        rn = np.array([s[2] for s in res["trace"]])[:horizon]
        dev = np.abs(rn - t["rnorm"][:horizon]) / np.maximum(t["rnorm"][:horizon], 1e-300)
        tol = np.maximum(RN_TOL, 10 * band[:horizon])
        rep["rnorm_trace"] = max(rep["rnorm_trace"], float(dev.max()))
        rep["band_used"] += int(np.count_nonzero(dev > RN_TOL))
        assert np.all(dev <= tol), (int(np.argmax(dev / tol)), float(dev.max()))
        assert tr["alpha_user"] / tr["maxeig"] == pytest.approx(t["alpha"][0], rel=1e-15)
        assert tr["maxeig"] == pytest.approx(O.max_eigenvalue(oracle_op(case))[0], rel=1e-10)   # the GPU power method
    for k, r in res["ck"].items():
        if k + 1 >= horizon and horizon < len(band):
            continue
        xo, ro = oracle_run(case, k, me)
        got = (r["its"], r["reason"], r["counts"]["nmv"], r["counts"]["ncg"], r["counts"]["nexp"], r["counts"]["nprop"])
        assert got == (ro["its"], ro["reason"], ro["nmv"], ro["ncg"], ro["nexp"], ro["nprop"]), (k, got)
        nx = max(np.linalg.norm(xo), 1e-300)
        dx, drn, dobj = np.linalg.norm(r["x"] - xo) / nx, _rel(r["rnorm"], ro["rnorm"]), _rel(r["objective"], ro["objective"])
        rep["x"], rep["rnorm_ck"], rep["objective"] = max(rep["x"], float(dx)), max(rep["rnorm_ck"], drn), max(rep["objective"], dobj)
        tx, trn, tobj = X_TOL, RN_TOL, F_TOL
        if dx > X_TOL or drn > RN_TOL or dobj > F_TOL:   # the oracle's own spread at this checkpoint
            rep["band_used"] += 1
            bx = brn = bobj = 0.0
            for nt in BAND_THREADS:
                xt, rt = oracle_run(case, k, me, nthreads=nt)
                bx = max(bx, np.linalg.norm(xt - xo) / nx)
                brn, bobj = max(brn, _rel(rt["rnorm"], ro["rnorm"])), max(bobj, _rel(rt["objective"], ro["objective"]))
            tx, trn, tobj = (min(MAX_TOL, max(t0, 10 * b)) for t0, b in ((X_TOL, bx), (RN_TOL, brn), (F_TOL, bobj)))
        assert dx <= tx, (k, dx, tx)
        assert drn <= trn, (k, r["rnorm"], ro["rnorm"], trn)
        assert dobj <= tobj, (k, r["objective"], ro["objective"], tobj)


# ---- 1. + 2. A-D: the production paths chosen by the data ---------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(L.CASES))
def test_lockstep(P, name):
    case = L.CASES[name]()
    if case.W is not None:
        assert np.diff(case.pr.ia).max() > 64 and len(case.pr.a) < (1 << 20)      # lanes-per-row kernel, not tile-ELL
        assert vector_bucket(case.pr) == case.W
    if case.B is not None:
        assert case.driver == ("fused" if case.B.shape[0] <= 4 else "generic")
    res = L.gpu_runs(P, case)
    check_lockstep(name, case, res)


@pytest.mark.gpu
def test_fused_driver_accepts_four_equality_rows_and_refuses_five(P):
    """the fused rank-m update keeps PB_MAXEQ = 4 accumulators; a fifth row takes the un-fused route, and forcing the fused driver is an error"""
    ok = L.gpu_solve(P, L.case_eq(4, True), f"-qps_mpgp_b200_driver fused -qps_max_it 3 {L.NOTOL}")
    assert ok["its"] == 4
    with pytest.raises(P.PermonError) as e:
        L.gpu_solve(P, L.case_eq(5, True), f"-qps_mpgp_b200_driver fused -qps_max_it 3 {L.NOTOL}")
    assert e.value.code == 56   # PETSC_ERR_SUP


# ---- E. schedule invariants ----------------------------------------------------------------------------------
def _same(a, b):
    return (a["its"], a["reason"], a["counts"], a["rnorm"]) == (b["its"], b["reason"], b["counts"], b["rnorm"]) and np.array_equal(a["x"], b["x"])


def _subprocess(tmp_path, name, env, args):
    out = tmp_path / f"{name}.npz"
    e = {**os.environ, **env}
    p = subprocess.run([sys.executable, os.path.join(HERE, "lockstep_worker.py"), name, str(out), *args], env=e, capture_output=True, text=True,
                       timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    return L.unpack(dict(np.load(out)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["st2d", "eq3_odd"])
def test_schedule_variants_are_bit_identical(P, name, monkeypatch, tmp_path):
    """batch size, monitor on / off, stand-alone control kernels and PDL off launch the same grids with the same reduction trees
    (DESIGN section 3): the iterate must be identical bit for bit"""
    case = L.CASES[name]()
    K = 34
    base = L.gpu_runs(P, case, checkpoints=[K], trace=False)
    me = base["maxeig"]
    ref = base["ck"][K]
    drv = f"-qps_mpgp_b200_driver {case.driver} -qps_rtol {case.rtol!r} -qps_atol 1e-300 -qps_max_it {K} -qps_mpgp_maxeig {me!r}"
    variants = {f"batch {b}": L.gpu_solve(P, case, f"{drv} -qps_mpgp_b200_batch {b}") for b in (1, 7, 16)}
    variants["monitor"] = L.gpu_solve(P, case, drv, monitor=lambda q, it, rn: None)
    monkeypatch.setenv("PERMON_B200_NOFOLD", "1")
    variants["NOFOLD"] = L.gpu_solve(P, case, drv)
    monkeypatch.delenv("PERMON_B200_NOFOLD")
    variants["PDL=0"] = _subprocess(tmp_path, name, {"PERMON_B200_PDL": "0"}, ["--no-trace", "--checkpoints", str(K), "--maxeig", repr(me)])["ck"][K]
    for v, r in variants.items():
        assert _same(r, ref), v


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["st2d", "eq3_odd"])
def test_serpentine_off_stays_in_lockstep(P, name, monkeypatch):
    """PERMON_B200_SERPENTINE=0 runs every K_B forwards: other summation order, the same iteration within the lockstep tolerance"""
    monkeypatch.setenv("PERMON_B200_SERPENTINE", "0")
    case = L.CASES[name]()
    check_lockstep(f"{name}+SERPENTINE=0", case, L.gpu_runs(P, case))


# ---- F. A/B switches, each in a fresh process -----------------------------------------------------------------
SWITCHES = [
    ("PERMON_B200_SD_PAIRS", "1", "st2d", 4),
    ("PERMON_B200_ST_KERNEL", "windows", "st3d", 4),
    ("PERMON_B200_NOVEC", "1", "st2d", 4),
    ("PERMON_B200_STAGES", "1", "csr_ring", 2),
    ("PERMON_B200_STAGES", "2", "packed", 3),
    ("PERMON_B200_STAGES", "4", "csr_ring", 2),
    ("PERMON_B200_PK_OCC", "4", "packed", 3),
    ("PERMON_B200_SPMV", "stream", "st2d", 0),
    ("PERMON_B200_SPMV", "vector", "st2d", 1),
    ("PERMON_B200_SPMV", "tma", "st2d", 2),
    ("PERMON_B200_NOELL", "1", "ell", 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("var,val,name,kind", SWITCHES, ids=[f"{v[len('PERMON_B200_'):]}={x}-{n}" for v, x, n, _ in SWITCHES])
def test_ab_switch_lockstep(P, tmp_path, var, val, name, kind):
    case = L.CASES[name]()
    res = _subprocess(tmp_path, name, {var: val}, [])
    check_lockstep(f"{name}+{var}={val}", case, res, kind=kind)


# ---- 3. one MPGP iteration in extended precision ---------------------------------------------------------------
def _exact_dot(u, v):
    """sum of u_i v_i: products in long double, each split into two doubles, summed exactly by math.fsum (result to ~2^-100)"""
    t = np.asarray(u, dtype=np.longdouble) * np.asarray(v, dtype=np.longdouble)
    hi = t.astype(np.float64)
    lo = (t - hi).astype(np.float64)
    parts = np.concatenate([hi, lo]).tolist()
    s = math.fsum(parts)
    return np.longdouble(s) + np.longdouble(math.fsum(parts + [-s]))


def one_step_reference(ia, ja, a, b, x0, lb=None, ub=None, B=None, rho=0.0, alpha=None):
    """One MPGP iteration (standard expansion, fixed length, gamma = 1) from x0, in np.longdouble: g = A x - b (+ rho B'B x), the gf / gc
    split of the box, then a CG, expansion or proportioning step.  Returns (step, x1, scale): |x1 - x1_exact| of a double-precision
    implementation is a few eps * scale (scale: the sums of |terms| that x1 is made of)."""
    LD = np.longdouble
    n = len(b)
    rows = np.repeat(np.arange(n), np.diff(ia))
    aL = np.asarray(a, dtype=LD)
    BL = None if B is None else np.asarray(B, dtype=LD).reshape(-1, n)

    def matvec(v, absolute=False):
        av = np.abs(aL) if absolute else aL
        vv = np.abs(v) if absolute else v
        y = np.zeros(n, dtype=LD)
        np.add.at(y, rows, av * vv[ja])
        if BL is not None:
            Bv = np.abs(BL) if absolute else BL
            t = np.array([_exact_dot(Bv[j], vv) for j in range(len(Bv))], dtype=LD)
            y += LD(rho) * (Bv.T @ t)
        return y

    astol = 10 * EPS
    lbL = None if lb is None else np.asarray(lb, dtype=LD)
    ubL = None if ub is None else np.asarray(ub, dtype=LD)

    def grads(x, g):
        gf, gc = g.copy(), np.zeros(n, dtype=LD)
        al = np.zeros(n, bool) if lbL is None else np.abs(x - lbL) <= astol
        au = (np.zeros(n, bool) if ubL is None else np.abs(x - ubL) <= astol) & ~al
        gf[al | au] = 0
        gc[al] = np.minimum(g[al], 0)
        gc[au] = np.maximum(g[au], 0)
        return gf, gc

    def feas(x, p):
        af = LD(np.inf)
        if lbL is not None:
            k = (p > 0) & (lbL > O.NINFINITY)
            if k.any():
                af = min(af, np.min((x[k] - lbL[k]) / p[k]))
        if ubL is not None:
            k = (p < 0) & (ubL < O.INFINITY)
            if k.any():
                af = min(af, np.min((x[k] - ubL[k]) / p[k]))
        return af

    x = np.asarray(x0, dtype=LD).copy()
    if lbL is not None:
        x = np.maximum(x, lbL)
    if ubL is not None:
        x = np.minimum(x, ubL)
    bL = np.asarray(b, dtype=LD)
    g = matvec(x) - bL
    gabs = matvec(x, True) + np.abs(bL)               # bound on the terms of g
    gf, gc = grads(x, g)
    if _exact_dot(gc, gc) <= _exact_dot(gf, gf):
        p = gf
    else:
        p = gc
    Ap = matvec(p)
    pAp = _exact_dot(p, Ap)
    gp = _exact_dot(g, p)
    acg = gp / pAp
    kappa = _exact_dot(gabs, np.abs(p)) / abs(gp) + _exact_dot(np.abs(p), matvec(p, True)) / abs(pAp)
    if p is gc:
        step = "p"
    else:
        afeas = feas(x, p)
        step = "c" if acg <= afeas else "e"
    if step in "cp":
        x1 = x - acg * p
        scale = np.abs(x) + np.abs(acg * p) * (1 + kappa)
    else:
        xe = x - afeas * p
        ge = g - afeas * Ap
        gfe, _ = grads(xe, ge)
        gr = gfe.copy()
        if lbL is not None:
            k = gfe > 0
            gr[k] = np.minimum(gfe[k], (xe[k] - lbL[k]) / LD(alpha))
        if ubL is not None:
            k = gfe < 0
            gr[k] = np.maximum(gfe[k], (xe[k] - ubL[k]) / LD(alpha))
        x1 = xe - LD(alpha) * gr
        scale = np.abs(x) + np.abs(afeas * p) + LD(alpha) * (gabs + np.abs(afeas) * matvec(np.abs(p), True))
    return step, x1, scale


def one_step_cases():
    """(name, step, case): 1-D chain and the 2-D grid with two penalised equality rows; x0 and the box chosen so that the first step is a
    CG step (obstacle far away), an expansion (obstacle close below) or a proportioning step (x0 on the obstacle, the load pulls it off)"""
    out = []
    for base in ("chain", "eq2"):
        for step in "cep":
            if base == "chain":
                S = L.lap1d(5001)
                n = 5001
            else:
                S = L.lap2d(45, 47)
                n = 45 * 47
            w = L._wave(n, 7.0)
            lb = {"c": -10.0, "e": -1e-3, "p": -0.01}[step] * (1.0 + 0.3 * L._wave(n, 11.0) ** 2)
            b = {"c": 0.02 * w, "e": -0.5 * (1.0 + 0.5 * w), "p": 0.02 * (1.2 + w)}[step]
            x0 = lb.copy() if step == "p" else np.zeros(n)
            pr = L._problem(f"onestep_{base}_{step}", S, b, lb=lb, x0=x0)
            case = L.Case(pr, kind=4) if base == "chain" else L.Case(pr, kind=4, B=L.eq_rows(n, 2), rho=5.0)
            out.append((f"{base}-{step}", step, case))
    return out


ONE_STEP = one_step_cases()


def _one_step_check(case, step, x1):
    pr = case.pr
    me = O.max_eigenvalue(oracle_op(case))[0]
    s, xr, scale = one_step_reference(pr.ia, pr.ja, pr.a, pr.b, pr.x0, pr.lb, pr.ub, case.B, case.rho, alpha=2.0 / me)
    assert s == step
    err = np.abs(np.asarray(x1, dtype=np.longdouble) - xr) / scale
    return float(err.max() / EPS)


@pytest.mark.parametrize("name,step,case", ONE_STEP, ids=[c[0] for c in ONE_STEP])
def test_one_step_reference_against_oracle(name, step, case):
    """CPU: the oracle's first iterate (max_it 0 = one iteration) within a few eps of the extended-precision restatement"""
    me = O.max_eigenvalue(oracle_op(case))[0]
    x1, r = oracle_run(case, 0, me, trace_cap=4)
    assert r["trace"]["step"] == " " + step and r["its"] == 1
    ulps = _one_step_check(case, step, x1)
    assert ulps <= STEP_ULPS, ulps


@pytest.mark.gpu
@pytest.mark.parametrize("name,step,case", ONE_STEP, ids=[c[0] for c in ONE_STEP])
def test_one_step_gpu_against_extended_precision(P, name, step, case):
    me = O.max_eigenvalue(oracle_op(case))[0]
    seen = []
    r = L.gpu_solve(P, case, f"-qps_mpgp_b200_driver fused {L.NOTOL} -qps_max_it 0 -qps_mpgp_maxeig {me!r}",
                    monitor=lambda q, it, rn: seen.append(P.QPSMPGPGetCurrentStepType(q)))
    assert r["storage"]["kind"] == 4 and r["its"] == 1 and seen == [" ", step]
    r = L.gpu_solve(P, case, f"-qps_mpgp_b200_driver fused {L.NOTOL} -qps_max_it 0 -qps_mpgp_maxeig {me!r}")   # folded schedule
    ulps = _one_step_check(case, step, r["x"])
    REPORT.setdefault("one_step_ulps", {})[name] = ulps
    assert ulps <= STEP_ULPS, ulps


# ---- 4. SpMV only --------------------------------------------------------------------------------------------------
def _spmv_check(P, ia, ja, a, n, kind=None):
    import scipy.sparse as sp
    rng = np.random.default_rng(21)
    x = rng.standard_normal(n)
    A = P.MatCreateAIJ(ia, ja, a)
    info = P.MatStorageInfo(A)
    vx, vy = P.VecFromArray(x.copy()), P.VecCreate(n)
    P.MatMult(A, vx, vy)
    y = P.VecGetArray(vy)
    P.VecDestroy(vx), P.VecDestroy(vy), P.MatDestroy(A)
    rows = np.repeat(np.arange(n), np.diff(ia))
    yr = np.zeros(n, dtype=np.longdouble)
    np.add.at(yr, rows, np.asarray(a, dtype=np.longdouble) * np.asarray(x, dtype=np.longdouble)[ja])
    scale = np.abs(sp.csr_matrix((np.abs(a), ja, ia), shape=(n, n)) @ np.abs(x)) + 1e-300
    err = float(np.max(np.abs(np.asarray(y, dtype=np.longdouble) - yr) / scale))
    if kind is not None:
        assert info["kind"] == kind, info
    return err, info


@pytest.mark.gpu
@pytest.mark.parametrize("offs", [(-1, 0, 1, 2), (-64, -1, 0, 1, 3, 64), (-130, -65, -1, 0, 1, 2, 65, 131)], ids=["4pt", "6pt", "8pt"])
def test_spmv_nonsymmetric_stencils(P, offs):
    """non-symmetric constant-coefficient stencils: all-stencil form, pattern lengths 4 / 6 / 8 (LMAX 5 / 7 / 8: the predicated loop)"""
    import scipy.sparse as sp
    n = 70001
    vals = [1.0 + 0.25 * k - 0.5 * (d < 0) for k, d in enumerate(offs)]
    S = sp.diags([np.full(n - abs(d), v) for d, v in zip(offs, vals)], list(offs), format="csr")
    ia, ja, a = L._csr(S)
    err, _ = _spmv_check(P, ia, ja, a, n, kind=4)
    assert err <= 4 * EPS, err


@pytest.mark.gpu
@pytest.mark.parametrize("W", sorted(L.W_BANDS))
def test_spmv_lanes_per_row_buckets(P, W):
    ia, ja, a = L._csr(L.band_plus_rank_one(20000, L.W_BANDS[W]))
    pr = L.PR.QPProblem("v", 20000, 0, 20000, ia, ja, a, np.zeros(20000), None, None, np.zeros(20000))
    assert vector_bucket(pr) == W
    err, _ = _spmv_check(P, ia, ja, a, 20000, kind=1)
    assert err <= 8 * EPS, err


@pytest.mark.gpu
def test_spmv_many_patterns_leaves_all_stencil_form(P):
    """tiles with more than 32 distinct row patterns do not fit the all-stencil form: the matrix falls back to another kind, same products"""
    import scipy.sparse as sp
    n = 40000
    rng = np.random.default_rng(8)
    offs = [0, 1, -1] + [int(d) for d in rng.choice(np.arange(2, 400), 60, replace=False)]
    S = sp.diags([np.full(n, 4.0)], [0], format="csr")
    pat = rng.integers(0, len(offs), size=(n, 3))        # each row: the diagonal and up to three other offsets out of 63
    r = np.repeat(np.arange(n), 3)
    c = np.clip(r + np.array(offs)[pat.ravel()], 0, n - 1)
    S = (S + sp.csr_matrix((np.full(len(r), -1.0), (r, c)), shape=(n, n))).tocsr()
    S.sum_duplicates()
    ia, ja, a = L._csr(S)
    err, info = _spmv_check(P, ia, ja, a, n)
    assert info["kind"] != 4, info
    assert err <= 4 * EPS, err
