"""Dense Hessians on one GPU: the dense stored form (MatCreateSeqDenseCUDA, kind 6) against the AIJ form of the same matrix
(MatB200CreateAIJWithDeviceArrays, tile-ELL), wherever n^2 < 2^31 lets AIJ hold it.

    python profiles/dense_bench.py [--sizes 8192,16384,32768,46000,65536,100000] [--mixed-sizes 16384,32768] [--warmup 20] [--its 200]
                                   [--svm 32768] [--out FILE]

D1 (MPGP, lower bound 0): an RBF kernel K_ij = exp(-|p_i - p_j|^2 / 8) of n points p in R^8 (standard normal) plus 1e-3 I, b standard
normal -- all generated on the device from fixed seeds with torch fp64.  D1 takes expansion steps only; D1-mixed (the same matrices,
b = K z with z ~ N(0.5, 1)) mixes CG, expansion and proportioning steps, so that the CG-step path (K_A + the c step of K_B) is timed too.
D2 (SMALXE): the kernel-SVM dual diag(y) K diag(y) + 1e-3 I, 0 <= a <= 1, y^T a = 0.  For each size and form: MPGP iterations per second over --its timed iterations after --warmup iterations
(tolerances off; CUDA events recorded on the library stream around QPSSolve), the c / e / p step counts of the timed window, set-up time
(construction + power method), and for the dense form the per-launch time of K_A (the fused SpMV of the MPGP iteration) from the
library's profiler with its bytes (8 n^2 + the epilogue vectors) over that time as a share of the device-to-device copy bandwidth
measured in the same run (a 4 GB torch copy: read + write bytes over time).  Parity: at n = 8192 the dense iterate of one uninterrupted
solve of --parity-its iterations against the oracle's (the timed window restarts MPGP after the warm-up, which the oracle does not).
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:   # pragma: no cover
        return dict(error=str(e))


def copy_bandwidth(torch):
    a = torch.empty(512 * 1024 * 1024, dtype=torch.float64, device="cuda")   # 4 GB, far beyond L2
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    sec = e0.elapsed_time(e1) / 1e3 / reps
    nbytes = 2 * a.numel() * 8
    del a, b
    torch.cuda.empty_cache()
    return nbytes / sec


def rbf(torch, n, seed, ridge=1e-3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    p = torch.randn(n, 8, generator=g, dtype=torch.float64, device="cuda")
    sq = (p * p).sum(1)
    K = p @ p.t()
    for r0 in range(0, n, 2048):   # in place, row blocks: no second n x n buffer; sq_i + sq_j is symmetric in i, j bit for bit
        K[r0:r0 + 2048].mul_(2.0).sub_(sq[r0:r0 + 2048, None] + sq[None, :]).clamp_(max=0.0).mul_(1.0 / 8.0).exp_()
    K.diagonal().add_(ridge)
    b = torch.randn(n, generator=g, dtype=torch.float64, device="cuda")
    return K, b


def make_mat(P, torch, K, form):
    """(Mat, construction seconds): K is symmetric, so its row-major storage is its own column-major form (K.t() is adopted)"""
    n = K.shape[0]
    torch.cuda.synchronize()
    P.synchronize()
    t0 = time.perf_counter()
    if form == "dense":
        A = P.MatCreateDenseFromTensor(K.t())
        P.MatDenseGetInfo(A)   # first use: adoption / device form
    else:
        ia = torch.arange(0, (n + 1) * n, n, dtype=torch.int32, device="cuda")
        ja = torch.arange(n, dtype=torch.int32, device="cuda").repeat(n)
        A = P.MatCreateAIJFromDeviceTensors(ia, ja, K.reshape(-1))
        del ia, ja
    P.synchronize()
    return A, time.perf_counter() - t0


def mpgp_window(P, torch, A, b_np, n, warmup, its, ub=None, B=None, profile=False):
    """MPGP (or SMALXE with B) from x = 0: set-up (power method) timed, then warm-up, then the timed window continued from the warm-up
    iterate (a second QPSSolve resumes from the resident x); returns rates, counts, final x"""
    P.options_clear()
    P.call("PetscOptionsInsertString", None, b"-qps_rtol 1e-300 -qps_atol 1e-300")
    x = P.VecFromArray(np.zeros(n))
    b = P.VecFromArray(np.ascontiguousarray(b_np))
    lb = P.VecFromArray(np.zeros(n))
    vub = P.VecFromArray(np.ascontiguousarray(ub)) if ub is not None else None
    qp = P.QPCreate()
    P.QPSetOperator(qp, A), P.QPSetRhs(qp, b), P.QPSetInitialVector(qp, x), P.QPSetBox(qp, None, lb, vub)
    keep = []
    if B is not None:
        brow = P.VecFromArray(np.ascontiguousarray(B))
        BE = P.MatCreateOneRow(brow)
        P.QPSetEq(qp, BE, None)
        keep = [brow, BE]
    qps = P.QPSCreate()
    P.QPSSetType(qps, "smalxe" if B is not None else "mpgp")
    P.QPSSetQP(qps, qp)
    P.QPSSetFromOptions(qps)
    out = {}
    if B is None:
        P.QPSSetTolerances(qps, maxits=warmup)
        P.synchronize()
        t0 = time.perf_counter()
        P.QPSSetUp(qps)
        P.synchronize()
        out["power_method_s"] = time.perf_counter() - t0
        P.QPSSolve(qps)
        c0 = P.QPSMPGPGetStepCounts(qps)
        out["warmup_steps"] = c0
        if its == 0:
            out["x"] = P.VecGetArray(x).copy()
            its = None
    if B is None and its is not None:
        P.QPSSetTolerances(qps, maxits=its)
        stream = torch.cuda.ExternalStream(P.get_stream())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        P.synchronize()
        if profile:
            P.profile_begin()
        e0.record(stream)
        P.QPSSolve(qps)
        e1.record(stream)
        e1.synchronize()
        if profile:
            out["profile"] = {k: v for k, v in P.profile_end().items() if v["launches"]}
        sec = e0.elapsed_time(e1) / 1e3
        c1 = P.QPSMPGPGetStepCounts(qps)
        k = P.QPSGetIterationNumber(qps)
        out.update(iterations=k, seconds=sec, it_per_s=k / sec, steps={s: c1[s] - c0.get(s, 0) for s in c1})
    elif B is not None:
        P.QPSSetTolerances(qps, rtol=1e-6)
        P.synchronize()
        t0 = time.perf_counter()
        P.QPSSolve(qps)
        P.synchronize()
        sec = time.perf_counter() - t0
        st = P.QPSSMALXEGetStatistics(qps)
        inner = P.QPSSMALXEGetInnerQPS(qps)
        out.update(outer_its=P.QPSGetIterationNumber(qps), inner_its=st["inner_iter_accu"], seconds=sec, inner_it_per_s=st["inner_iter_accu"] / sec,
                   steps=P.QPSMPGPGetStepCounts(inner), reason=P.QPSGetConvergedReason(qps))
    out.setdefault("x", P.VecGetArray(x).copy())
    P.QPSDestroy(qps), P.QPDestroy(qp)
    for v in (x, b, lb, vub):
        if v is not None:
            P.VecDestroy(v)
    if keep:
        P.VecDestroy(keep[0]), P.MatDestroy(keep[1])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="8192,16384,32768,46000,65536,100000")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--its", type=int, default=200)
    ap.add_argument("--mixed-sizes", default="16384,32768")
    ap.add_argument("--svm", type=int, default=32768)
    ap.add_argument("--parity-n", type=int, default=8192)
    ap.add_argument("--parity-its", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from permon_b200 import api as P
    if P.device_count() == 0:
        raise SystemExit("needs a CUDA device")
    P.initialize()
    res = dict(card=card(), warmup=args.warmup, its=args.its, copy_bw_bytes_per_s=copy_bandwidth(torch), d1={}, d1_mixed={}, d2={})
    print(json.dumps({k: res[k] for k in ("card", "copy_bw_bytes_per_s")}), flush=True)
    jobs = [("d1", int(v)) for v in args.sizes.split(",") if v] + [("d1_mixed", int(v)) for v in args.mixed_sizes.split(",") if v]
    for key, n in jobs:
        K, b = rbf(torch, n, seed=n)
        if key == "d1_mixed":   # b = K z with z ~ N(0.5, 1): an unconstrained minimiser z, about a third of it below the bound
            g = torch.Generator(device="cuda").manual_seed(n + 1)
            b = K @ torch.randn(n, generator=g, dtype=torch.float64, device="cuda").add_(0.5)
        b_np = b.cpu().numpy()
        row = dict(n=n, matrix_bytes=8.0 * n * n)
        forms = ["dense"] + (["aij"] if n * n < 2 ** 31 else [])
        for form in forms:
            A, t_ctor = make_mat(P, torch, K, form)
            r = mpgp_window(P, torch, A, b_np, n, args.warmup, args.its, profile=(form == "dense"))
            r["construct_s"] = t_ctor
            r["setup_s"] = t_ctor + r["power_method_s"]
            r["storage"] = P.MatStorageInfo(A)
            if form == "dense":
                r["dense_info"] = P.MatDenseGetInfo(A)
                ka = r["profile"].get("K_A spmv+dots+feas")
                if ka:
                    per = ka["working_ms"] / max(ka["working_launches"], 1) / 1e3
                    r["K_A"] = dict(launches=ka["working_launches"], ms_per_launch=1e3 * per, bytes_per_launch=ka["bytes_per_launch"],
                                    bytes_per_s=ka["bytes_per_launch"] / per, share_of_copy_bw=ka["bytes_per_launch"] / per / res["copy_bw_bytes_per_s"])
            r.pop("x")
            if key == "d1" and n == args.parity_n and form == "dense":   # one uninterrupted solve of Kp iterations against the oracle's
                from oracle import oracle_py as O
                rp = mpgp_window(P, torch, A, b_np, n, args.parity_its, 0)
                ia = (np.arange(n + 1, dtype=np.int64) * n).astype(np.int32)
                ja = np.tile(np.arange(n, dtype=np.int32), n)
                op = O.Operator(ia, ja, K.cpu().numpy().ravel())
                xr, ro = O.mpgp_solve(op, b_np, O.BoxC(n, np.zeros(n), None), np.zeros(n), O.mpgp_opts(rtol=1e-300, atol=1e-300, max_it=args.parity_its))
                row["parity"] = dict(max_it=args.parity_its, relx=float(np.linalg.norm(rp["x"] - xr) / np.linalg.norm(xr)), gpu_steps=rp["warmup_steps"],
                                     oracle_steps=dict(ncg=ro["ncg"], nexp=ro["nexp"], nprop=ro["nprop"]))
            row[form] = r
            P.MatDestroy(A)
            torch.cuda.empty_cache()
        if "aij" in row:
            row["dense_over_aij_it_per_s"] = row["dense"]["it_per_s"] / row["aij"]["it_per_s"]
            row["steps_match"] = row["dense"]["steps"] == row["aij"]["steps"]
        del K, b
        torch.cuda.empty_cache()
        res[key][str(n)] = row
        print(json.dumps({key: {n: row}}, default=float), flush=True)
    if args.svm:
        n = args.svm
        K, _ = rbf(torch, n, seed=7)
        g = torch.Generator(device="cuda").manual_seed(8)
        y = (torch.rand(n, generator=g, dtype=torch.float64, device="cuda") < 0.5).to(torch.float64).mul_(2.0).sub_(1.0)
        K.mul_(y[:, None]).mul_(y[None, :])
        row = dict(n=n)
        for form in ("dense", "aij"):
            A, t_ctor = make_mat(P, torch, K, form)
            r = mpgp_window(P, torch, A, np.ones(n), n, 0, 0, ub=np.ones(n), B=y.cpu().numpy())
            r["construct_s"] = t_ctor
            x = r.pop("x")
            r["yTa"] = float(abs(y.cpu().numpy() @ x))
            row[form] = r
            P.MatDestroy(A)
            torch.cuda.empty_cache()
        row["dense_over_aij_inner_it_per_s"] = row["dense"]["inner_it_per_s"] / row["aij"]["inner_it_per_s"]
        res["d2"][str(n)] = row
        print(json.dumps({"svm": row}, default=float), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
