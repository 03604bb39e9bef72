"""Device-resident AIJ input: MatB200CreateAIJWithDeviceArrays (CSR in HBM, re-coded on the GPU) against MatCreateSeqAIJWithArrays
(CSR in pinned host memory, re-coded on the host and uploaded), on one GPU.

    python profiles/device_recode_bench.py [--workloads c2,c2r,c5,c3] [--its 200] [--out FILE]

For each workload (the bench.py generators): the wall time of each constructor, device-synchronised on both sides; the storage info of
both matrices (they must agree); MPGP iterations per second over --its iterations of each matrix, after a warm-up solve (the stored
forms are identical, so the two rates only differ by noise).  The card's name and power limit are read in the same run."""
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


def mpgp_rate(P, A, pr, its):
    def run(maxit):
        P.options_clear()
        P.call("PetscOptionsInsertString", None, b"-qps_rtol 1e-300")
        x = P.VecFromArray(np.zeros(pr.r1 - pr.r0))
        b = P.VecFromArray(np.ascontiguousarray(pr.b))
        lb = P.VecFromArray(np.ascontiguousarray(pr.lb)) if pr.lb is not None else None
        ub = P.VecFromArray(np.ascontiguousarray(pr.ub)) if pr.ub is not None else None
        qp = P.QPCreate()
        P.QPSetOperator(qp, A), P.QPSetRhs(qp, b), P.QPSetInitialVector(qp, x), P.QPSetBox(qp, None, lb, ub)
        qps = P.QPSCreate()
        P.QPSSetType(qps, "mpgp")
        P.QPSSetQP(qps, qp)
        P.QPSSetFromOptions(qps)
        P.QPSSetTolerances(qps, maxits=maxit)
        P.QPSSetUp(qps)
        P.synchronize()
        t0 = time.perf_counter()
        P.QPSSolve(qps)
        P.synchronize()
        dt = time.perf_counter() - t0
        n = P.QPSGetIterationNumber(qps)
        P.QPSDestroy(qps), P.QPDestroy(qp)
        for v in (x, b, lb, ub):
            if v is not None:
                P.VecDestroy(v)
        return n, dt
    run(20)
    n, dt = run(its)
    return dict(iterations=n, seconds=dt, it_per_s=n / dt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c2r,c5,c3")
    ap.add_argument("--its", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from permon_b200 import api as P
    if P.device_count() == 0:
        raise SystemExit("needs a CUDA device")
    P.initialize()
    res = dict(card=card(), its=args.its, workloads={})
    print(json.dumps(res["card"]), flush=True)
    for w in args.workloads.split(","):
        spec = bench.workload_spec(w)
        pr = bench.generate(spec, 0, 1)
        n, nnz = pr.r1 - pr.r0, int(pr.ia[-1])
        ia = torch.from_numpy(np.ascontiguousarray(pr.ia, np.int32)).pin_memory()
        ja = torch.from_numpy(np.ascontiguousarray(pr.ja, np.int32)).pin_memory()
        a = torch.from_numpy(np.ascontiguousarray(pr.a, np.float64)).pin_memory()
        pr.ia = pr.ja = pr.a = None
        dia, dja, da = ia.cuda(), ja.cuda(), a.cuda()
        torch.cuda.synchronize()
        P.synchronize()
        t0 = time.perf_counter()
        Ad = P.MatCreateAIJFromDeviceTensors(dia, dja, da)
        P.synchronize()
        t_dev = time.perf_counter() - t0
        del dia, dja, da
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        P.synchronize()
        t0 = time.perf_counter()
        Ah = P.MatCreateAIJ(ia.numpy(), ja.numpy(), a.numpy())
        P.synchronize()
        t_host = time.perf_counter() - t0
        del ia, ja, a
        si_d, si_h = P.MatStorageInfo(Ad), P.MatStorageInfo(Ah)
        rd = mpgp_rate(P, Ad, pr, args.its)
        rh = mpgp_rate(P, Ah, pr, args.its)
        r = dict(label=spec["label"], n=n, nnz=nnz, csr_bytes=12 * nnz + 4 * (n + 1),
                 device_ctor_ms=1e3 * t_dev, host_ctor_ms=1e3 * t_host, storage_device=si_d, storage_host=si_h, storage_equal=si_d == si_h,
                 mpgp_device_built=rd, mpgp_host_built=rh)
        res["workloads"][w] = r
        print(json.dumps({w: r}), flush=True)
        P.MatDestroy(Ad)
        P.MatDestroy(Ah)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
