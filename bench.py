#!/usr/bin/env python
"""bench.py -- MPGP iterations/second on the named configurations (BASELINE.json), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload auto|c3|c2|c2x|c2r|c5|c4|...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is ONE MPGP iteration (SpMV + fused update + direction update, src/qps/impls/mpgp/mpgp.c:511-641) of a
QPSSolve that runs through the C ABI of libpermon_b200.so.  W warm-up iterations, then exactly K timed ones:

  value         device-resident leg: matrix + vectors already in HBM, CUDA events on the library's stream, max over ranks
  e2e           a fresh solve of K iterations through the reference-facing calls with HOST (pinned) buffers:
                MatCreate...WithArrays (re-code + H2D), VecCreate...WithArray, QPSSetUp (power method), QPSSolve,
                VecGetArrayRead (D2H of x), all inside the timed region (wall clock, device synchronised on both sides)
  roofline      every fused kernel timed per launch with CUDA events in a repeat of the timed region; the object describes
                the kernel with the largest share of the step, `per_kernel` lists all of them (working launches only)
  cpu_baseline  the CPU oracle (restatement of the reference's un-fused PETSc call sequence, OpenMP threads standing in
                for MPI ranks) on a bounded sample of the same workload, on this box's host cores (rank 0)
  parity        GPU iterate after Kp iterations from x0 against the oracle's iterate after the same Kp iterations of the
                same full-size problem: relx, objective, step mix, active set (rank 0 gathers x at N > 1)

The headline workload is the SAME at every N: C3 (3-D obstacle 512^3, 134 M dofs, z-slab row partition, strong scaling).
The N = 1 line additionally carries C2 (2-D obstacle 4096^2, 16.7 M dofs) as a nested `c2` object with its own
roofline / e2e / parity / cpu_baseline.

--dump-outputs DIR writes the iterate x the timed window ended with (what QPSSolve hands back to its caller) as
DIR/<workload>_x.npy in float64, one file per measured workload: every entry up to DUMP_MAX entries, beyond that the
entries at dump_index(n), a fixed seeded sample of global row numbers.  The inputs are generated from fixed seeds, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank "to avoid overloading the system" and asks the application to tune it: the host side
# of the e2e leg (diagonal / off-diagonal split and re-coding of this rank's rows) is an OpenMP region, so the ranks of one node share
# the host cores evenly.  Must happen before the OpenMP runtime starts (numpy / torch / the library).
if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("OMP_NUM_THREADS", "1") == "1" and not os.environ.get("PERMON_B200_KEEP_OMP"):
    os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // int(os.environ.get("LOCAL_WORLD_SIZE", os.environ["WORLD_SIZE"]))))

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mpgp_iterations_per_second"
UNIT = "it/s"
ASTOL = 10 * 2.2204460492503131e-16      # QPC active-set tolerance (qpc.c:28)
L2_NOTE = "inputs larger than L2 (every kernel streams >= 3 vectors of 8n bytes, n >= 8.4M rows per GPU, vs 126 MB L2)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


WORKLOADS = {
    "c1": dict(kind="2d", N=256, bscale=-30.0, label="C1 2-D obstacle 256^2 (65 536 dofs), 5-point Laplacian, lower bound"),
    "c2": dict(kind="2d", N=4096, bscale=-30.0, label="C2 2-D obstacle 4096^2 (16.7M dofs), 5-point Laplacian, lower bound"),
    "c2x": dict(kind="2d", N=4096, bscale=-100.0, label="C2x expansion-heavy 2-D obstacle 4096^2, b=-100h^2"),
    "c2r": dict(kind="2d", N=4096, bscale=-30.0, scaled=True,
                label="C2r 2-D obstacle 4096^2 with the Hessian scaled D*A*D (every value distinct: incompressible, 12 B per non-zero)"),
    "c3": dict(kind="3d", N=512, label="C3 3-D obstacle 512^3 (134M dofs), 7-point Laplacian, lower bound, z-slab row partition"),
    "c3s": dict(kind="3d", N=256, label="3-D obstacle 256^3 (16.7M dofs) stand-in"),
    "c5": dict(kind="var", N=256, label="C5 variable-coefficient 3-D Laplacian 256^3 (16.7M dofs, contrast 1e4), lb and ub arrays, ~50% active at the solution"),
    "c5s": dict(kind="var", N=128, label="variable-coefficient 3-D Laplacian 128^3 stand-in"),
    "t2d": dict(kind="2d", N=512, bscale=-30.0, label="tiny 2-D obstacle 512^2 (harness self-test)"),
    "t3d": dict(kind="3d", N=64, label="tiny 3-D obstacle 64^3 (harness self-test)"),
}


DUMP_MAX = 1 << 21      # entries per dumped array: 16 MB in float64, so that the C3 + C2 line stays under 64 MB


def dump_index(n):
    """the global rows of an n-vector that --dump-outputs writes: all of them up to DUMP_MAX, else a fixed seeded sample, sorted"""
    if n <= DUMP_MAX:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX, replace=False))


def owned_sample(x_loc, r0, idx):
    """entries of the global sample idx held by this rank's rows [r0, r0 + len(x_loc)), 0 at the others: summed over the ranks it is x[idx],
    exactly (every entry has one owner)"""
    own = (idx >= r0) & (idx < r0 + len(x_loc))
    out = x_loc.new_zeros(len(idx))
    out[own] = x_loc[idx[own] - r0]
    return out


def dump(dump_dir, name, x):
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, f"{name}_x.npy"), np.asarray(x, dtype=np.float64))


def workload_spec(name):
    if name == "auto":
        name = "c3"
    spec = dict(WORKLOADS[name])
    spec["name"] = name
    return spec


def generate(spec, rank, size):
    """this rank's row block, generated in ~2M-row chunks on a thread pool (numpy releases the GIL)"""
    from concurrent.futures import ThreadPoolExecutor
    from permon_b200 import problems as PR
    if spec["kind"] == "2d":
        N = spec["N"]
        starts = PR.row_partition(N * N, size, align=N)
        step = max(N, (2_000_000 // N) * N)
        make = lambda r0, r1: PR.obstacle2d(N, spec["bscale"], rows=(r0, r1), scaled=bool(spec.get("scaled")))
    else:
        N = spec["N"]
        P = N * N
        starts = PR.row_partition(N ** 3, size, align=P)
        step = max(P, (2_000_000 // P) * P)
        if spec["kind"] == "var":
            make = lambda r0, r1: PR.varcoef3d(N, rows=(r0, r1))
        else:
            make = lambda r0, r1: PR.obstacle3d(N, rows=(r0, r1))
    rows = (starts[rank], starts[rank + 1])
    ranges = [(r0, min(r0 + step, rows[1])) for r0 in range(rows[0], rows[1], step)]
    workers = max(1, min(len(ranges), (os.cpu_count() or 1) // max(1, min(size, 8))))
    with ThreadPoolExecutor(workers) as ex:
        chunks = list(ex.map(lambda ab: make(*ab), ranges))
    ia = [np.zeros(1, np.int64)]
    off = 0
    for c in chunks:
        ia.append(c.ia[1:].astype(np.int64) + off)
        off += int(c.ia[-1])
    pr = chunks[0]
    pr.ia = np.concatenate(ia).astype(np.int32)
    pr.ja = np.concatenate([c.ja for c in chunks])
    pr.a = np.concatenate([c.a for c in chunks])
    pr.b = np.concatenate([c.b for c in chunks])
    pr.lb = np.concatenate([c.lb for c in chunks])
    pr.ub = np.concatenate([c.ub for c in chunks]) if chunks[0].ub is not None else None
    pr.x0 = np.zeros(rows[1] - rows[0])
    pr.r0, pr.r1 = rows
    pr.meta = {}
    return pr


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line).  The sampler is
    started before the warm-up so that it is already running when the (possibly very short) timed window opens; samples
    are selected by wall-clock time stamps, falling back to warm-up + timed when the window caught none."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout=8.0):
        """nvidia-smi needs a few hundred ms to start (longer on 8-GPU boxes): block until it delivers"""
        t = time.time()
        while self.proc and not self.rows and time.time() - t < timeout:
            time.sleep(0.01)

    def window_open(self):
        self.t0 = time.time()

    def window_close(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

        def parse(rows):
            sm, mx, reasons, pw = [], [], set(), []
            for _, r in rows:
                f = [t.strip() for t in r.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons, pw

        inwin = [r for r in self.rows if self.t0 is not None and self.t1 is not None and self.t0 <= r[0] <= self.t1 + 0.03]
        window = "timed"
        if not inwin:
            inwin, window = self.rows, "set-up + warm-up + timed (timed window shorter than the sampling period)"
        sm, mx, reasons, pw = parse(inwin)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)), samples=len(sm), window=window, reasons=sorted(reasons))


def algorithmic_bytes(n, nnz, counts, both_bounds=False, matrix_bytes=None):
    """SURVEY.md 8d: B_cg = M + 8 n V ; B_exp = 2 M + 8 n V_e ; proportioning ~ B_cg, with M the matrix stream of one SpMV:
    12 nnz + 4(n+1) for CSR (the survey's formula), or the bytes of the packed tile format the library actually keeps in HBM."""
    V, Ve = (18, 19) if both_bounds else (16, 16)
    if matrix_bytes is not None:
        V -= 1.75          # layout actually streamed: K_B writes a byte mask instead of gf (-7/8 pass), K_C reads g + the mask (+1/8),
                           # K_A does not read g (g.p comes from the kernel that wrote p: -1 pass)
    M = 12 * nnz + 4 * (n + 1) if matrix_bytes is None else matrix_bytes
    b_cg = M + 8 * n * V
    b_exp = 2 * M + 8 * n * Ve
    return (counts["ncg"] + counts["nprop"]) * b_cg + counts["nexp"] * b_exp, b_cg, b_exp


# ----------------------------------------------------------------------------------------------------------
# the oracle on the host cores: reference arm, cpu_baseline and the parity checker
# ----------------------------------------------------------------------------------------------------------
def oracle_window(pr, Kp, maxeig=None):
    """Kp MPGP iterations from x0 on all host cores; returns (x, dict).  The timed region is the iteration loop (the power
    method of the set-up is outside, as on the GPU side's `value`)."""
    from oracle import oracle_py as O
    threads = os.cpu_count() or 1
    op = O.Operator(pr.ia, pr.ja, pr.a)
    bx = O.BoxC(pr.n, pr.lb, pr.ub)
    kw = dict(nthreads=threads, max_it=Kp - 1, rtol=1e-30, atol=1e-300)
    if maxeig:
        kw["maxeig"] = float(maxeig)
    x, r = O.mpgp_solve(op, pr.b, bx, pr.x0, O.mpgp_opts(**kw))
    f = O.objective(op, pr.b, x)
    return x, dict(value=r["its"] / r["seconds"], its=r["its"], seconds=r["seconds"], threads=threads, maxeig=r["maxeig"], objective=f,
                   counts={k: r[k] for k in ("ncg", "nexp", "nprop", "nmv")}, op=op)


def oracle_sample_size(n_global, nnz_global, K, budget_s):
    """iterations the CPU sample may take: ~5.5e-10 s per (non-zero + 8 dofs) and iteration on 16 cores (measured: C2 45 ms, C3 ~0.45 s)"""
    cores = os.cpu_count() or 1
    t_it = 6.0e-10 * (nnz_global + 8.0 * n_global) * 16.0 / max(cores, 1)
    return int(max(5, min(K, budget_s / max(t_it, 1e-9))))


def parity_compare(pr, x_gpu, f_gpu, counts_gpu, x_cpu, res_cpu, Kp):
    """BASELINE.json tolerances at the cut after Kp iterations (SURVEY 8d 'truncated runs')"""
    from oracle import oracle_py as O
    nx = float(np.linalg.norm(x_cpu))
    relx = float(np.linalg.norm(x_gpu - x_cpu) / nx) if nx > 0 else float(np.linalg.norm(x_gpu - x_cpu))
    f_cpu = res_cpu["objective"]
    f_gpu_on_cpu = O.objective(res_cpu["op"], pr.b, np.ascontiguousarray(x_gpu))      # same evaluator on both iterates
    obj_rel = abs(f_gpu_on_cpu - f_cpu) / max(abs(f_cpu), 1e-300)
    mism = 0
    for bound in (pr.lb, pr.ub):
        if bound is None:
            continue
        dg, dc = np.abs(x_gpu - bound), np.abs(x_cpu - bound)
        diff = (dg <= ASTOL) != (dc <= ASTOL)
        mism += int(np.count_nonzero(diff & (np.maximum(dg, dc) > 1e-12)))       # excused: within 1e-12 of the bound on both sides
    cg = {k: int(counts_gpu[k]) for k in ("ncg", "nexp", "nprop", "nmv")}
    cc = {k: int(res_cpu["counts"][k]) for k in cg}
    out = dict(iterations=Kp, relx=relx, objective_rel_diff=obj_rel, objective_cpu=f_cpu, objective_gpu_x_cpu_evaluator=f_gpu_on_cpu,
               active_set_mismatches=mism, step_mix_gpu=cg, step_mix_cpu=cc, step_mix_equal=(cg == cc),
               x_norm2_cpu=nx, x_sum_gpu=float(np.sum(x_gpu)), x_sum_cpu=float(np.sum(x_cpu)),
               tolerances=dict(relx=1e-7, objective_rel_diff=1e-10, active_set_mismatches=0))
    if f_gpu is not None:
        out["objective_gpu"] = f_gpu
        out["objective_gpu_rel_diff"] = abs(f_gpu - f_cpu) / max(abs(f_cpu), 1e-300)
    out["ok"] = bool(relx <= 1e-7 and obj_rel <= 1e-10 and mism == 0 and cg == cc)
    return out


def load_traffic(workload_name):
    """DRAM bytes per launch from the committed `ncu --set full` captures (never measured inside a bench run)"""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = tj.get(workload_name)
        if e:
            return e["dram_bytes_per_launch"], e["source"]
    except Exception:
        pass
    return {}, None


# ----------------------------------------------------------------------------------------------------------
# one workload, all legs
# ----------------------------------------------------------------------------------------------------------
class Env:
    pass


def measure(env, spec, K, W, want_e2e=True, want_cpu=True, want_parity=True, cpu_budget=20.0, sampler=None, dump_dir=None):
    P, torch, dev, stream, rank, size = env.P, env.torch, env.dev, env.stream, env.rank, env.size
    dist = env.dist

    def barrier():
        torch.cuda.synchronize()
        if size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if size == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(vals):
        if size == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.cpu()]

    t_gen = time.time()
    pr = generate(spec, rank, size)
    t_gen = time.time() - t_gen
    n_loc, nnz_loc = pr.n, pr.nnz
    n_glob, nnz_glob = [int(v) for v in sum_over_ranks([n_loc, nnz_loc])]
    vec_keys = ("b", "lb") + (("ub",) if pr.ub is not None else ())
    # pinned host buffers (the e2e leg copies from these)
    host = {k: torch.from_numpy(np.ascontiguousarray(getattr(pr, k))).pin_memory() for k in ("ia", "ja", "a") + vec_keys}
    both = pr.ub is not None

    def make_solver(device_resident):
        """QP + QPS through the C ABI; returns handles"""
        h = {}
        if device_resident:
            # the matrix goes through the host constructor (the library re-codes it into its packed tile format and, when
            # row-partitioned, splits diagonal / off-diagonal blocks) and is resident before the timed region; vectors are
            # device arrays owned by the caller
            h["A"] = P.MatCreateAIJ(pr.ia, pr.ja, pr.a, ncols_local=n_loc)
            d = {k: host[k].to(dev) for k in vec_keys}
            d["x"] = torch.zeros(n_loc, dtype=torch.float64, device=dev)
            for k in vec_keys + ("x",):
                h[k] = P.VecFromDevicePointer(d[k].data_ptr(), n_loc)
            h["dev"] = d
        else:
            h["xh"] = xh_pinned                       # the caller's x buffer (x0 in, solution out): pinned host memory that exists before the timed region
            h["A"] = P.MatCreateAIJ(host["ia"].numpy(), host["ja"].numpy(), host["a"].numpy(), ncols_local=n_loc)
            for k in vec_keys:
                h[k] = P.VecFromArray(host[k].numpy())
            h["x"] = P.VecFromArray(h["xh"].numpy())
        qp = P.QPCreate()
        P.QPSetOperator(qp, h["A"]); P.QPSetRhs(qp, h["b"]); P.QPSetInitialVector(qp, h["x"]); P.QPSetBox(qp, None, h["lb"], h.get("ub"))
        qps = P.QPSCreate()
        P.QPSSetType(qps, "mpgp")
        P.QPSSetQP(qps, qp)
        P.QPSSetAutoPostSolve(qps, False)
        h["qp"], h["qps"] = qp, qps
        return h

    def destroy(h):
        P.QPSDestroy(h["qps"]); P.QPDestroy(h["qp"])
        for k in ("x",) + vec_keys:
            P.VecDestroy(h[k])
        P.MatDestroy(h["A"])

    # ---------------- device-resident leg -----------------------------------------------------------------
    h = make_solver(True)
    P.QPSSetTolerances(h["qps"], rtol=1e-30, atol=1e-300, maxits=W - 1)     # never converge inside the window
    P.QPSSetUp(h["qps"])                                                      # upload done, power method done
    maxeig = P.QPSMPGPGetOperatorMaxEigenvalue(h["qps"])
    storage = P.MatStorageInfo(h["A"])
    if sampler:
        sampler.wait_first()
    P.QPSSolve(h["qps"])                                                      # W warm-up iterations
    assert P.QPSGetIterationNumber(h["qps"]) == W, (P.QPSGetIterationNumber(h["qps"]), W)
    x_after_warmup = h["dev"]["x"].clone()
    c_warm = P.QPSMPGPGetStepCounts(h["qps"])
    P.QPSSetTolerances(h["qps"], maxits=K - 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = P.launch_count()
    barrier()
    if sampler:
        sampler.window_open()
    e0.record(stream)
    P.QPSSolve(h["qps"])                                                      # exactly K timed iterations
    e1.record(stream)
    barrier()
    if sampler:
        sampler.window_close()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = P.launch_count() - launches0
    its = P.QPSGetIterationNumber(h["qps"])
    assert its == K, (its, K)
    c_all = P.QPSMPGPGetStepCounts(h["qps"])
    counts = {k: c_all[k] - c_warm[k] for k in c_all}
    value = K / (ms * 1e-3)
    if dump_dir:
        x_dump = owned_sample(h["dev"]["x"], pr.r0, torch.from_numpy(dump_index(n_glob)).to(dev))
        if size > 1:
            dist.all_reduce(x_dump)
        if rank == 0:
            dump(dump_dir, spec["name"], x_dump.cpu().numpy())
        del x_dump

    # ---------------- roofline: every fused kernel timed per launch in a repeat of the timed region ----------
    h["dev"]["x"].copy_(x_after_warmup)
    barrier()
    P.profile_begin()
    P.QPSSolve(h["qps"])
    prof = P.profile_end()
    if os.environ.get("PERMON_B200_TIMELINE"):
        P.call("PermonB200ProfileDump", (os.environ["PERMON_B200_TIMELINE"] + f".{spec['name']}.rank{rank}.csv").encode())
    barrier()
    peak, peak_src = peaks()
    nb = 1 + (1 if both else 0)                      # bound vectors
    M = storage["stream_bytes"]
    n_cg, n_ex = counts["ncg"] + counts["nprop"], counts["nexp"]
    # algorithmic bytes per launch of each fused kernel in the layout it streams (DESIGN.md section 3), averaged over the
    # window's step mix where the kernel does different work per step kind
    kbytes = {
        "K_A spmv+dots+feas": M + 8 * n_loc * (3 + nb),                                                   # p x bounds -> Ap
        "K_B update+split": 8 * n_loc * ((n_cg * (6.125 + nb) + n_ex * (5 + nb)) / max(n_cg + n_ex, 1)),  # c/p: 4+nb r, x g + byte mask w; e: 4+nb r, 1 w
        "K_A' spmv+grad+split": M + 8 * n_loc * (4 + nb),                                                 # x b bounds -> g p
        "K_C direction": 8 * n_loc * 3.125,                                                                # g, byte mask, p -> p
    }
    # launches that did work, by the step counters: K_A and K_B once per iteration, K_A' per expansion step, K_C (sweep) per CG /
    # proportioning step.  The per-launch timings classify the same way (early exits take a few microseconds): both are reported.
    expect = {"K_A spmv+dots+feas": n_cg + n_ex, "K_B update+split": n_cg + n_ex, "K_A' spmv+grad+split": n_ex, "K_C direction": n_cg}
    per_kernel = {}
    for fam, byts in kbytes.items():
        pf = prof.get(fam)
        if not pf or not pf["launches"] or not expect[fam]:
            continue
        # launches that did work, classified by their duration (an early exit takes microseconds); the step counters give the same
        # number except for K_C, whose last launch of a window that ends by max_it has nothing left to do
        real = pf["working_launches"] if pf["working_launches"] else expect[fam]
        work_ms = pf["working_ms"] if pf["working_launches"] else pf["total_ms"]
        avg = work_ms / real
        gbs = byts / (avg * 1e-3) / 1e9
        per_kernel[fam] = dict(total_ms=round(pf["total_ms"], 3), launches=int(pf["launches"]), working_launches=int(real),
                               working_launches_by_step_counters=int(expect[fam]), working_ms=round(work_ms, 3), avg_ms=round(avg, 5),
                               bytes_per_launch=int(byts), achieved_gbs=round(gbs, 1), frac_of_measured_peak=round(gbs / peak, 4))
    fam_ms = {k: round(v["total_ms"], 3) for k, v in prof.items() if v["launches"]}
    total_prof_ms = sum(v["total_ms"] for v in prof.values())
    dom = max(per_kernel, key=lambda k: per_kernel[k]["working_ms"]) if per_kernel else None
    dk = per_kernel.get(dom, dict(achieved_gbs=0.0, avg_ms=0.0, bytes_per_launch=0, working_launches=0, working_ms=0.0))
    csr_M = 12 * nnz_loc + 4 * (n_loc + 1)
    tr, tr_src = load_traffic(spec["name"]) if size == 1 else ({}, None)
    roofline = dict(bound="hbm", kernel=dom, achieved=dk["achieved_gbs"], peak=peak, unit="GB/s", frac=round(dk["achieved_gbs"] / peak, 4),
                    traffic=tr.get(dom), traffic_source=tr_src if tr.get(dom) else None,
                    peak_source=peak_src, launches=dk["working_launches"], avg_launch_ms=dk["avg_ms"], algorithmic_bytes_per_launch=dk["bytes_per_launch"],
                    kernel_share_of_step=round(dk["working_ms"] / total_prof_ms, 4) if total_prof_ms else None,
                    bytes_note="bytes of the layout the kernels stream (packed matrix tiles + fp64 vectors); with the CSR formula of SURVEY 8d K_A / K_A' "
                               "would count csr_matrix_bytes instead of matrix_bytes",
                    matrix_bytes=int(M), csr_matrix_bytes=int(csr_M), per_kernel=per_kernel, family_ms=fam_ms)
    step_bytes, b_cg, b_exp = algorithmic_bytes(n_loc, nnz_loc, counts, both_bounds=both, matrix_bytes=storage["stream_bytes"])
    step_bytes_csr, b_cg_csr, b_exp_csr = algorithmic_bytes(n_loc, nnz_loc, counts, both_bounds=both)
    whole_iter_gbs = step_bytes / (ms * 1e-3) / 1e9
    whole_iter_gbs_csr = step_bytes_csr / (ms * 1e-3) / 1e9
    destroy(h)
    del h, x_after_warmup
    torch.cuda.empty_cache()

    # ---------------- e2e leg: host buffers, every copy inside the timed region ------------------------------
    e2e, h2 = None, None
    if want_e2e or want_parity:
        host_in = sum(host[k].numel() * host[k].element_size() for k in host) + n_loc * 8      # CSR + b, bounds, x0 handed over in host memory
        d2h = n_loc * 8
        xh_pinned = torch.zeros(n_loc, dtype=torch.float64).pin_memory()      # host input like ia / ja / a / b / lb (page-locking 1 GB takes ~0.4 s)
        barrier()
        t0 = time.perf_counter()
        h2 = make_solver(False)
        P.QPSSetTolerances(h2["qps"], rtol=1e-30, atol=1e-300, maxits=K - 1)
        P.QPSSolve(h2["qps"])                                                 # set-up (upload, power method) + K iterations
        P.VecSyncToHost(h2["x"])                                              # D2H of the iterate into the caller's (pinned) x buffer
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        te = max_over_ranks(t1 - t0)
        assert P.QPSGetIterationNumber(h2["qps"]) == K
        # what crosses PCIe: the matrix as the library stores it (packed tiles) + the vectors; the CSR itself is read on the host only
        h2d = P.MatStorageInfo(h2["A"])["stream_bytes"] + sum(host[k].numel() * host[k].element_size() for k in vec_keys) + n_loc * 8
        e2e = dict(value=K / te, unit=UNIT, h2d_bytes_per_step=h2d / K, d2h_bytes_per_step=d2h / K, seconds=round(te, 4),
                   seconds_outside_iterations=round(te - ms * 1e-3, 4), host_input_bytes=host_in,
                   x_checksum=float(sum_over_ranks([float(np.sum(h2["xh"].numpy()))])[0]),
                   note="host CSR + vectors -> re-code + upload + power-method set-up + K iterations + one download per QPSSolve; bytes are the totals of the solve divided by K")

    # ---------------- parity + CPU baseline (oracle on rank 0, same full-size problem) -----------------------
    cpu, parity = None, None
    if want_parity or want_cpu:
        Kp = oracle_sample_size(n_glob, nnz_glob, K, cpu_budget)
        x_gpu, f_gpu, counts_gpu = None, None, None
        if want_parity:
            # the GPU iterate after Kp iterations from x0: the e2e solve itself when Kp == K, else one more (short) solve on its handles
            if Kp != K:
                P.VecSetArray(h2["x"], np.zeros(n_loc))
                P.QPSSetTolerances(h2["qps"], maxits=Kp - 1)
                c0 = P.QPSMPGPGetStepCounts(h2["qps"])
                P.QPSSolve(h2["qps"])
                P.VecSyncToHost(h2["x"])
                torch.cuda.synchronize()
                c1 = P.QPSMPGPGetStepCounts(h2["qps"])
                counts_gpu = {k: c1[k] - c0[k] for k in c1}
            else:
                counts_gpu = P.QPSMPGPGetStepCounts(h2["qps"])
            f_gpu = P.QPComputeObjective(h2["qp"], h2["x"])
            x_loc = h2["xh"].numpy().copy()
            if size == 1:
                x_gpu = x_loc
            else:
                # rank 0 collects the slabs (NCCL send/recv of device copies)
                sizes = [int(v) for v in env.all_gather_int(n_loc)]
                mine = torch.from_numpy(x_loc).to(dev)
                if rank == 0:
                    parts = [x_loc]
                    for r in range(1, size):
                        buf = torch.empty(sizes[r], dtype=torch.float64, device=dev)
                        dist.recv(buf, src=r)
                        parts.append(buf.cpu().numpy())
                    x_gpu = np.concatenate(parts)
                else:
                    dist.send(mine, dst=0)
                del mine
        if rank == 0:
            t_or = time.time()
            prf = pr if size == 1 else generate(spec, 0, 1)        # the whole problem on rank 0
            x_cpu, res = oracle_window(prf, Kp, maxeig=maxeig)
            cores = res["threads"]
            sample = (f"{res['its']} MPGP iterations from x0 of the full-size workload ({n_glob} dofs), {cores} OpenMP threads standing in for MPI ranks; "
                      "iteration loop timed, power-method set-up outside (as for `value`)")
            if want_cpu and size == 1:
                cpu = dict(value=round(res["value"], 3), unit=UNIT, cores=cores, kind="port", sample=sample, seconds=round(res["seconds"], 2),
                           note="restatement of the reference CPU path (un-fused PETSc call sequence), not PETSc itself; the reference cannot be built here")
            if want_parity:
                parity = parity_compare(prf, x_gpu, f_gpu, counts_gpu, x_cpu, res, Kp)
                parity["oracle_wall_s"] = round(time.time() - t_or, 1)
            del prf, x_cpu, res
        if size > 1:
            dist.barrier()
    if h2 is not None:
        destroy(h2)
    if not want_e2e:
        e2e = None

    out = dict(value=round(value, 2), unit=UNIT, ms_per_step=round(ms / K, 5), steps=K, warmup=W,
               config=dict(workload=spec["label"], n=n_glob, nnz=nnz_glob, l2=L2_NOTE),
               details=dict(n_local=n_loc, nnz_local=nnz_loc, step_mix=counts, matrix_storage=storage, maxeig=maxeig,
                            bytes_per_cg_step=b_cg, bytes_per_expansion_step=b_exp,
                            bytes_per_cg_step_csr_formula=b_cg_csr, bytes_per_expansion_step_csr_formula=b_exp_csr,
                            csr_equivalent_gbs_whole_iteration=round(whole_iter_gbs_csr * size, 1),
                            achieved_gbs_whole_iteration=round(whole_iter_gbs * size, 1),
                            frac_of_measured_hbm_whole_iteration=round(whole_iter_gbs / peak, 4), frac_of_8tbs_whole_iteration=round(whole_iter_gbs / 8000.0, 4),
                            generate_s=round(t_gen, 1)),
               e2e=e2e, gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu, parity=parity)
    del host, pr
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------
# C4: SVM dual through SMALXE + MPGP, Hessian applied as two long-row SpMVs (BASELINE.json configs[3])
# ----------------------------------------------------------------------------------------------------------
def measure_c4(env, n, K, W, want_cpu=True, want_parity=True, dump_dir=None):
    """min 1/2 a'(Z Z')a - 1'a, 0 <= a <= 1, y'a = 0; Z = diag(y) X, X n x n with n/1000 (at most 1000) non-zeros per row.  A step is one
    INNER MPGP iteration of a bounded SMALXE window (1 outer iteration, K inner iterations; at n = d the dual is too ill-conditioned to
    converge inside any bench window, in the oracle as well).  The dominant kernel is the long-row SpMV pair of the Hessian."""
    P, torch, dev, stream = env.P, env.torch, env.dev, env.stream
    from permon_b200 import problems as PR
    t0 = time.time()
    k = max(1, min(1000, n // 100))
    pr = PR.svm_dual_fast(n, n, nnz_per_row=k)
    t_gen = time.time() - t0
    nnz = len(pr.a)
    peak, peak_src = peaks()

    def build(host_side):
        h = {}
        h["A1"] = P.MatCreateAIJ(pr.ia, pr.ja, pr.a, ncols_local=n)
        h["A2"] = P.MatCreateAIJ(pr.second[0], pr.second[1], pr.second[2], ncols_local=n)
        h["A"] = P.MatCreateProd([h["A2"], h["A1"]])
        h["xh"] = np.zeros(n)
        h["b"], h["x"] = P.VecFromArray(np.ones(n)), P.VecFromArray(h["xh"])
        h["lb"], h["ub"] = P.VecFromArray(np.zeros(n)), P.VecFromArray(np.full(n, 1.0))
        h["brow"] = P.VecFromArray(pr.B[0].copy())
        h["BE"] = P.MatCreateOneRow(h["brow"])
        qp = P.QPCreate()
        P.QPSetOperator(qp, h["A"]); P.QPSetRhs(qp, h["b"]); P.QPSetInitialVector(qp, h["x"]); P.QPSetBox(qp, None, h["lb"], h["ub"]); P.QPSetEq(qp, h["BE"], None)
        qps = P.QPSCreate()
        P.QPSSetType(qps, "smalxe"); P.QPSSetQP(qps, qp); P.QPSSetAutoPostSolve(qps, False)
        h["qp"], h["qps"] = qp, qps
        return h

    def destroy(h):
        P.QPSDestroy(h["qps"]); P.QPDestroy(h["qp"])
        for kk in ("b", "x", "lb", "ub", "brow"):
            P.VecDestroy(h[kk])
        for kk in ("BE", "A", "A2", "A1"):
            P.MatDestroy(h[kk])

    def window(h, iters):
        P.options_clear()
        P.call("PetscOptionsInsertString", None, f"-qps_max_it 1 -smalxe_qps_max_it {iters - 1} -qps_rtol 1e-30 -smalxe_qps_rtol 1e-30".encode())
        P.QPSSetFromOptions(h["qps"])

    # ---- Hessian application alone (the two long-row SpMVs)
    h = build(False)
    storage = [P.MatStorageInfo(h["A1"]), P.MatStorageInfo(h["A2"])]
    vx, vy = P.VecFromArray(np.random.default_rng(0).standard_normal(n)), P.VecCreate(n)
    for _ in range(3):
        P.MatMult(h["A"], vx, vy)
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        P.MatMult(h["A"], vx, vy)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_mult = e0.elapsed_time(e1) / reps
    bytes_mult = sum(st["stream_bytes"] for st in storage) + 8 * n * 4       # two matrix streams, x, t (written + read), y
    P.VecDestroy(vx); P.VecDestroy(vy)
    # ---- device-resident window: set-up outside, K inner iterations timed
    window(h, W)
    P.QPSSetUp(h["qps"])
    P.QPSSolve(h["qps"])                                                       # warm-up window
    inner = P.QPSSMALXEGetInnerQPS(h["qps"])
    maxeig_inner = P.QPSMPGPGetOperatorMaxEigenvalue(inner)
    P.VecSetArray(h["x"], np.zeros(n))
    window(h, K)
    st0 = P.QPSSMALXEGetStatistics(h["qps"])["inner_iter_accu"]
    launches0 = P.launch_count()
    torch.cuda.synchronize()
    e0.record(stream)
    P.QPSSolve(h["qps"])
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = P.launch_count() - launches0
    its = P.QPSSMALXEGetStatistics(h["qps"])["inner_iter_accu"]
    counts = P.QPSMPGPGetStepCounts(inner)
    value = its / (ms * 1e-3)
    if dump_dir:
        P.VecSyncToHost(h["x"])
        dump(dump_dir, "c4", h["xh"][dump_index(n)])
    destroy(h)
    torch.cuda.empty_cache()
    # ---- e2e: host arrays -> upload (+ tile-ELL re-layout on the device) -> set-up (two power methods) -> K inner iterations -> download
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h2 = build(True)
    window(h2, K)
    P.QPSSolve(h2["qps"])
    P.VecSyncToHost(h2["x"])
    torch.cuda.synchronize()
    te = time.perf_counter() - t0
    its2 = P.QPSSMALXEGetStatistics(h2["qps"])["inner_iter_accu"]
    host_in = 2 * (12 * nnz + 4 * (n + 1)) + 8 * n * 5
    e2e = dict(value=its2 / te, unit=UNIT, h2d_bytes_per_step=host_in / max(its2, 1), d2h_bytes_per_step=8 * n / max(its2, 1), seconds=round(te, 3),
               note="host CSR of both factors + vectors -> upload, tile-ELL re-layout on the device, SMALXE set-up (two power methods), K inner iterations, download of x")
    # ---- oracle: bounded sample + parity at the cut
    cpu, parity = None, None
    if want_cpu or want_parity:
        from oracle import oracle_py as O
        threads = os.cpu_count() or 1
        Kc = max(3, min(K, int(25.0 / max(1e-9, 6.0e-10 * 2 * nnz * 16.0 / max(threads, 1)))))
        P.VecSetArray(h2["x"], np.zeros(n))
        window(h2, Kc)
        P.QPSSolve(h2["qps"])
        P.VecSyncToHost(h2["x"])
        torch.cuda.synchronize()
        x_gpu = h2["xh"].copy()
        c_gpu = P.QPSMPGPGetStepCounts(P.QPSSMALXEGetInnerQPS(h2["qps"]))
        op = O.Operator(pr.ia, pr.ja, pr.a, second=pr.second)
        bx = O.BoxC(n, pr.lb, pr.ub)
        maxeig = P.MatGetMaxEigenvalue(h2["A"])
        xr, ro = O.smalxe_solve(op, pr.b, bx, pr.B, None, pr.x0,
                                O.smalxe_opts(inner=dict(nthreads=threads, max_it=Kc - 1, rtol=1e-30, maxeig=maxeig_inner), max_it=1, rtol=1e-30, maxeig=maxeig))
        if want_cpu:
            cpu = dict(value=round(ro["inner_its_accu"] / ro["seconds"], 3), unit=UNIT, cores=threads, kind="port", seconds=round(ro["seconds"], 2),
                       sample=f"{ro['inner_its_accu']} inner MPGP iterations of one SMALXE outer iteration on the full-size problem ({n} x {n}, {nnz} non-zeros per factor), "
                              f"{threads} OpenMP threads; eigenvalue estimates handed over from the GPU run (the two power methods alone would take minutes on the CPU)")
        if want_parity:
            nx = float(np.linalg.norm(xr))
            parity = dict(iterations=int(ro["inner_its_accu"]), relx=float(np.linalg.norm(x_gpu - xr) / max(nx, 1e-300)),
                          step_mix_gpu={kk: int(c_gpu[kk]) for kk in ("ncg", "nexp", "nprop", "nmv")},
                          step_mix_cpu={kk: int(ro[kk]) for kk in ("ncg", "nexp", "nprop", "nmv")}, tolerances=dict(relx=1e-7))
            parity["step_mix_equal"] = parity["step_mix_gpu"] == parity["step_mix_cpu"]
            parity["ok"] = bool(parity["relx"] <= 1e-7 and parity["step_mix_equal"])
    destroy(h2)
    gbs = bytes_mult / (ms_mult * 1e-3) / 1e9
    roofline = dict(bound="hbm", kernel="long-row SpMV pair (Hessian Z Z^T)", achieved=round(gbs, 1), peak=peak, unit="GB/s", frac=round(gbs / peak, 4), traffic=None,
                    peak_source=peak_src, launches=reps, avg_launch_ms=round(ms_mult, 4), algorithmic_bytes_per_launch=int(bytes_mult), matrix_storage=storage)
    return dict(value=round(value, 2), unit=UNIT, ms_per_step=round(ms / max(its, 1), 5), steps=int(its), warmup=W,
                config=dict(workload=f"C4 SVM dual {n} x {n}, {k} non-zeros per row ({nnz / 1e6:.0f}M per factor), SMALXE + MPGP, Hessian = two long-row SpMVs", n=n, nnz=2 * nnz,
                            l2="inputs larger than L2 (each factor streams 12 B per non-zero)"),
                details=dict(step_mix=counts, inner_iterations=int(its), maxeig_inner=maxeig_inner, generate_s=round(t_gen, 1)),
                e2e=e2e, gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu, parity=parity)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-c2", action="store_true", help="N = 1, workload auto: skip the nested C2 object")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--c4-n", type=int, default=1_000_000, help="--workload c4: rows = columns of X (BASELINE config 4: 1M)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the iterate of the timed window's last step as DIR/<workload>_x.npy")
    args = ap.parse_args()
    K, W = max(1, args.steps), max(3, args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    spec = workload_spec(args.workload if args.workload != "c4" else "c3")

    if args.impl == "reference":
        # the reference's own CPU implementation needs PETSc + MPI: time the oracle port on all host cores, with the protocol of the GPU arm --
        # W warm-up iterations from x0, then exactly K timed iterations of a new solve from that iterate, the power method's estimate reused
        if rank != 0:
            return
        pr = generate(spec, 0, 1)
        pr.x0, res_w = oracle_window(pr, W)
        x, res = oracle_window(pr, K, maxeig=res_w["maxeig"])
        assert (res_w["its"], res["its"]) == (W, K), (res_w["its"], res["its"], W, K)
        if args.dump_outputs:
            dump(args.dump_outputs, spec["name"], x[dump_index(pr.N)])
        sample = (f"{res['its']} MPGP iterations after {W} warm-up iterations from x0 of the full-size workload ({pr.N} dofs), {res['threads']} OpenMP "
                  "threads standing in for MPI ranks; iteration loop timed, power-method set-up outside")
        line = dict(metric=METRIC, value=res["value"], unit=UNIT, n_gpus=args.gpus, steps=K, warmup=W, ms_per_step=1e3 / res["value"],
                    higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                    config=dict(workload=spec["label"], n=int(pr.N), nnz=int(pr.nnz), l2=L2_NOTE),
                    details=dict(step_mix=res["counts"], objective=res["objective"]),
                    cpu_baseline=dict(value=res["value"], unit=UNIT, cores=res["threads"], kind="port", sample=sample),
                    e2e=dict(value=res["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line), flush=True)
        return

    import torch
    from permon_b200 import api as P

    if P.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    P.call("PermonB200SetDevice", local_rank)
    P.initialize()
    env = Env()
    env.P, env.torch, env.dev, env.rank, env.size, env.dist = P, torch, dev, rank, size, None
    if size > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        env.dist = dist
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(P.get_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        P.comm_init_rank(size, rank, bytes(idt.cpu().numpy().tobytes()))

        def all_gather_int(v):
            t = torch.zeros(size, dtype=torch.int64, device=dev)
            t[rank] = int(v)
            dist.all_reduce(t)
            return t.cpu().tolist()
        env.all_gather_int = all_gather_int
    # CUDA events must be recorded on the stream the kernels are launched on: torch's current stream becomes the library's stream
    # (a null stream handed to PermonB200SetStream would select the library's own non-blocking stream, which events on torch's
    # default stream do not see)
    env.stream = torch.cuda.ExternalStream(P.get_stream(), device=dev)
    torch.cuda.set_stream(env.stream)

    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.workload == "c4":
        assert size == 1, "the C4 product operator is single-GPU"
        res = measure_c4(env, args.c4_n, K, W, want_cpu=not args.no_cpu_baseline, want_parity=not args.no_parity, dump_dir=args.dump_outputs)
        line = dict(metric=METRIC, value=res["value"], unit=UNIT, n_gpus=1, steps=res["steps"], warmup=W, ms_per_step=res["ms_per_step"], higher_is_better=True,
                    scaling="strong", vs_baseline=None, dtype="f64", data="synthetic", config=res["config"], details=res["details"], clocks=sampler.stop(),
                    e2e=res["e2e"], gpu_launches=res["gpu_launches"], roofline=res["roofline"], cpu_baseline=res["cpu_baseline"], parity=res["parity"])
        print(json.dumps(line), flush=True)
        return
    res = measure(env, spec, K, W, want_e2e=not args.no_e2e, want_cpu=not args.no_cpu_baseline, want_parity=not args.no_parity,
                  cpu_budget=args.cpu_budget, sampler=sampler, dump_dir=args.dump_outputs)
    clocks = sampler.stop()

    c2 = None
    if size == 1 and args.workload == "auto" and not args.no_c2:
        # BASELINE.json also quotes the metric on C2 (16.7M dofs, one GPU): same legs, nested
        c2 = measure(env, workload_spec("c2"), K, W, want_e2e=not args.no_e2e, want_cpu=not args.no_cpu_baseline, want_parity=not args.no_parity,
                     cpu_budget=min(args.cpu_budget, 10.0), dump_dir=args.dump_outputs)
        c2["note"] = "C2 = BASELINE.json configs[1] (the 16.7M-dof single-GPU case); the headline workload of this line is C3 so that the --gpus N series is one workload"

    if rank == 0:
        line = dict(metric=METRIC, value=res["value"], unit=UNIT, n_gpus=size, steps=K, warmup=W, ms_per_step=res["ms_per_step"], higher_is_better=True,
                    scaling="strong", vs_baseline=None, dtype="f64", data="synthetic", config=res["config"], details=res["details"],
                    clocks=clocks, e2e=res["e2e"], gpu_launches=res["gpu_launches"], roofline=res["roofline"], cpu_baseline=res["cpu_baseline"],
                    parity=res["parity"])
        if c2 is not None:
            line["c2"] = c2
        if size > 1:
            line["scaling_note"] = ("strong scaling of the fixed C3 problem; efficiency(N) = value(N) / (N * value(1)) with value(1) the headline of the "
                                    "--gpus 1 line (same workload, same W)")
        print(json.dumps(line), flush=True)
    if size > 1:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
