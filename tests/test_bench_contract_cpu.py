"""bench.py's reference arm runs without a GPU (it times the oracle on the host cores): check the JSON contract of that line on the
small C1 workload and the iterate it writes with --dump-outputs, and that the default arm refuses to run without a CUDA device instead of
falling back to the CPU."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_json_line():
    p = run("--impl", "reference", "--workload", "c1", "--steps", "40", "--warmup", "5")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "impl",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "mpgp_iterations_per_second" and line["unit"] == "it/s"
    assert line["vs_baseline"] is None and line["dtype"] == "f64" and line["data"] == "synthetic" and line["gpu_launches"] == 0
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "workload" in line["config"]
    assert line["config"]["workload"].startswith("C1 ")


def steps_of(line):
    mix = line["details"]["step_mix"]
    return mix["ncg"] + mix["nexp"] + mix["nprop"]


def test_reference_arm_dumps_its_iterate(tmp_path):
    """the dump is the iterate after W warm-up iterations from x0 and K more from there, the same protocol as the GPU arm's"""
    from oracle import oracle_py as O
    from permon_b200 import problems as PR
    K, W = 40, 5
    p = run("--impl", "reference", "--workload", "c1", "--steps", str(K), "--warmup", str(W), "--dump-outputs", str(tmp_path / "out"))
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert (line["steps"], line["warmup"], steps_of(line)) == (K, W, K)
    assert os.listdir(tmp_path / "out") == ["c1_x.npy"]
    x = np.load(tmp_path / "out" / "c1_x.npy")
    pr = PR.obstacle2d(256, -30.0)
    assert x.dtype == np.float64 and x.shape == (pr.n,)
    op, box = O.Operator(pr.ia, pr.ja, pr.a), O.BoxC(pr.n, pr.lb, pr.ub)
    opts = lambda k, maxeig=O.DECIDE: O.mpgp_opts(max_it=k - 1, rtol=1e-30, atol=1e-300, nthreads=os.cpu_count() or 1, maxeig=maxeig)
    x1, r1 = O.mpgp_solve(op, pr.b, box, np.zeros(pr.n), opts(W))
    xr, r2 = O.mpgp_solve(op, pr.b, box, x1, opts(K, r1["maxeig"]))
    assert (r1["its"], r2["its"]) == (W, K)
    assert np.linalg.norm(x - xr) <= 1e-10 * np.linalg.norm(xr)


def test_reference_arm_runs_every_step_it_is_given(tmp_path):
    """C2 with one step more than ~60 s of host time were estimated to allow (the bound the CPU sample of the GPU arm keeps): --steps is still
    the number of timed iterations, and the dump (a sample: C2 is larger than DUMP_MAX) is the iterate after them"""
    from bench import DUMP_MAX, oracle_sample_size
    n = 4096 * 4096
    K = oracle_sample_size(n, 5 * n - 4 * 4096, 10 ** 9, 60.0) + 1
    p = run("--impl", "reference", "--workload", "c2", "--steps", str(K), "--warmup", "3", "--dump-outputs", str(tmp_path), timeout=1800)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert (line["config"]["n"], line["config"]["nnz"]) == (n, 5 * n - 4 * 4096)
    assert (line["steps"], steps_of(line)) == (K, K) and line["cpu_baseline"]["sample"].startswith(f"{K} MPGP iterations after 3 warm-up")
    assert np.load(tmp_path / "c2_x.npy").shape == (DUMP_MAX,)


def test_owned_sample_gathers_rows_across_ranks():
    """the multi-GPU dump: every rank contributes the sampled rows of its slab, the sum over the ranks is the sample of the whole vector"""
    import torch
    from bench import owned_sample
    x = torch.from_numpy(np.random.default_rng(3).standard_normal(1000))
    idx = torch.from_numpy(np.sort(np.random.default_rng(4).choice(1000, 97, replace=False)))
    for starts in ([0, 1000], [0, 400, 1000], [0, 1, 333, 700, 999, 1000]):
        parts = [owned_sample(x[a:b], a, idx) for a, b in zip(starts[:-1], starts[1:])]
        assert all(int(torch.count_nonzero(q)) == int(((idx >= a) & (idx < b)).sum()) for q, a, b in zip(parts, starts[:-1], starts[1:]))
        assert torch.equal(sum(parts), x[idx])


def test_dump_sample_is_fixed_and_bounded():
    from bench import DUMP_MAX, dump_index
    assert np.array_equal(dump_index(1000), np.arange(1000))
    i = dump_index(512 ** 3)
    assert np.array_equal(i, dump_index(512 ** 3))
    assert len(i) == DUMP_MAX and np.all(np.diff(i) > 0) and i[0] >= 0 and i[-1] < 512 ** 3
    assert 2 * DUMP_MAX * 8 <= 64e6          # the C3 + C2 line in float64


def test_default_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return   # on a GPU box this arm is exercised by the driver itself
    p = run("--workload", "c1", "--steps", "5", "--warmup", "3")
    assert p.returncode != 0
    assert "no CUDA device" in (p.stderr + p.stdout) or "no CPU" in (p.stderr + p.stdout)
