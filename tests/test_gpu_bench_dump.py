"""bench.py --dump-outputs on the GPU path: with the same arguments the GPU arm and the reference arm (the CPU oracle, same protocol: W warm-up
iterations from x0, then K more of a new solve from there) write the same iterate.  C2 is larger than DUMP_MAX, so the file is the seeded sample
of rows gathered from the device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from bench import DUMP_MAX

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", "7", "--warmup", "4", *args],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def test_gpu_and_reference_arms_dump_the_same_iterate(tmp_path):
    ours = bench("--no-e2e", "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "ours"))
    ref = bench("--impl", "reference", "--dump-outputs", str(tmp_path / "ref"))
    assert (ours["steps"], ours["warmup"]) == (ref["steps"], ref["warmup"]) == (7, 4)
    assert ours["details"]["step_mix"] == ref["details"]["step_mix"]
    x, xr = np.load(tmp_path / "ours" / "c2_x.npy"), np.load(tmp_path / "ref" / "c2_x.npy")
    assert x.dtype == xr.dtype == np.float64 and x.shape == xr.shape == (DUMP_MAX,)
    assert np.linalg.norm(xr) > 0 and np.linalg.norm(x - xr) <= 1e-7 * np.linalg.norm(xr)
