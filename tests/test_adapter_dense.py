"""The dense route of the PETSc adapter (adapters/qpsb200.c): a MATSEQDENSE Hessian is read through MatDenseGetArrayRead + MatDenseGetLDA
and handed to MatCreateSeqDense + MatDenseSetLDA of libpermon_b200.so.  CPU part: against a stub of the library (tests/adapter_stub_lib.c)
that reports what the adapter passed -- m, n, the user's own array and its leading dimension.  GPU part: the reference's ex3 dual problem,
a dense Hessian held with a padded leading dimension, solved through the plug-in reproduces the golden counts of ex3_1.out."""
import os
import re
import subprocess

import numpy as np
import pytest

from permon_b200 import problems as PR

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB = os.path.join(ROOT, "permon_b200", "libpermon_b200.so")


@pytest.fixture(scope="module")
def build(tmp_path_factory):
    d = tmp_path_factory.mktemp("adapter_dense")
    cc = ["/usr/bin/gcc", "-std=c11", "-D_GNU_SOURCE", "-O1", "-Wall", "-Wextra", "-Werror"]
    subprocess.check_call(cc + ["-DPERMON_B200_MOCK_PETSC", "-I" + os.path.join(ROOT, "adapters"), "-c", os.path.join(ROOT, "adapters", "qpsb200.c"), "-o", str(d / "qpsb200.o")])
    subprocess.check_call(cc + ["-c", os.path.join(ROOT, "adapters", "mock", "permon_mock.c"), "-o", str(d / "mock.o")])
    subprocess.check_call(cc + ["-c", os.path.join(HERE, "adapter_dense_driver.c"), "-o", str(d / "driver.o")])
    exe = str(d / "adapter_dense_driver")
    subprocess.check_call(["/usr/bin/gcc", str(d / "driver.o"), str(d / "qpsb200.o"), str(d / "mock.o"), "-ldl", "-o", exe])
    stub = str(d / "libstub.so")
    subprocess.check_call(cc + ["-fPIC", "-shared", os.path.join(HERE, "adapter_stub_lib.c"), "-o", stub])
    return exe, stub, d


def write_problem(path, F, lda, b, x0, lb):
    n = F.shape[0]
    big = np.zeros((lda, n), order="F")
    big[:n, :] = F
    with open(path, "wb") as f:
        np.array([n, lda, lb is not None], dtype=np.int32).tofile(f)
        big.ravel(order="F").tofile(f)
        for arr in (b, x0, lb):
            if arr is not None:
                np.asarray(arr, dtype=np.float64).tofile(f)


def run(build, lib, pr, lda):
    exe, _, d = build
    write_problem(d / "problem.bin", pr.a.reshape(pr.n, pr.n), lda, pr.b, pr.x0, pr.lb)
    env = dict(os.environ, PERMON_B200_LIBRARY=lib)
    return subprocess.run([exe, str(d / "problem.bin"), str(d / "x.bin"), "mpgp"], env=env, capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("pad", [0, 3])
def test_dense_route_hands_over_sizes_array_and_lda(build, pad):
    pr = PR.tutorial_ex3_dual(100)
    lda = pr.n + pad
    p = run(build, build[1], pr, lda)
    assert p.returncode == 0, p.stdout + p.stderr
    user = re.search(r"user MatCreateSeqDense n (\d+) lda (\d+) data (\S+)", p.stdout)
    made = re.findall(r"stub MatCreateSeqDense m (\d+) n (\d+) data (\S+) handle (\S+)", p.stdout)
    setlda = re.findall(r"stub MatDenseSetLDA lda (\d+) handle (\S+)", p.stdout)
    assert user and len(made) == 1, p.stdout
    m, n, data, handle = made[0]
    assert (int(m), int(n)) == (pr.n, pr.n)
    assert data == user.group(3)                      # the user's own array, no copy on the adapter side
    assert "stub MatCreateMPIAIJWithArrays" not in p.stdout
    if pad:
        assert setlda == [(str(lda), handle)]
    else:
        assert setlda == []                           # lda == m is the library's default


@pytest.mark.gpu
def test_ex3_dual_through_the_plugin_as_dense(build, golden):
    from oracle import oracle_py as O
    g = golden["ex3_1"]
    pr = PR.tutorial_ex3_dual(g["n"])
    p = run(build, LIB, pr, pr.n + 3)
    assert p.returncode == 0, p.stderr
    assert f"iterations {g['its']}" in p.stdout and f"reason {g['reason']}" in p.stdout
    for line in (f"number of Hessian multiplications {g['nmv']}", f"number of CG steps {g['ncg']}", f"number of expansion steps {g['nexp']}",
                 f"number of proportioning steps {g['nprop']}"):
        assert line + "\n" in p.stdout, p.stdout
    x = np.fromfile(build[2] / "x.bin")
    xr, ro = O.mpgp_solve(O.Operator(pr.ia, pr.ja, pr.a), pr.b, O.BoxC(pr.n, pr.lb, None), pr.x0, O.mpgp_opts())
    assert np.linalg.norm(x - xr) <= 1e-9 * np.linalg.norm(xr)
