"""The UNMODIFIED reference driver cuda/acg-cuda.c linked against libacgb200_mpi.so.

CPU part (build container, where /root/reference exists): the driver and the
reference's host layer compile from where they lie and link against the library
with no undefined symbol (tools/build_driver.sh) -- the "drop-in" claim of
INTEGRATION.md, option A.  GPU part: the prebuilt binary (oracle/_ref/driver/,
shipped by gpurun) reads a Matrix Market file, solves on the B200 through
acgsolvercuda_init/_solvempi/_solve_pipelined/_fwritempi and prints x; iteration
count, norms and solution are compared with the oracle.
"""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from acg_b200 import matgen as mg
from acg_b200 import mtxio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "oracle", "_ref", "driver", "acg-cuda")


@pytest.mark.skipif(not os.path.isdir("/root/reference/cuda"), reason="reference tree not present (GPU box)")
def test_unmodified_driver_links_against_library():
    p = subprocess.run(["bash", os.path.join(ROOT, "tools", "build_driver.sh")], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert "undefined reference" not in p.stderr
    v = subprocess.run([DRIVER, "--version"], capture_output=True, text=True)
    assert v.returncode == 0 and "acg-cuda" in v.stdout
    # the solver symbols resolve to the library, not to reference objects
    nm = subprocess.run(["nm", "-D", "--undefined-only", DRIVER], capture_output=True, text=True).stdout
    for sym in ("acgsolvercuda_init", "acgsolvercuda_solvempi", "acgsolvercuda_solve_pipelined",
                "acgsolvercuda_fwritempi", "acgsolvercuda_free", "acgcomm_init_nccl", "acgcomm_init_mpi"):
        assert re.search(rf"\bU {sym}\b", nm), sym


@pytest.mark.gpu
@pytest.mark.parametrize("solver,method", [("acg", "cg"), ("acg-pipelined", "cg_pipelined"),
                                           ("acg-device", "cg"), ("acg-device-pipelined", "cg_pipelined")])
def test_driver_solves_on_gpu(solver, method, oracle):
    if not os.path.exists(DRIVER):
        pytest.skip("driver binary not built (needs the reference tree at build time)")
    n, r, c, v = mg.stencil3d_27pt(20)
    csr = oracle.full_csr(n, r, c, v)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "A.mtx")
        mtxio.write_symmetric(path, n, r, c, v, binary=True)
        p = subprocess.run([DRIVER, path, "--binary", "--solver", solver, "--max-iterations", "200",
                            "--residual-rtol", "1e-9", "--warmup", "2", "--numfmt", "%.17g"],
                           capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    rep = p.stderr
    its = int(re.search(r"^\s*iterations: ([\d,]+)", rep, re.M).group(1).replace(",", ""))
    rnrm2 = float(re.search(r"^\s*residual 2-norm: (\S+)", rep, re.M).group(1))
    r0 = float(re.search(r"^\s*initial residual 2-norm: (\S+)", rep, re.M).group(1))
    # the driver's default right-hand side is all ones (cuda/acg-cuda.c:1949-1967)
    want = getattr(oracle, method)(csr, np.ones(n), maxits=200, rtol=1e-9)
    assert its == want["niterations"]
    assert r0 == pytest.approx(want["r0nrm2"], rel=1e-13)
    assert rnrm2 / r0 == pytest.approx(want["rnrm2"] / want["r0nrm2"], rel=1e-6, abs=1e-10)
    lines = [l for l in p.stdout.splitlines() if l and not l.startswith("%")]
    x = np.array([float(t) for t in lines[1:]])
    assert int(lines[0].split()[0]) == n and len(x) == n
    assert np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()


MPIRUN = os.path.join(ROOT, "compat", "mpi", "acgb200-mpirun")


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.parametrize("solver,method", [("acg", "cg"), ("acg-pipelined", "cg_pipelined")])
def test_driver_solves_on_several_gpus(solver, method, oracle):
    """The unmodified driver as one process per GPU under compat/mpi/acgb200-mpirun (MPI stand-in over Unix
    sockets for the bootstrap, METIS partition by the reference's own code, NCCL + peer memory for the solve):
    `acg-cuda A.mtx --comm nccl` exactly as the reference's README starts it under mpirun."""
    n = min(_ngpu(), 8)
    if n < 2:
        pytest.skip("needs at least 2 GPUs on the box (gpurun --gpus 2)")
    if not os.path.exists(DRIVER) or not os.path.exists(MPIRUN):
        pytest.skip("driver binary / launcher not built")
    N, r, c, v = mg.stencil3d_27pt(24)
    csr = oracle.full_csr(N, r, c, v)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "A.mtx")
        mtxio.write_symmetric(path, N, r, c, v, binary=True)
        p = subprocess.run([MPIRUN, "-n", str(n), DRIVER, path, "--binary", "--comm", "nccl", "--solver", solver,
                            "--max-iterations", "200", "--residual-rtol", "1e-9", "--warmup", "2", "--numfmt", "%.17g"],
                           capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    its = int(re.search(r"^\s*iterations: ([\d,]+)", p.stderr, re.M).group(1).replace(",", ""))
    r0 = float(re.search(r"^\s*initial residual 2-norm: (\S+)", p.stderr, re.M).group(1))
    want = getattr(oracle, method)(csr, np.ones(N), maxits=200, rtol=1e-9)
    assert its == want["niterations"] and r0 == pytest.approx(want["r0nrm2"], rel=1e-12)
    # (NCCL may print its version banner on stdout: NCCL_DEBUG=VERSION on the GPU boxes)
    lines = [ln for ln in p.stdout.splitlines() if ln and not ln.startswith("%") and not ln.startswith("NCCL")]
    x = np.array([float(t) for t in lines[1:]])
    assert int(lines[0].split()[0]) == N and np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()


STOCK = os.path.join(ROOT, "tests", "golden", "reference", "stock_gpu_27pt20.npz")


@pytest.mark.parametrize("solver,method", [("acg", "cg"), ("acg-pipelined", "cg_pipelined")])
def test_stock_reference_gpu_solver_pins_the_oracle(solver, method, oracle):
    """The reference's OWN GPU solver (acg/cgcuda.c with cuSPARSE/cuBLAS, built unmodified
    for sm_100a by tools/build_driver.sh) on the same matrix, as stored from a run on a B200
    (tools/make_reference_golden.py --stock-gpu): the oracle restatement -- in particular of
    pipelined CG, which the reference has no CPU version of -- must give the same residual
    norms and solution after a fixed number of iterations.  Nothing of libacgb200 is involved."""
    g = np.load(STOCK)
    n, r, c, v = mg.stencil3d_27pt(20)
    csr = oracle.full_csr(n, r, c, v)
    its = 30
    got_its, rnrm2, r0 = int(g[solver + "__niterations"]), float(g[solver + "__rnrm2"]), float(g[solver + "__r0nrm2"])
    x = g[solver + "__x"]
    want = getattr(oracle, method)(csr, np.ones(n), maxits=its, rtol=0.0)
    assert got_its == want["niterations"] == its
    assert r0 == pytest.approx(want["r0nrm2"], rel=1e-13)
    assert rnrm2 / r0 == pytest.approx(want["rnrm2"] / want["r0nrm2"], rel=1e-8)
    assert len(x) == n
    assert np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["acg", "acg-pipelined"])
def test_driver_manufactured_solution(solver):
    """KAT-4 (cuda/acg-cuda.c:1969-1979, :2090-2130, :2376-2385): the driver draws a random
    unit vector x*, sets b = A x* with the reference's host SpMV, solves on the GPU through
    the library and prints ||x*|| and ||x - x*||.  With a residual tolerance of 1e-10 on a
    well-conditioned matrix the error must fall by many orders of magnitude."""
    if not os.path.exists(DRIVER):
        pytest.skip("driver binary not built (needs the reference tree at build time)")
    n, r, c, v = mg.stencil3d_27pt(24)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "A.mtx")
        mtxio.write_symmetric(path, n, r, c, v, binary=True)
        p = subprocess.run([DRIVER, path, "--binary", "--solver", solver, "--max-iterations", "500",
                            "--residual-rtol", "1e-10", "--manufactured-solution", "--seed", "7", "-q"],
                           capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    e0 = float(re.search(r"^initial error 2-norm: (\S+)", p.stderr, re.M).group(1))
    e1 = float(re.search(r"^error 2-norm: (\S+)", p.stderr, re.M).group(1))
    assert e0 == pytest.approx(1.0, rel=1e-12)            # x* is normalised
    assert e1 < 1e-7 * e0
