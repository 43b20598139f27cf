"""Host logic of the solver (acg_b200/csrc/cgcuda.c: set-up, warm-up, iteration
control, CUDA-graph capture and replay, polling, convergence, return codes,
reports) driven end to end on a device stand-in -- tests/hostsim/: the library's
own C sources built against a mock of the CUDA runtime and plain-C stand-ins of
the kernels' launch interface -- and compared with the oracle.  This checks the
code around the kernels, not the kernels (those are checked on the B200 by
test_gpu_parity.py).  The stand-in lives under tests/, is never loaded by the
product package, and runs in a subprocess."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM = os.path.join(ROOT, "tests", "hostsim")


@pytest.fixture(scope="module")
def simlib():
    p = subprocess.run(["make", "-C", SIM], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert "warning" not in p.stderr
    return os.path.join(SIM, "libacgb200_hostsim.so")


def _run(spec):
    p = subprocess.run([sys.executable, os.path.join(SIM, "run_sim.py"), json.dumps(spec)], capture_output=True, text=True,
                       timeout=600, env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


def _check(out, xtol=1e-10):
    assert out["spmv_err"] < 1e-13 and out["report_ok"]
    for i, r in enumerate(out["runs"]):
        assert r["code"] == r["ref_code"], r
        assert r["its"] == r["ref_its"], r
        assert r["nsolves"] == i + 1
        assert r["r0nrm2"] == pytest.approx(r["ref_r0nrm2"], rel=1e-13)
        assert r["rnrm2"] == pytest.approx(r["ref_rnrm2"], rel=1e-6, abs=1e-12 * r["ref_r0nrm2"]), r
        assert r["xerr"] < xtol, r


RUNS = [{"method": "solvempi", "maxits": 200, "rtol": 1e-9, "warmup": 2},
        {"method": "solve_pipelined", "maxits": 200, "rtol": 1e-9, "warmup": 1},
        {"method": "solvempi", "maxits": 0}, {"method": "solvempi", "maxits": 1}, {"method": "solvempi", "maxits": 7},
        {"method": "solve_pipelined", "maxits": 1}, {"method": "solve_pipelined", "maxits": 2},
        {"method": "solve_pipelined", "maxits": 5}, {"method": "solve_pipelined", "maxits": 12},
        {"method": "solvempi", "maxits": 3, "rtol": 1e-30}, {"method": "solve_pipelined", "maxits": 2, "rtol": 1e-30},
        {"method": "solve_device", "maxits": 9}, {"method": "solve_device_pipelined", "maxits": 8}]


@pytest.mark.parametrize("slices", [1, 0], ids=["slices", "tiles-only"])
def test_pattern_slices_and_device_expansion(slices, simlib):
    """The stencil's rows go to pattern slices (slices.c) and the rest to tiles -- the stand-in fails a row
    the two plans forget or cover twice; and a matrix without full storage is expanded on the device by
    acgsolvercuda_init (expand_host.c; here the stand-in's serial fill) with the same results."""
    out = _run({"matrix": "27pt", "options": {"spmv_slices": slices}, "no_full_storage": 1, "runs": RUNS[:4] + RUNS[7:9]})
    _check(out)
    assert (out["slices"] > 0) == bool(slices) and out["slice_rows"] == 32 * out["slices"]
    if slices:
        assert out["slice_rows"] >= 600 and out["ntiles"] >= 1        # 720 rows: most of the 22 full slices; the ragged end and padding-heavy slices in tiles


@pytest.mark.parametrize("matrix", ["27pt", "7pt"])
@pytest.mark.parametrize("graph", [1, 0], ids=["graph-replay", "direct"])
def test_default_loops(matrix, graph, simlib):
    """Classic and pipelined loops as shipped: tolerances on and off, odd and even iteration
    counts (below and above the graph threshold), not-converged return code, warm-up, several
    solves on one solver, with and without graph replay."""
    out = _run({"matrix": matrix, "options": {"graph": graph}, "runs": RUNS})
    _check(out)
    launches = {(r["method"], r["maxits"]): r["launches"] for r in out["runs"]}
    # per SpMV: the slice kernel plus the tile kernel for the rows outside slices (both matrices have a ragged end);
    # 2 more kernels per classic iteration, 1 more per pipelined one; set-up products: r0 (classic), r0 and w0 (pipelined)
    assert out["slices"] > 0 and out["ntiles"] > 0
    assert launches[("solvempi", 7)] == 4 * 7 + 2 and launches[("solve_pipelined", 12)] == 3 * 12 + 4


@pytest.mark.parametrize("options", [{"spmv_merge": 0}, {"spmv_merge": 0, "spmv_medium": 64}, {}, {"merge_items": 256},
                                     {"merge_items": 4096, "merge_threads": 256}],
                         ids=["row-tiles", "row-tiles+medium-rows", "merge-tiles", "merge-tiles-256", "merge-tiles-4096"])
def test_power_law_rows(options, simlib):
    """Power-law row lengths.  Row-aligned tiles: long rows (and, on request, medium rows) leave the tiles.
    Merge-path tiles (the default for such a matrix, mergeplan.c): rows of any length in equal tiles of
    merged items, rows cut by tile boundaries finished from partial sums.  Either way every row is computed
    exactly once (the stand-in checks that) and the solves reproduce the oracle."""
    spec = {"matrix": "rmat", "options": options,
            "runs": [{"method": "solvempi", "maxits": 10}, {"method": "solve_pipelined", "maxits": 11},
                     {"method": "solve_pipelined", "maxits": 6, "warmup": 2}]}
    out = _run(spec)
    _check(out, xtol=1e-8)
    if options.get("spmv_merge", -1) == 0:
        assert out["nlong"] > 0 and out["merge_tiles"] == 0
        assert (out["nmedium"] > 0) == ("spmv_medium" in options)
    else:
        assert out["merge_tiles"] > 0 and out["merge_rows"] == 30000 and out["merge_split"] > 0
        assert out["nlong"] == 0 and out["ntiles"] == 0
    two_kernel = [r["launches"] for r in out["runs"] if r["method"] == "solve_pipelined"]
    assert two_kernel[0] > 2 * 11                             # SpMV (+ row-list kernels) + update per iteration


def test_tiny_system(simlib):
    out = _run({"matrix": "n3", "options": {},
                "runs": [{"method": "solve_pipelined", "maxits": 2}, {"method": "solvempi", "maxits": 10, "rtol": 1e-12}]})
    _check(out)


def test_profile_mode_and_poll_interval(simlib):
    """profile=1 (what bench.py uses for the SpMV roofline): every SpMV of the solve window is
    bracketed by events -- count = iterations + set-up products -- and graphs are not used;
    the convergence poll interval does not change iteration counts or results."""
    runs = [{"method": "solvempi", "maxits": 100, "rtol": 1e-9}, {"method": "solve_pipelined", "maxits": 100, "rtol": 1e-9},
            {"method": "solve_pipelined", "maxits": 9}]
    out = _run({"matrix": "7pt", "options": {"profile": 1}, "runs": runs})
    _check(out)
    for r in out["runs"]:
        setup = 1 if r["method"] == "solvempi" else 2
        if r["its"] == r["maxits"]:
            assert r["spmv_count"] == r["its"] + setup       # tolerances off (bench.py's case): exact
        else:
            # the host enqueues ahead of the device-side stopping test: up to two poll intervals of
            # launches that return at once are bracketed too
            assert r["its"] + setup <= r["spmv_count"] <= r["its"] + setup + 16
    base = [(r["its"], r["rnrm2"]) for r in out["runs"]]
    for every in (1, 3, 64):
        o = _run({"matrix": "7pt", "options": {"check_every": every}, "runs": runs})
        _check(o)
        assert [(r["its"], r["rnrm2"]) for r in o["runs"]] == base


def test_rejected_calls_leave_the_counters_alone(simlib):
    out = _run({"matrix": "7pt", "runs": [{"method": "solvempi", "maxits": 4}]})
    assert out["errors"]["diffatol"] == 26                 # ACG_ERR_NOT_SUPPORTED (acg/cgcuda.c:424)
    assert out["errors"]["short_b"] == 31                  # ACG_ERR_INDEX_OUT_OF_BOUNDS (acg/cgcuda.c:417-421)
    assert out["nsolves_after_errors"] == 1


def _free_port():
    import socket
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


@pytest.mark.parametrize("nproc,matrix,size,partition,backends,extra", [
    (2, "27pt", 8, "block", "p2p-fused,p2p-unfused,nccl,nccl-graph,nccl-serial-reduce,tiles-only", []),
    (3, "7pt", 9, "slab", "watchdog,p2p-fused,tiles-only,nccl", []),
    (4, "rmat", 3000, "random", "p2p-fused,nccl", ["--maxits", "12", "--rtol", "0"]),
    # 2x2x2 blocks: the interior rows next to a block's border shell are exception rows of their slices (slices.c)
    (8, "27pt", 24, "block", "p2p-fused,tiles-only", []),
], ids=["2-ranks-all-backends", "3-ranks", "4-ranks-power-law", "8-ranks-blocks"])
def test_multi_rank_loops(nproc, matrix, size, partition, backends, extra, simlib):
    """The distributed solver, one process per rank: the library's host code on the stand-in,
    "device" allocations in shared memory so that the CUDA-IPC windows of the peer-memory exchange
    are really shared between the processes, NCCL replaced by a file-based stand-in, and the
    simulated kernels speaking the exchange protocol of kernels.cu (sequence-numbered flags,
    parity-buffered ghost values and reduction slots).  Every loop back-end -- peer memory with
    and without the pushes fused into the kernels, with and without pattern slices for the interior rows, NCCL
    with and without graph replay and with the reduction on the main stream -- must reproduce the
    single-rank oracle.  What this cannot see: anything inside the CUDA kernels, and stream-level
    concurrency on a real device."""
    worker = os.path.join(ROOT, "tests", "_dist_worker.py")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), worker, "--mode", "gpu",
           "--matrix", matrix, "--size", str(size), "--partition", partition, "--backends", backends] + extra
    # "watchdog": one rank stops publishing mid-solve; the others must give up after the timeout,
    # report ACG_ERR_CUDA / cudaErrorLaunchTimeout, and the next solver on the same ranks must work
    import glob
    before = set(glob.glob("/dev/shm/acgb200sim_*"))          # leftovers of killed processes are not this run's
    env = dict(os.environ, OMP_NUM_THREADS="2", ACGB200_TEST_HOSTSIM=simlib,
               ACGB200_P2P_TIMEOUT_MS="1500" if "watchdog" in backends else "20000")
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    sys.stdout.write(p.stdout[-3000:])
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "FAIL" not in p.stdout
    names = backends.split(",")
    assert p.stdout.count(" OK") == 4 * len([b for b in names if b != "watchdog"]) + (nproc if "watchdog" in names else 0)
    assert not set(glob.glob("/dev/shm/acgb200sim_*")) - before      # every "device" allocation was released
    for f in glob.glob("/dev/shm/acgb200nccl_*"):            # NCCL stand-in leftovers of killed runs, if any
        os.remove(f)


CONTRACT_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks")


@pytest.mark.parametrize("nproc", [1, 2])
def test_bench_main_runs_and_prints_the_contract_line(nproc, simlib, tmp_path):
    """bench.py's main(), unchanged, on the stand-in (tests/hostsim/run_bench_sim.py patches
    torch.cuda availability and the nvidia-smi sampler around it): matrix set-up for one and
    several ranks, timed pass, profiled pass, one JSON line from rank 0 with every key of the
    bench contract; on one rank, the outputs of the last timed step under --dump-outputs.
    Shape only -- nothing it prints is a measurement."""
    script = os.path.join(SIM, "run_bench_sim.py")
    args = ["--gpus", str(nproc), "--workload", "27pt-64", "--steps", "2", "--warmup", "1", "--iters", "6", "--cpu-iters", "2"]
    dump = str(tmp_path / "out")
    if nproc == 1:
        cmd = [sys.executable, script] + args + ["--dump-outputs", dump]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
               "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), script] + args
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="2"), cwd=ROOT)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1                                   # rank 0 only, one line
    d = json.loads(lines[0])
    for k in CONTRACT_KEYS:
        assert k in d, k
    assert d["n_gpus"] == nproc and d["steps"] == 2 and d["warmup"] == 1 and d["unit"] == "iterations/s"
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    if nproc == 1:
        assert d["gpu_launches"] == 2 * (2 * 6 + 2)          # 2 steps x (2 kernels x 6 iterations + 2 set-up products)
    else:
        assert d["gpu_launches"] > 2 * (2 * 6 + 2)           # + halo exchange and border x ghost block of the set-up products
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["launches_timed"] == 2 * (6 + 2) and r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    assert d["config"]["workload"].startswith("27pt stencil 64^3") and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert ("cpu_baseline" in d) == (nproc == 1)
    if nproc == 1:
        assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0
        import numpy as np
        out = {k: np.load(os.path.join(dump, k + ".npy")) for k in ("x", "x_rows", "residual_norms")}
        assert sorted(os.listdir(dump)) == ["residual_norms.npy", "x.npy", "x_rows.npy"]
        assert all(a.dtype == np.float64 for a in out.values())
        assert np.array_equal(out["x_rows"], np.arange(64 ** 3)) and out["x"].shape == (64 ** 3,)
        assert np.isfinite(out["x"]).all() and np.abs(out["x"]).max() > 0
        rn, r0 = out["residual_norms"]
        assert rn / r0 == pytest.approx(d["residual_after_step"], rel=1e-12)
    else:
        assert d["config"]["partition"].startswith("2 parts")


def test_smoke_entry_point(simlib):
    """__graft_entry__.smoke() unchanged, on the stand-in: both solvers against the oracle."""
    p = subprocess.run([sys.executable, os.path.join(SIM, "run_module_sim.py"), "__graft_entry__:smoke"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS="2"), cwd=ROOT)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    assert p.stdout.count("status 0") == 2 and "smoke launches" in p.stdout


@pytest.mark.parametrize("nproc,partition", [(1, "rows"), (2, "nnz"), (3, "rows")])   # METIS is not linked into the stand-in
def test_python_driver_solves(nproc, partition, simlib, tmp_path):
    """python -m acg_b200.driver through its whole flow (per-rank ingest, partition, solver,
    report, manufactured-solution error, gathered solution file) on the stand-in."""
    import numpy as np
    from acg_b200 import matgen as mg, mtxio
    n, r, c, v = mg.stencil3d_27pt(10, 9, 8)
    path, sol = str(tmp_path / "A.mtx"), str(tmp_path / "x.mtx")
    mtxio.write_symmetric(path, n, r, c, v, binary=True)
    args = [path, "--binary", "--solver", "acg-pipelined", "--max-iterations", "300", "--residual-rtol", "1e-10",
            "--manufactured-solution", "--seed", "3", "--partition", partition, "--output-solution", sol, "-v"]
    script = os.path.join(SIM, "run_module_sim.py")
    if nproc == 1:
        cmd = [sys.executable, script, "acg_b200.driver"] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
               "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), script, "acg_b200.driver"] + args
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS="2"), cwd=ROOT)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    import re
    e1 = float(re.search(r"^error 2-norm: (\S+)", p.stderr, re.M).group(1))
    assert e1 < 1e-8 and "total solver time:" in p.stderr
    # the report is the aggregate over the ranks (as acgsolvercuda_fwritempi): the SpMV bytes of the whole
    # matrix whatever the number of parts -- 12 B per nonzero plus vector terms per SpMV
    gemv = re.search(r"gemv: \S+ seconds (\d+) times (\d+) B", p.stderr)
    nspmv, nbytes = int(gemv.group(1)), int(gemv.group(2))
    nnz_full = 2 * len(v) - n
    assert nspmv * 12 * nnz_full <= nbytes <= nspmv * (12 * nnz_full + 60 * n)
    xs = np.random.default_rng(3).uniform(-1.0, 1.0, n); xs /= np.linalg.norm(xs)
    x = np.array([float(t) for t in open(sol).read().split("\n")[2:] if t])
    assert len(x) == n and np.linalg.norm(x - xs) == pytest.approx(e1, rel=1e-6, abs=1e-14)


def test_c_example_program(simlib, tmp_path):
    """examples/acgb200_solve.c, unchanged, linked against the stand-in instead of the product
    library: read a Matrix Market file, solve, print the report and the solution."""
    import numpy as np
    from acg_b200 import matgen as mg, mtxio
    from oracle import Oracle
    exe = str(tmp_path / "acgb200_solve_sim")
    cc = subprocess.run(["/usr/bin/gcc", "-O2", "-std=gnu11", "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
                         os.path.join(ROOT, "examples", "acgb200_solve.c"), "-o", exe, "-L" + SIM, "-lacgb200_hostsim",
                         "-Wl,-rpath," + SIM], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr[-2000:]
    n, r, c, v = mg.stencil3d_27pt(9)
    for binary in (True, False):
        path = str(tmp_path / ("A.bin.mtx" if binary else "A.txt.mtx"))
        mtxio.write_symmetric(path, n, r, c, v, binary=binary)
        p = subprocess.run([exe, path] + (["--binary"] if binary else []) +
                           ["--solver", "acg-pipelined", "--residual-rtol", "1e-9", "--max-iterations", "200", "--print-solution"],
                           capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-2000:]
        O = Oracle()
        want = O.cg_pipelined(O.full_csr(n, r, c, v), np.ones(n), maxits=200, rtol=1e-9)
        x = np.array([float(t) for t in p.stdout.splitlines()[2:]])
        assert len(x) == n and np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()
        assert f"iterations: {want['niterations']}" in p.stderr


@pytest.mark.parametrize("nranks,solver,method", [(2, "acg", "cg"), (2, "acg-pipelined", "cg_pipelined"),
                                                  (4, "acg-pipelined", "cg_pipelined"), (3, "acg-device", "cg")])
def test_unmodified_reference_driver_on_several_ranks(nranks, solver, method, simlib, tmp_path):
    """The same unmodified driver as N processes under compat/mpi/acgb200-mpirun: MPI_Init over the
    stand-in (compat/mpi/mpishim.c), the matrix read on rank 0, partitioned with METIS by the
    reference's own acg/metis.c (compat/metis/metis.h + the toolkit's archive), scattered over MPI
    (acg/symcsrmatrix.c, acg/graph.c), the NCCL id broadcast over MPI (cuda/acg-cuda.c:1104-1122),
    the solve through libacgb200 with the peer-memory exchange between the processes, the solution
    gathered back and printed by rank 0 -- against the single-rank oracle."""
    import re
    import numpy as np
    from acg_b200 import matgen as mg, mtxio
    from oracle import Oracle
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "driver", "acg-cuda.o")):
        pytest.skip("driver objects not built (needs the reference tree: tools/build_driver.sh)")
    p = subprocess.run(["make", "-C", SIM, "driver"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]
    exe = os.path.join(SIM, "acg-cuda-sim")
    mpirun = os.path.join(ROOT, "compat", "mpi", "acgb200-mpirun")
    n, r, c, v = mg.stencil3d_27pt(12, 10, 11)
    path = str(tmp_path / "A.mtx")
    mtxio.write_symmetric(path, n, r, c, v, binary=True)
    p = subprocess.run([mpirun, "-n", str(nranks), exe, path, "--binary", "--comm", "nccl", "--solver", solver,
                        "--max-iterations", "200", "--residual-rtol", "1e-9", "--warmup", "2", "--numfmt", "%.17g"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stderr[-3000:]
    assert f"{nranks} MPI processes" in p.stderr or True
    O = Oracle()
    want = getattr(O, method)(O.full_csr(n, r, c, v), np.ones(n), maxits=200, rtol=1e-9)
    its = int(re.search(r"^\s*iterations: ([\d,]+)", p.stderr, re.M).group(1).replace(",", ""))
    r0 = float(re.search(r"^\s*initial residual 2-norm: (\S+)", p.stderr, re.M).group(1))
    assert its == want["niterations"] and r0 == pytest.approx(want["r0nrm2"], rel=1e-12)
    lines = [ln for ln in p.stdout.splitlines() if ln and not ln.startswith("%")]
    x = np.array([float(t) for t in lines[1:]])
    assert int(lines[0].split()[0]) == n and np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()


@pytest.mark.parametrize("solver,method", [("acg", "cg"), ("acg-pipelined", "cg_pipelined"),
                                           ("acg-device", "cg"), ("acg-device-pipelined", "cg_pipelined")])
def test_unmodified_reference_driver(solver, method, simlib, tmp_path):
    """The objects of the UNMODIFIED cuda/acg-cuda.c and of the reference's host layer
    (tools/build_driver.sh, compiled from where they lie) linked against the stand-in build of the
    MPI flavour of the library: the whole drop-in boundary -- the reference's own Matrix Market
    reader, acgsolvercuda_init, the solver dispatch of cuda/acg-cuda.c:2242-2262,
    acgsolvercuda_fwritempi, the solution on stdout -- on the CPU, against the oracle."""
    import re
    import numpy as np
    from acg_b200 import matgen as mg, mtxio
    from oracle import Oracle
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "driver", "acg-cuda.o")):
        pytest.skip("driver objects not built (needs the reference tree: tools/build_driver.sh)")
    p = subprocess.run(["make", "-C", SIM, "driver"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]
    exe = os.path.join(SIM, "acg-cuda-sim")
    n, r, c, v = mg.stencil3d_27pt(12, 10, 11)
    path = str(tmp_path / "A.mtx")
    mtxio.write_symmetric(path, n, r, c, v, binary=True)
    p = subprocess.run([exe, path, "--binary", "--solver", solver, "--max-iterations", "200", "--residual-rtol", "1e-9",
                        "--warmup", "2", "--numfmt", "%.17g"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    O = Oracle()
    want = getattr(O, method)(O.full_csr(n, r, c, v), np.ones(n), maxits=200, rtol=1e-9)
    its = int(re.search(r"^\s*iterations: ([\d,]+)", p.stderr, re.M).group(1).replace(",", ""))
    r0 = float(re.search(r"^\s*initial residual 2-norm: (\S+)", p.stderr, re.M).group(1))
    assert its == want["niterations"] and r0 == pytest.approx(want["r0nrm2"], rel=1e-13)
    lines = [ln for ln in p.stdout.splitlines() if ln and not ln.startswith("%")]
    x = np.array([float(t) for t in lines[1:]])
    assert int(lines[0].split()[0]) == n and np.abs(x - want["x"]).max() <= 1e-9 * np.abs(want["x"]).max()
    if solver == "acg":
        q = subprocess.run([exe, path, "--binary", "--solver", solver, "--max-iterations", "300", "--residual-rtol", "1e-10",
                            "--manufactured-solution", "--seed", "7", "-q"], capture_output=True, text=True, timeout=300)
        assert q.returncode == 0, q.stderr[-3000:]
        e0 = float(re.search(r"^initial error 2-norm: (\S+)", q.stderr, re.M).group(1))
        e1 = float(re.search(r"^error 2-norm: (\S+)", q.stderr, re.M).group(1))
        assert e0 == pytest.approx(1.0, rel=1e-12) and e1 < 1e-7


def test_public_blas1_building_blocks(simlib):
    """acg/cg-kernels-cuda.h:45-97 (alpha, beta, daxpy_alpha, daxpy_minus_alpha, daypx_beta,
    pipelined_daxpy_fused, init_constants): entry points, argument order and semantics."""
    out = _run({"matrix": "n3", "blas1_blocks": 1, "runs": []})
    assert out["blas1_blocks"] == {"scalars": True, "axpy": True, "pipelined": True, "constants": True}


def test_failing_device_allocations_are_survived(simlib):
    """Fault injection (tests/hostsim/cuda_mock.c, HOSTSIM_FAIL_MALLOC_AT): whichever "device"
    allocation of set-up or of the solves fails, the call returns ACG_ERR_CUDA, the process survives
    and tears down what had been built (the AddressSanitizer run of tools/asan_hostsim.sh repeats
    this on every allocation)."""
    script = os.path.join(SIM, "run_fault.py")
    seen = []
    for k in list(range(1, 25, 3)) + [24, 52, 55, 58, 60, 1000]:     # 52.. : inside acgsymcsrmatrix_dsymv_init_cuda
        p = subprocess.run([sys.executable, script], capture_output=True, text=True, timeout=120,
                           env=dict(os.environ, HOSTSIM_FAIL_MALLOC_AT=str(k), OMP_NUM_THREADS="2"))
        assert p.returncode == 0, (k, p.stderr[-2000:])
        seen.append((k, p.stdout.strip().splitlines()[-1]))
    assert all(out == "error 4" for k, out in seen if k <= 60), seen          # ACG_ERR_CUDA
    assert seen[-1] == (1000, "ok")
    # the same for any runtime call (copies, memsets, streams, events, graph capture / instantiate / launch)
    seen = []
    for k in list(range(2, 160, 13)) + [200, 220, 235, 100000]:
        p = subprocess.run([sys.executable, script], capture_output=True, text=True, timeout=120,
                           env=dict(os.environ, HOSTSIM_FAIL_CALL_AT=str(k), OMP_NUM_THREADS="2"))
        assert p.returncode == 0, (k, p.stderr[-2000:])
        seen.append((k, p.stdout.strip().splitlines()[-1]))
    assert all(out == "error 4" for k, out in seen if k <= 235), seen
    assert seen[-1] == (100000, "ok")


def test_gpu_test_files_rehearsed_on_the_stand_in(simlib):
    """The GPU parity files themselves, run against the stand-in instead of the product library
    (ACGB200_TEST_LIB): expected iteration counts, return codes, plan assertions (slices, merge tiles,
    exception rows), the byte-identity checks of the device-side expansion (here: expand_host.c around the
    stand-in's serial fill) -- so that a change of the host logic that would break the hardware run at round
    end shows up in the CPU suite.  Says nothing about the kernels."""
    env = dict(os.environ, ACGB200_TEST_LIB=simlib, OMP_NUM_THREADS="2")
    p = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_expand.py"),
                        os.path.join(ROOT, "tests", "test_gpu_parity.py"), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
                        "-k", "not public_blas1 and not full_size and not power_law"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-2000:]
    assert " passed" in p.stdout and "failed" not in p.stdout
