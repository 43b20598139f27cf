#!/usr/bin/env python
"""bench.py -- CG iterations/s and SpMV roofline of the B200 hot path.

    python bench.py --gpus N --steps K --warmup W            (N=1)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N>1)
    python bench.py --impl reference ...                     (the reference's CPU path)

Workload (BASELINE.json configs[2], the configuration the metric is quoted on):
27-point stencil 224^3 (n = 11 239 424, nnz = 300 763 000), FP64, b = 1, x0 = 0,
pipelined CG.  N>1 splits the same matrix into N geometric blocks (strong
scaling), halo + allreduce over NCCL.

A *step* is one call of the reference-facing solver entry point
(acgsolvercuda_solve_pipelined / acgsolvercuda_solvempi) for ITERS iterations
with all tolerances off -- one pass of the hot path over one right-hand side.

  value   iterations/s from the device-side solve window (CUDA events inside the
          library around the region the reference times as "total solver time",
          acg/cgcuda.c:719-722,:1021): b and x are already in HBM.  Max over
          ranks of the summed window, K*ITERS iterations.
  e2e     iterations/s of the whole C-ABI call with HOST vectors: pinned b, x ->
          H2D, solve, x -> D2H, inside the timed region (host clock, device
          synchronised by the call itself; barrier before every step; max over
          ranks).
  roofline  the SpMV kernel (replaces cusparseSpMV): 16*nnz contract bytes
          (2*nnz*8, BASELINE.md §3) per launch / mean launch duration, measured
          with CUDA events on the launching stream inside the timed steps.
  cpu_baseline  the reference's own CPU solver (acg/cg.c, oracle/_ref) -- or the
          oracle port when that build is absent -- on the box's host cores, same
          matrix, a bounded number of iterations.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "27pt-224": dict(kind="27pt", N=224, solver="pipelined"),     # BASELINE.json configs[2]  (metric config)
    "7pt-256": dict(kind="7pt", N=256, solver="classic"),          # configs[1]
    "27pt-128": dict(kind="27pt", N=128, solver="pipelined"),      # quick check
    "27pt-112": dict(kind="27pt", N=112, solver="pipelined"),      # one rank's share of 27pt-224 on 8 GPUs, without the exchange
    "27pt-64": dict(kind="27pt", N=64, solver="pipelined"),
    "27pt-448": dict(kind="27pt", N=448, solver="pipelined"),      # configs[3]: 8 GPUs only (weak-scaled x8 point)
    # configs[4]: power-law rows (long-row path, gathers without locality); contiguous row blocks or METIS for N>1
    # (classic CG: on these ill-conditioned matrices -- hubs of degree 1e5 -- the recurrence residual of pipelined CG
    # drifts away from the true one within 100 iterations, profiles/r02/d_bench_rmat20m.json)
    "rmat-20M": dict(kind="rmat", N=20_000_000, edges=200_000_000, solver="classic"),
    "rmat-2M": dict(kind="rmat", N=2_000_000, edges=20_000_000, solver="classic"),
}


def make_matrix(w):
    """Upper-triangle COO of the whole matrix as the product's host generators build it (GPU arm only:
    METIS runs, the file handed to the stock reference GPU solver, and the R-MAT matrix, which is
    defined by the counter-based generator of acg_b200/csrc/rmat.c)."""
    import acg_b200 as ab
    N = w["N"]
    if w["kind"] == "rmat":
        A = ab.SymCsrMatrix.rmat_spd(N, w["edges"], seed=42)
    else:
        A = ab.SymCsrMatrix.stencil_part(27 if w["kind"] == "27pt" else 7, N, N, N, 1, 1, 1, 0)
    rp = A.rowptr
    rows = np.repeat(np.arange(A.c.nprows, dtype=np.int32), np.diff(rp).astype(np.int64))
    cols, vals = A.colidx.copy(), A.a.copy()
    n = int(A.c.nprows)
    A.free()
    return n, rows, cols, vals


def build_local_matrix(w, partition, rank, world):
    """This rank's part of the workload matrix with full storage initialised (GPU arm only)."""
    import acg_b200 as ab
    from acg_b200 import dist as abdist
    N = w["N"]
    if w["kind"] == "rmat":
        # power-law graph: no geometry; every rank generates the (deterministic) matrix and keeps its part
        A = ab.SymCsrMatrix.rmat_spd(N, w["edges"], seed=42)
        if world > 1:
            rowparts = (A.partition_rows(world, seed=0)[0] if partition == "metis"
                        else abdist.balanced_rows_partition(A, world))     # equal nonzeros, not equal rows
            parts = A.partition(world, rowparts)
            A.free()
            A = parts[rank]
            for p, m in enumerate(parts):
                if p != rank:
                    m.free()
        return A.dsymv_init(0.0)
    k = 27 if w["kind"] == "27pt" else 7
    if partition == "block" or world == 1:
        # every rank builds only its own block (no global matrix anywhere); one rank = the whole box
        if (N ** 3 * k) // world >= 2 ** 31:
            raise SystemExit(f"bench.py: {w['kind']} {N}^3 does not fit 32-bit indices on {world} GPU(s)")
        return abdist.local_stencil_part(k, N, N, N, rank, world)
    if N ** 3 * k >= 2 ** 31:
        raise SystemExit(f"bench.py: {w['kind']} {N}^3 is too large for a global METIS partition in one process")
    n, r, c, v = make_matrix(w)
    A = abdist.local_part(n, r, c, v, "metis", rank, world)
    del r, c, v
    return A


def rhs(w, gidx):
    """Right-hand side at the given global row numbers: all ones (the driver's default,
    cuda/acg-cuda.c:1949-1967) -- except for the R-MAT matrix, whose rows sum to 1 so that
    b = 1 is an eigenvector and CG would finish in one step."""
    if w["kind"] == "rmat":
        return 1.0 + 0.5 * np.sin(0.37 * np.asarray(gidx, dtype=np.float64))
    return np.ones(len(gidx))


def rhs_name(w):
    return "b_i=1+sin(0.37i)/2" if w["kind"] == "rmat" else "b=1"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [t.strip() for t in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc:
            self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 7] or [r for (_, r) in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def cpu_arm(w, iters, steps, warmup, save_x=None):
    """Run oracle/cpu_arm.py in a fresh process (threads pinned one per physical core, nothing of
    the product in it) and return its JSON.  Stencil matrices are generated inside that process;
    the R-MAT matrix is defined by the product's generator, so it is handed over as a file."""
    import tempfile
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "cpu_arm.py"), "--iters", str(iters),
           "--steps", str(steps), "--warmup", str(warmup)]
    tmp = None
    if w["kind"] == "rmat":
        n, r, c, v = make_matrix(w)
        tmp = tempfile.NamedTemporaryFile(suffix=".npz", dir="/dev/shm" if os.path.isdir("/dev/shm") else None, delete=False)
        np.savez(tmp, n=n, rows=r, cols=c, vals=v, b=rhs(w, np.arange(n)))
        tmp.close()
        del r, c, v
        cmd += ["--matrix", tmp.name]
    else:
        cmd += ["--kind", w["kind"], "--N", str(w["N"])]
    if save_x:
        cmd += ["--save-x", save_x]
    env = {k: v for k, v in os.environ.items() if not k.startswith(("OMP_", "GOMP_", "KMP_"))}
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, env=env)
    finally:
        if tmp:
            os.unlink(tmp.name)
    if p.returncode != 0:
        raise RuntimeError("oracle/cpu_arm.py failed: " + p.stderr[-2000:])
    return json.loads(p.stdout.strip().splitlines()[-1])


def cpu_reference(w, steps, warmup, iters, solver_note, save_x=None):
    """Time the reference's CPU CG (acg/cg.c through oracle/_ref; the oracle port when that build
    is absent) on the host's physical cores."""
    r = cpu_arm(w, iters, steps, warmup, save_x)
    times = r["times"]
    tot = sum(times)
    what = f"R-MAT n={w['N']}" if w["kind"] == "rmat" else f"{w['kind']} {w['N']}^3"
    return dict(value=len(times) * iters / tot, unit="iterations/s", cores=r["cores"], kind=r["kind"],
                sample=f"{len(times)} x {iters} classic CG iterations (acgsolver_solve, acg/cg.c:198) on the full {what} "
                       f"matrix, {rhs_name(w)}, x0=0; OpenMP dsymv on {r['cores']} threads pinned one per physical core, "
                       f"BLAS-1 serial as in the reference{solver_note}",
                seconds=tot, best_its_per_s=iters / min(times), median_its_per_s=iters / statistics.median(times),
                numa_interleave_nodes=r["numa_interleave_nodes"], matrix_placed_by_threads=r["matrix_placed_by_threads"],
                setup_s=r["setup_s"], rnrm2=r["rnrm2"], r0nrm2=r["r0nrm2"], niterations=r["niterations"])


def reference_gpu(w, iters, solver):
    """The stock reference GPU solver (acg/cgcuda.c: cusparseSpMV + cublasDdot + its own axpy
    kernels), built unmodified for sm_100a by tools/build_driver.sh, on the same matrix through a
    binary Matrix Market file.  Optional extra arm (--with-reference-gpu): the kernel to beat."""
    import re
    import tempfile
    from acg_b200 import mtxio
    exe = os.path.join(ROOT, "oracle", "_ref", "driver_ref", "acg-cuda-ref")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/driver_ref/acg-cuda-ref not built (needs the reference tree at build time)"}
    n, r, c, v = make_matrix(w)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "A.mtx")
        mtxio.write_symmetric(path, n, r, c, v, binary=True)
        del r, c, v
        p = subprocess.run([exe, path, "--binary", "--solver", "acg-pipelined" if solver == "pipelined" else "acg",
                            "--max-iterations", str(iters), "--residual-rtol", "0", "--warmup", "10", "-q"],
                           capture_output=True, text=True)
    if p.returncode != 0:
        return {"unavailable": "reference GPU solver failed: " + p.stderr[-300:]}
    t = float(re.search(r"total solver time: ([\d.,]+) seconds", p.stderr).group(1).replace(",", ""))
    its = int(re.search(r"^\s*iterations: ([\d,]+)", p.stderr, re.M).group(1).replace(",", ""))
    return {"value": its / t, "unit": "iterations/s", "iterations": its, "tsolve_s": t,
            "what": "unmodified aCG GPU solver (cuSPARSE SpMV, cuBLAS dot), 'total solver time' of its own report"}


DUMP_ROWS = 1 << 21       # 2 x 16 MB of float64 at most, whatever the workload


def dump_sample(x, rnrm2, r0nrm2):
    """What a caller of the timed solve receives, as float64 arrays: x at a fixed, seeded sample of
    DUMP_ROWS rows (every row of a smaller problem) with those row numbers, and ||r||, ||r0||."""
    n = len(x)
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    return {"x": x[rows].astype(np.float64), "x_rows": rows.astype(np.float64),
            "residual_norms": np.array([rnrm2, r0nrm2], dtype=np.float64)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="acgb200", choices=["acgb200", "reference"])
    ap.add_argument("--workload", default="27pt-224", choices=sorted(WORKLOADS))
    ap.add_argument("--solver", default=None, choices=["pipelined", "classic"])
    ap.add_argument("--iters", type=int, default=100, help="CG iterations per step (reference default --max-iterations 100)")
    ap.add_argument("--cpu-iters", type=int, default=None,
                    help="classic iterations per CPU step (default: 5 for --impl reference; --iters for the GPU arm's "
                         "cpu_baseline leg, whose x is also the full-size parity check)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-reference-gpu", action="store_true",
                    help="also run the stock reference GPU solver (cuSPARSE/cuBLAS) on the same matrix (1 GPU, adds minutes)")
    ap.add_argument("--partition", default="block", choices=["block", "metis"],
                    help="row partition for N>1: geometric blocks or METIS (acgsymcsrmatrix_partition_rows)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (x at a fixed sample of rows, the solver's residual "
                         "norms) as DIR/*.npy, to compare two builds output for output (1 GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.gpus != 1 or args.impl != "acgb200" or args.steps < 1):
        ap.error("--dump-outputs needs --gpus 1, --impl acgb200 and at least one step")
    # torchrun exports OMP_NUM_THREADS=1 to every rank unless the caller set it.  The host-side set-up
    # (matrix generator, full-storage expansion) is OpenMP code: give a rank of the GPU arm its share of
    # the host cores.  (The CPU arm sets its own OpenMP environment in its own process, oracle/cpu_arm.py.)
    # Must happen before anything loads libgomp (it reads the variable once).
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("OMP_NUM_THREADS") == "1" \
            and not os.environ.get("BENCH_KEEP_OMP_NUM_THREADS"):
        ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        os.environ["OMP_NUM_THREADS"] = str(max(1, ncpu // int(os.environ.get("LOCAL_WORLD_SIZE", os.environ["WORLD_SIZE"]))))
    w = WORKLOADS[args.workload]
    solver = args.solver or os.environ.get("BENCH_SOLVER") or w["solver"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    metric = "CG iterations/sec (27-pt stencil ~10M rows); SpMV achieved-HBM GB/s in roofline"
    what = (f"R-MAT power-law SPD, n={w['N']}, {w['edges']} draws" if w["kind"] == "rmat"
            else f"{w['kind']} stencil {w['N']}^3")
    config = {"workload": f"{what}, FP64, {rhs_name(w)}, x0=0, {solver} CG, {args.iters} iterations/step, "
                          f"tolerances off", "n": w["N"] if w["kind"] == "rmat" else w["N"] ** 3,
              "solver": solver, "iters_per_step": args.iters,
              "partition": (f"{world} parts, " + ("METIS recursive" if args.partition == "metis" else
                                                  ("contiguous row blocks of equal nonzero count" if w["kind"] == "rmat" else "geometric blocks")))
                           if world > 1 else "none",
              "reference_arm": {"solver": "classic", "iters_per_step": args.cpu_iters or 5,
                                "what": "--impl reference: the reference's CPU path is classic CG (acg/cg.c:198; it has no CPU "
                                        "pipelined CG); a step = this many of its iterations on the same matrix, b and x0"},
              "l2": None}
    k = 27 if w["kind"] == "27pt" else 7
    if w["kind"] == "rmat":
        csr_gb = 12.0 * 2.1 * w["edges"] / world / 1e9
    else:
        csr_gb = 12.0 * ((3 * w["N"] - 2) ** 3 if k == 27 else 7 * w["N"] ** 3 - 6 * w["N"] ** 2) / world / 1e9
    config["l2"] = (f"inputs larger than L2 (CSR {csr_gb:.2f} GB per SpMV per GPU vs 126 MB L2), no flush needed"
                    if csr_gb > 0.26 else f"CSR {csr_gb:.2f} GB per GPU: partly L2-resident, not a roofline-valid size")

    if args.impl == "reference":
        if rank != 0:
            return 0
        # The reference has no CPU pipelined CG: its CPU path is classic CG (acg/cg.c); a step of this
        # arm is config.reference_arm.iters_per_step of those iterations on the same matrix and
        # right-hand side (the metric, iterations/s, is per iteration either way).  Both arms print
        # the same config, which states what each of them runs.
        cpu_iters = config["reference_arm"]["iters_per_step"]
        cb = cpu_reference(w, args.steps, args.warmup, cpu_iters, "")
        line = {"impl": "reference", "metric": metric, "value": cb["value"], "unit": "iterations/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * cb["seconds"] / max(args.steps, 1), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import acg_b200 as ab
    from acg_b200 import dist as abdist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    rank, world, local = abdist.init_process(backend="gloo")
    import torch.distributed as dist
    comm = abdist.nccl_comm(rank, world)

    A = build_local_matrix(w, args.partition, rank, world)
    nnz_local = int(A.c.fnpnzs + A.c.onpnzs)
    cg = ab.SolverCuda(A, comm)
    b = A.vector()
    nown = A.c.nownedrows
    gidx = A.nzrows[:nown] if len(A.nzrows) >= nown else np.arange(nown)     # global row numbers of the owned rows
    b.x[:] = 0.0
    b.x[:nown] = rhs(w, gidx)
    x = A.vector()
    b.pin(); x.pin()
    h2d = 2 * b.c.num_nonzeros * 8
    d2h = x.c.num_nonzeros * 8
    solve = cg.solve_pipelined if solver == "pipelined" else cg.solvempi

    def step(fn=None):
        x.x[:] = 0.0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        code = (fn or solve)(b, x, maxits=args.iters)
        t1 = time.perf_counter()
        assert code == 0 and cg.c.niterations == args.iters
        return t1 - t0

    for _ in range(max(args.warmup, 0)):
        step()
    # ---- timed region: K steps, no profiling hooks (iterations replay as CUDA graphs)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    tw0 = time.time()
    host_s = dev_ms = 0.0
    launches = 0
    for _ in range(args.steps):
        host_s += step()
        inf = cg.info()
        dev_ms += inf["last_solve_ms"]
        launches += inf["last_launches"]
    if args.dump_outputs:
        dumped = dump_sample(x.x[:nown], cg.c.rnrm2, cg.c.r0nrm2)
    # ---- same steps again with a CUDA-event pair around every SpMV on its launching
    # stream (the library's profile mode; it issues the same kernels un-graphed)
    ab.set_option("profile", 1)
    spmv_ms = blas_ms = 0.0
    spmv_n = 0
    for _ in range(args.steps):
        step()
        inf = cg.info()
        spmv_ms += inf["last_spmv_ms"]; spmv_n += inf["last_spmv_count"]
        blas_ms += inf["last_blas_ms"]
    ab.set_option("profile", 0)
    torch.cuda.synchronize()
    tw1 = time.time()
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    info = cg.info()
    resid = cg.c.rnrm2 / cg.c.r0nrm2
    x_main = x.x[:nown].copy()
    check = None
    if world == 1:
        # outside every timed region: the residual recomputed from the returned x with one more
        # SpMV, next to the recurrence residual the solver reports (pipelined CG reports the last
        # tested iterate, one step behind)
        ax, _ = cg.spmv(x_main)
        true_rel = float(np.linalg.norm(b.x[:nown] - ax) / cg.c.r0nrm2)
        check = {"true_residual_rel": true_rel, "reported_residual_rel": float(resid),
                 "what": "||b - A x|| / ||r0|| from the x of the last step vs the solver's own figure"}

    t = torch.tensor([dev_ms, host_s], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, host_s_max = float(t[0]), float(t[1])
    total_iters = args.steps * args.iters

    # ---- full-size parity against the reference's CPU solver (1 GPU, outside the timed regions):
    # the same args.iters classic iterations of acg/cg.c on the same matrix; its timing is the
    # cpu_baseline, its x and residual the parity figures (north_star: 1e-10 relative)
    cpu_baseline = parity = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        import tempfile
        cpu_iters = args.cpu_iters or args.iters
        xs = None
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
            xfile = os.path.join(td, "x_cpu.npy") if cpu_iters == args.iters else None
            cpu_baseline = cpu_reference(w, 1, 0, cpu_iters, "" if solver == "classic" else "; GPU arm runs pipelined CG", xfile)
            if xfile and os.path.exists(xfile):
                xs = np.load(xfile)
        if xs is not None:
            step(cg.solvempi)                                   # GPU classic CG, same iterations
            x_classic = x.x[:nown].copy()
            r0 = cpu_baseline["r0nrm2"]
            scale = float(np.abs(xs).max())
            parity = {"iterations": args.iters, "cpu": "acgsolver_solve (acg/cg.c:198), oracle/_ref" if cpu_baseline["kind"] == "reference" else "oracle port",
                      "gpu_classic_vs_cpu": {
                          "rel_residual_diff": abs(cg.c.rnrm2 - cpu_baseline["rnrm2"]) / r0,
                          "residual_ratio_minus_1": cg.c.rnrm2 / cpu_baseline["rnrm2"] - 1.0,
                          "max_rel_x_diff": float(np.abs(x_classic - xs).max() / scale),
                          "gpu_rnrm2": cg.c.rnrm2, "cpu_rnrm2": cpu_baseline["rnrm2"], "r0nrm2": r0},
                      "tolerance": 1e-10}
            if solver == "pipelined":
                parity["gpu_pipelined_vs_gpu_classic"] = {
                    "max_rel_x_diff": float(np.abs(x_main - x_classic).max() / scale),
                    "note": "pipelined CG is a different recurrence (acg/cgcuda.c:1676-1788): same Krylov iterates in exact "
                            "arithmetic, rounding differs; its reported residual is one iteration behind"}
            parity["pass"] = bool(parity["gpu_classic_vs_cpu"]["rel_residual_diff"] <= 1e-10
                                  and parity["gpu_classic_vs_cpu"]["max_rel_x_diff"] <= 1e-10)

    if rank == 0:
        peak, peak_src = peaks()
        t_spmv = spmv_ms / max(spmv_n, 1) * 1e-3
        nloc = nown
        achieved = 16.0 * nnz_local / t_spmv / 1e9
        # the SpMV of one vector: rows that repeat a pattern through spmv_slices_kernel, the others through spmv_tiles_kernel
        parts = (["spmv_slices_kernel"] if info["spmv_slices"] > 0 else []) + \
                (["spmv_merge_kernel"] if info["spmv_merge_tiles"] > 0 else []) + \
                (["spmv_tiles_kernel"] if info["spmv_ntiles"] > 0 else [])
        kernel_name = " + ".join(parts) or "spmv_tiles_kernel"
        min_bytes = float(info["spmv_min_bytes"])
        prof = os.path.join(ROOT, "profiles", "r02", "h_ncu_slices.json")
        traffic_source = None
        if os.path.exists(prof) and world == 1 and args.workload == "27pt-224" and info["spmv_slice_rows"] == nloc:
            pj = json.load(open(prof))
            traffic_source = {"file": "profiles/r02/h_ncu_slices.json", "kernel": pj.get("kernel"),
                              "dram_bytes_per_launch": pj.get("dram_bytes_per_launch"),
                              "note": "ncu --set full capture of the same kernel and workload, committed; not measured in this run"}
        line = {
            "metric": metric, "value": total_iters / (dev_ms_max * 1e-3), "unit": "iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "e2e": {"value": total_iters / host_s_max, "unit": "iterations/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "whole acgsolvercuda_solve* call with pinned host b, x: H2D of b and x0, set-up, iterations, D2H of x"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": kernel_name,
                         "slice_rows": info["spmv_slice_rows"], "merge_rows": info["spmv_merge_rows"],
                         "tile_rows": nloc - info["spmv_slice_rows"] - info["spmv_merge_rows"],
                         "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": None, "traffic_source": traffic_source,
                         "bytes_per_launch": 16 * nnz_local, "ms_per_launch": t_spmv * 1e3, "launches_timed": spmv_n,
                         "peak_source": peak_src,
                         "min_bytes_per_launch": min_bytes,
                         "achieved_min_traffic_gbs": min_bytes / t_spmv / 1e9,
                         "frac_min_traffic": min_bytes / t_spmv / 1e9 / peak,
                         "spmv_gflops": 2.0 * nnz_local / t_spmv / 1e9,
                         "update_ms_per_iteration": blas_ms / max(args.steps * args.iters, 1),
                         "note": "achieved/frac: 16*nnz contract bytes (BASELINE.md, SURVEY 8d); *_min_traffic: the bytes the "
                                 "kernel's data layout must move at least (values, indices or pattern ids, row pointers, x, y); "
                                 "rank 0's local block"},
            "clocks": clocks,
            "residual_after_step": resid,
            "check": check,
        }
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        if parity:
            line["parity"] = parity
        if world == 1 and args.with_reference_gpu:
            cg.free(); b.free(); x.free(); A.free()          # give the memory back first
            line["reference_gpu"] = reference_gpu(w, args.iters, solver)
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    cg.free(); b.free(); x.free()
    comm.destroy()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
