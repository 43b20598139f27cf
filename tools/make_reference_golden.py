"""Store what the reference computes for the tests that compare with it, under tests/golden/reference/.

The tests read these files instead of the reference build, so that they run from a clean checkout on any
machine.  Needs oracle/_ref (built by __graft_entry__.build() where the reference tree exists):

    python tools/make_reference_golden.py              # CPU library and headers of the reference
    python tools/make_reference_golden.py --stock-gpu  # its own GPU solver instead (on a B200)

Inputs are not stored: the tests regenerate them with the same seeded generators used here.  Arrays
that the tests compare bit for bit are stored as digests (tests/conftest.py, digest), in JSON files.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from acg_b200 import matgen as mg  # noqa: E402
from conftest import digest  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference")
REF_TREE = os.environ.get("ACG_REFERENCE_DIR", "")


def oracle_pin(R):
    """test_oracle_pin.py: full storage, dsymv, ddot, dnrm2sqr and acgsolver_solve on the CASES, the
    unsorted-input case and the status codes."""
    from test_oracle_pin import CASES
    out = {}
    for name, gen in CASES:
        n, r, c, v = gen()
        for k, a in zip(("frowptr", "fcolidx", "fa"), R.full_csr(n, r, c, v)):
            out[f"{name}__{k}"] = digest(a)
        rng = np.random.default_rng(1)
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        for i, (alpha, beta) in enumerate(((-1.0, 1.0), (1.0, 0.0), (0.5, 2.0))):
            out[f"{name}__dsymv{i}"] = digest(R.dsymv(n, r, c, v, alpha, x, beta, y))
        out[f"{name}__ddot"] = float(R.ddot(x, y))
        out[f"{name}__dnrm2sqr"] = float(R.dnrm2sqr(x))
        b = rng.standard_normal(n)
        for i, (maxits, rtol) in enumerate(((7, 0.0), (200, 1e-9))):
            f = R.cg(n, r, c, v, b, maxits=maxits, rtol=rtol)
            for k in ("status", "niterations"):
                out[f"{name}__cg{i}__{k}"] = int(f[k])
            for k in ("bnrm2", "r0nrm2", "rnrm2"):
                out[f"{name}__cg{i}__{k}"] = float(f[k])
            out[f"{name}__cg{i}__x"] = digest(f["x"])
    n, r, c, v = mg.stencil3d_27pt(5)
    perm = np.random.default_rng(3).permutation(len(v))
    r2, c2, v2 = (np.ascontiguousarray(a[perm]) for a in (r, c, v))
    for k, a in zip(("frowptr", "fcolidx", "fa"), R.full_csr(n, r2, c2, v2)):
        out[f"unsorted__{k}"] = digest(a)
    n, r, c, v = mg.stencil3d_27pt(6)
    b, z = np.ones(n), np.zeros(n)
    out["status__maxits"] = R.cg(n, r, c, v, b, maxits=3)["status"]
    out["status__not_converged"] = R.cg(n, r, c, v, b, maxits=3, rtol=1e-14)["status"]
    out["status__indefinite"] = R.cg(n, r, c, v, z, maxits=3, rtol=1e-9)["status"]
    xs = np.random.default_rng(4).standard_normal(n)
    bb = R.dsymv(n, r, c, v, 1.0, xs, 0.0, z)
    f = R.cg(n, r, c, v, bb, x0=xs, maxits=10, atol=1e-6)
    out["status__converged_x0"] = f["status"]
    out["status__converged_x0_niterations"] = f["niterations"]
    return out


def host_structs(R):
    """test_host_structs.py: full storage with a diagonal shift, and every part of the row partitions."""
    from test_host_structs import GENS, _parts, _rows_as_sets
    full, parts = {}, {}
    for name, gen in GENS:
        n, r, c, v = gen()
        for k, a in zip(("frowptr", "fcolidx", "fa"), R.full_csr(n, r, c, v, eps=0.25)):
            full[f"{name}__{k}"] = digest(a)
        for kind, nparts in (("slab", 3), ("cyclic", 2), ("random", 5)):
            rowparts = _parts(kind, n, nparts)
            for p in range(nparts):
                w = R.partition_part(n, r, c, v, nparts, rowparts, p)
                pre = f"{name}-{kind}-{p}__"
                for k in ("nprows", "nownedrows", "ninnerrows", "nborderrows", "nghostrows"):
                    parts[pre + k] = int(w[k])
                for k in ("nzrows", "recipients", "sendcounts", "sendbufidx", "senders", "recvcounts", "recvbufidx",
                          "frowptr", "orowptr"):
                    parts[pre + k] = digest(w[k])
                for s, nr in (("f", w["nownedrows"]), ("o", w["nborderrows"])):
                    ci, va = _rows_as_sets(w[s + "rowptr"], w[s + "colidx"], w[s + "a"], nr)
                    parts[pre + s + "colidx_rowsets"], parts[pre + s + "a_rowsets"] = digest(ci), digest(va)
    return full, parts


def struct_layouts():
    """test_abi.py: the layout probe compiled against the reference's headers."""
    from test_abi import _run_probe
    return _run_probe('#include "acg/vector.h"\n#include "acg/graph.h"\n#include "acg/symcsrmatrix.h"\n'
                      '#include "acg/cgcuda.h"\n#include "acg/error.h"', ["-I" + REF_TREE])


def stock_gpu(out_dir):
    """test_reference_driver.py: the reference's own GPU solver (acg/cgcuda.c with cuSPARSE/cuBLAS) after 30
    iterations on the 27-point 20^3 matrix, b = 1: its report and the solution it prints."""
    from acg_b200 import mtxio
    exe = os.path.join(ROOT, "oracle", "_ref", "driver_ref", "acg-cuda-ref")
    n, r, c, v = mg.stencil3d_27pt(20)
    out = {}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "A.mtx")
        mtxio.write_symmetric(path, n, r, c, v, binary=True)
        for solver in ("acg", "acg-pipelined"):
            p = subprocess.run([exe, path, "--binary", "--solver", solver, "--max-iterations", "30",
                                "--residual-rtol", "0", "--warmup", "1", "--numfmt", "%.17g"],
                               capture_output=True, text=True, timeout=300, check=True)
            rep = p.stderr
            out[f"{solver}__niterations"] = int(re.search(r"^\s*iterations: ([\d,]+)", rep, re.M).group(1).replace(",", ""))
            out[f"{solver}__rnrm2"] = float(re.search(r"^\s*residual 2-norm: (\S+)", rep, re.M).group(1))
            out[f"{solver}__r0nrm2"] = float(re.search(r"^\s*initial residual 2-norm: (\S+)", rep, re.M).group(1))
            lines = [ln for ln in p.stdout.splitlines() if ln and not ln.startswith("%") and not ln.startswith("NCCL")]
            out[f"{solver}__x"] = np.array([float(t) for t in lines[1:]])
            assert len(out[f"{solver}__x"]) == n
    np.savez_compressed(os.path.join(out_dir, "stock_gpu_27pt20.npz"), **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stock-gpu", action="store_true", help="store only what the reference's GPU solver computes (needs a GPU)")
    ap.add_argument("--out", default=OUT)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    if args.stock_gpu:
        stock_gpu(args.out)
        return
    from oracle import Ref, ref_available
    if not ref_available() or not os.path.isdir(os.path.join(REF_TREE, "acg")):
        raise SystemExit("needs oracle/_ref/libacgref.so and ACG_REFERENCE_DIR set to the reference tree")
    R = Ref()
    full, parts = host_structs(R)
    for name, d in (("oracle_pin", oracle_pin(R)), ("full_storage", full), ("partition", parts)):
        with open(os.path.join(args.out, name + ".json"), "w") as f:
            json.dump(d, f, indent=0, sort_keys=True)
            f.write("\n")
    with open(os.path.join(args.out, "struct_layouts.txt"), "w") as f:
        f.write(struct_layouts())


if __name__ == "__main__":
    main()
