"""The oracle (oracle/cg_oracle.c) against the reference's own code and vectors.

* bit-for-bit against what oracle/_ref/libacgref.so (the unmodified reference
  sources, compiled with -ffp-contract=off like the oracle) computed on seeded
  inputs, stored in tests/golden/reference/oracle_pin.json as scalars and
  array digests (tools/make_reference_golden.py);
* bit-for-bit against the committed fixtures tests/golden/*.npz, which were
  produced by that library alone (tools/make_golden.py);
* the known-answer tests SURVEY.md §8(c) lists (KAT-1, KAT-2, KAT-3, KAT-6).
"""
import os

import numpy as np
import pytest

from acg_b200 import matgen as mg
from conftest import GOLDEN, digest, load_golden, load_golden_json

CASES = [
    ("27pt", lambda: mg.stencil3d_27pt(8)),
    ("27pt-aniso", lambda: mg.stencil3d_27pt(5, 9, 4)),
    ("7pt", lambda: mg.laplace3d_7pt(9, 10, 11)),
    ("1d5", lambda: mg.poisson1d_5pt(777)),
    ("1d3", lambda: mg.poisson1d_3pt(64)),
    ("rand", lambda: mg.random_spd(150, 0.2, 3)),
    ("rmat", lambda: mg.rmat_spd(2000, 20000)),
]


@pytest.fixture(scope="module")
def pin():
    return load_golden_json("oracle_pin")


@pytest.mark.parametrize("name,gen", CASES, ids=[c[0] for c in CASES])
def test_oracle_equals_reference_bitwise(name, gen, oracle, pin):
    n, r, c, v = gen()
    csr_o = oracle.full_csr(n, r, c, v)
    for a, k in zip(csr_o, ("frowptr", "fcolidx", "fa")):
        assert digest(a) == pin[f"{name}__{k}"], k
    rng = np.random.default_rng(1)
    x, y = rng.standard_normal(n), rng.standard_normal(n)
    # the two uses in acg/cg.c: r -= A x (alpha=-1,beta=1) and t = A p (alpha=1,beta=0)
    for i, (alpha, beta) in enumerate(((-1.0, 1.0), (1.0, 0.0), (0.5, 2.0))):
        assert digest(oracle.dsymv(csr_o, alpha, x, beta, y)) == pin[f"{name}__dsymv{i}"]
    assert oracle.ddot(x, y) == pin[f"{name}__ddot"]
    assert oracle.dnrm2sqr(x) == pin[f"{name}__dnrm2sqr"]
    b = rng.standard_normal(n)
    for i, (maxits, rtol) in enumerate(((7, 0.0), (200, 1e-9))):
        o = oracle.cg(csr_o, b, maxits=maxits, rtol=rtol)
        for k in ("status", "niterations", "bnrm2", "r0nrm2", "rnrm2"):
            assert o[k] == pin[f"{name}__cg{i}__{k}"], k
        assert digest(o["x"]) == pin[f"{name}__cg{i}__x"]


def test_unsorted_coo_input(oracle, pin):
    """acg/symcsrmatrix.c:133-141: unsorted input takes the scatter branch."""
    n, r, c, v = mg.stencil3d_27pt(5)
    perm = np.random.default_rng(3).permutation(len(v))
    r2, c2, v2 = (np.ascontiguousarray(a[perm]) for a in (r, c, v))
    for a, k in zip(oracle.full_csr(n, r2, c2, v2), ("frowptr", "fcolidx", "fa")):
        assert digest(a) == pin[f"unsorted__{k}"], k


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_matches_golden_vectors(path, oracle):
    g = load_golden(path)
    n = int(g["n"])
    csr = oracle.full_csr(n, g["rows"], g["cols"], g["vals"])
    assert np.array_equal(csr[0], g["frowptr"]) and np.array_equal(csr[1], g["fcolidx"]) and np.array_equal(csr[2], g["fa"])
    assert np.array_equal(oracle.dsymv(csr, 1.0, g["xs"], 0.0, np.zeros(n)), g["y"])
    assert np.array_equal(oracle.dsymv(csr, -1.0, g["xs"], 1.0, g["b"]), g["y2"])
    o = oracle.cg(csr, g["b"], maxits=int(g["maxits"]), rtol=float(g["rtol"]))
    assert o["status"] == int(g["status"]) and o["niterations"] == int(g["niterations"])
    assert np.array_equal(o["x"], g["x"])
    assert o["bnrm2"] == float(g["bnrm2"]) and o["r0nrm2"] == float(g["r0nrm2"]) and o["rnrm2"] == float(g["rnrm2"])


def test_kat1_poisson_closed_form(oracle):
    """tridiag(-1,2,-1), b=1: x_i=(i+1)(n-i)/2 after exactly n/2 iterations."""
    n, r, c, v = mg.poisson1d_3pt(1000)
    o = oracle.cg(oracle.full_csr(n, r, c, v), np.ones(n), maxits=2000, rtol=1e-10)
    i = np.arange(n)
    assert o["status"] == 0 and o["niterations"] == 500
    assert o["bnrm2"] == pytest.approx(np.sqrt(n), rel=1e-15)
    assert np.allclose(o["x"], (i + 1) * (n - i) / 2, rtol=1e-12, atol=0)
    assert o["x"][0] == 500.0 and o["x"][500] == 125250.0


def test_kat2_dsymv_vs_dense(oracle):
    n, r, c, v = mg.random_spd(180, 0.15, 11)
    A = mg.upper_to_dense(n, r, c, v)
    csr = oracle.full_csr(n, r, c, v)
    rng = np.random.default_rng(0)
    x, y = rng.standard_normal(n), rng.standard_normal(n)
    for alpha, beta in ((1.0, 0.0), (-1.0, 1.0)):
        assert np.allclose(oracle.dsymv(csr, alpha, x, beta, y), alpha * A @ x + beta * y, rtol=1e-13, atol=1e-13)


def test_kat3_ddot_summation_order(oracle):
    """acg/vector.c:581-588: four interleaved partial sums, remainder into the first."""
    x = np.array([1e16, 1.0, -1e16, 1.0, 1.0, 1.0, 1.0, 1.0, 3.0])
    y = np.ones_like(x)
    c = [x[0] + x[4], x[1] + x[5], x[2] + x[6], x[3] + x[7]]
    c[0] = c[0] + x[8]
    assert oracle.ddot(x, y) == ((c[0] + c[1]) + c[2]) + c[3]


def test_kat6_pipelined_tracks_classic(oracle):
    n, r, c, v = mg.stencil3d_27pt(12)
    csr = oracle.full_csr(n, r, c, v)
    b = np.random.default_rng(2).standard_normal(n)
    a = oracle.cg(csr, b, maxits=60, history=True)
    p = oracle.cg_pipelined(csr, b, maxits=60, history=True)
    k = 30
    assert np.allclose(a["rnrm2hist"][:k], p["rnrm2hist"][:k], rtol=1e-8)
    assert np.abs(a["x"] - p["x"]).max() <= 1e-9 * np.abs(a["x"]).max()


def test_status_codes_and_edge_cases(oracle, pin):
    n, r, c, v = mg.stencil3d_27pt(6)
    csr = oracle.full_csr(n, r, c, v)
    b = np.ones(n)
    # maxits only -> success; tolerance not met -> ACG_ERR_NOT_CONVERGED (39)
    assert oracle.cg(csr, b, maxits=3)["status"] == pin["status__maxits"] == 0
    assert oracle.cg(csr, b, maxits=3, rtol=1e-14)["status"] == pin["status__not_converged"] == 39
    # b = 0: r0 = 0, the scaled tolerance is 0, p.Ap = 0 -> indefinite (40)
    z = np.zeros(n)
    assert oracle.cg(csr, z, maxits=3, rtol=1e-9)["status"] == pin["status__indefinite"] == 40
    # already converged initial guess
    xs = np.random.default_rng(4).standard_normal(n)
    bb = oracle.dsymv(csr, 1.0, xs, 0.0, z)
    o = oracle.cg(csr, bb, x0=xs, maxits=10, atol=1e-6)
    assert o["niterations"] == pin["status__converged_x0_niterations"] == 0
    assert o["status"] == pin["status__converged_x0"] == 0
