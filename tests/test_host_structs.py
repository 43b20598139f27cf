"""Host-side data structures of libacgb200 (no GPU): packed/full storage,
row partition, halo pattern.  Checked against what the reference build computed
(tests/golden/reference/, tools/make_reference_golden.py) and against the
invariants of SURVEY.md §8(c) KAT-5."""
import os

import numpy as np
import pytest

from acg_b200 import matgen as mg
from conftest import digest, load_golden_json

GENS = [
    ("27pt", lambda: mg.stencil3d_27pt(7)),
    ("7pt", lambda: mg.laplace3d_7pt(5, 6, 7)),
    ("rand", lambda: mg.random_spd(120, 0.15, 1)),
    ("rmat", lambda: mg.rmat_spd(500, 4000, seed=5)),
    ("1d5", lambda: mg.poisson1d_5pt(300)),
]


def _parts(kind, n, nparts):
    if kind == "slab":
        return (np.arange(n) * nparts // n).astype(np.int32)
    if kind == "cyclic":
        return (np.arange(n) % nparts).astype(np.int32)
    return np.random.default_rng(9).integers(0, nparts, n).astype(np.int32)


def _rows_as_sets(rowptr, colidx, vals, nrows):
    """Entries of the first nrows rows, each row sorted by (column, value): a canonical form of every row
    taken as a set of (column, value) pairs."""
    order = [rowptr[i] + np.lexsort((vals[rowptr[i]:rowptr[i + 1]], colidx[rowptr[i]:rowptr[i + 1]]))
             for i in range(nrows)]
    order = np.concatenate(order) if order else np.zeros(0, np.int64)
    return colidx[order], vals[order]


@pytest.mark.parametrize("name,gen", GENS, ids=[g[0] for g in GENS])
def test_full_storage_matches_reference(name, gen, ab):
    n, r, c, v = gen()
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v).dsymv_init(0.25)
    want = load_golden_json("full_storage")
    for k in ("frowptr", "fcolidx", "fa"):
        assert digest(getattr(A, k)) == want[f"{name}__{k}"], k
    assert A.c.nownedrows == n and A.c.nghostrows == 0 and A.c.onpnzs == 0


def test_unsorted_and_one_based_input(ab, oracle):
    n, r, c, v = mg.stencil3d_27pt(5)
    perm = np.random.default_rng(3).permutation(len(v))
    A = ab.SymCsrMatrix.init_real_double(n, r[perm] + 1, c[perm] + 1, v[perm], idxbase=1).dsymv_init(0.0)
    rp, ci, va = oracle.full_csr(n, np.ascontiguousarray(r[perm]), np.ascontiguousarray(c[perm]), np.ascontiguousarray(v[perm]))
    assert np.array_equal(A.frowptr, rp) and np.array_equal(A.fcolidx - 1, ci) and np.array_equal(A.fa, va)
    with pytest.raises(ab.AcgError) as e:
        ab.SymCsrMatrix.init_real_double(n, r, c + n, v)
    assert e.value.code == 31   # ACG_ERR_INDEX_OUT_OF_BOUNDS


@pytest.mark.parametrize("name,gen", GENS, ids=[g[0] for g in GENS])
@pytest.mark.parametrize("kind,nparts", [("slab", 3), ("cyclic", 2), ("random", 5)])
def test_partition_matches_reference(name, gen, kind, nparts, ab):
    n, r, c, v = gen()
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
    rowparts = _parts(kind, n, nparts)
    parts = A.partition(nparts, rowparts)
    golden = load_golden_json("partition")
    for p, m in enumerate(parts):
        m.dsymv_init(0.0)
        want = {k[len(f"{name}-{kind}-{p}__"):]: a for k, a in golden.items() if k.startswith(f"{name}-{kind}-{p}__")}
        for k in ("nprows", "nownedrows", "ninnerrows", "nborderrows", "nghostrows"):
            assert getattr(m.c, k) == want[k], k
        assert digest(m.nzrows) == want["nzrows"]
        h = m.halo()
        for k in ("recipients", "sendcounts", "sendbufidx", "senders", "recvcounts", "recvbufidx"):
            assert digest(h[k]) == want[k], k
        for k in ("frowptr", "orowptr"):
            assert digest(getattr(m, k)) == want[k], k
        # The order of entries inside a row may legitimately differ (the reference
        # lists a row's own upper-triangle entries before the mirrored ones, this
        # library follows global row order); compare rows as sets of (column, value).
        for s, nr in (("f", m.c.nownedrows), ("o", m.c.nborderrows)):
            ci, va = _rows_as_sets(getattr(m, s + "rowptr"), getattr(m, s + "colidx"), getattr(m, s + "a"), nr)
            assert digest(ci) == want[s + "colidx_rowsets"] and digest(va) == want[s + "a_rowsets"], s


@pytest.mark.parametrize("kind,nparts", [("slab", 4), ("random", 3)])
def test_partition_invariants_and_distributed_product(kind, nparts, ab, oracle):
    """KAT-5 plus an end-to-end check that the partitioned blocks and the halo
    pattern reproduce y = A x (host arithmetic in numpy, test-only)."""
    n, r, c, v = mg.stencil3d_27pt(6, 5, 7)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v).dsymv_init(0.0)
    csr = (A.frowptr.copy(), A.fcolidx.copy(), A.fa.copy())
    x = np.random.default_rng(0).standard_normal(n)
    ywant = oracle.dsymv(csr, 1.0, x, 0.0, np.zeros(n))
    rowparts = _parts(kind, n, nparts)
    parts = A.partition(nparts, rowparts)
    for m in parts:
        m.dsymv_init(0.0)
    assert sum(m.c.nownedrows for m in parts) == n
    halos = [m.halo() for m in parts]
    xloc = []
    for p, m in enumerate(parts):
        assert m.c.borderrowoffset == m.c.ninnerrows and m.c.ghostrowoffset == m.c.nownedrows
        assert np.all(rowparts[m.nzrows[:m.c.nownedrows]] == p)
        assert np.all(rowparts[m.nzrows[m.c.nownedrows:]] != p)
        h = halos[p]
        assert np.array_equal(h["recvbufidx"], m.c.ghostrowoffset + np.arange(m.c.nghostrows))
        assert np.all((h["sendbufidx"] >= m.c.borderrowoffset) & (h["sendbufidx"] < m.c.ghostrowoffset))
        assert np.all(m.fcolidx < m.c.ghostrowoffset)            # local block never touches ghosts
        xl = np.zeros(m.c.nprows)
        xl[:m.c.nownedrows] = x[m.nzrows[:m.c.nownedrows]]
        xloc.append(xl)
    # halo exchange "by hand": what p sends to q lands in q's segment for sender p
    for p in range(nparts):
        hp = halos[p]
        for i, q in enumerate(hp["recipients"]):
            seg = xloc[p][hp["sendbufidx"][hp["sdispls"][i]:hp["sdispls"][i] + hp["sendcounts"][i]]]
            hq = halos[q]
            j = list(hq["senders"]).index(p)
            assert hq["recvcounts"][j] == len(seg)
            xloc[q][hq["recvbufidx"][hq["rdispls"][j]:hq["rdispls"][j] + len(seg)]] = seg
    y = np.zeros(n)
    for p, m in enumerate(parts):
        assert np.array_equal(xloc[p][m.c.nownedrows:], x[m.nzrows[m.c.nownedrows:]])
        yl = np.zeros(m.c.nownedrows)
        for i in range(m.c.nownedrows):
            k0, k1 = m.frowptr[i], m.frowptr[i + 1]
            yl[i] = m.fa[k0:k1] @ xloc[p][m.fcolidx[k0:k1]]
        b0 = m.c.borderrowoffset
        for i in range(m.c.nborderrows):
            k0, k1 = m.orowptr[i], m.orowptr[i + 1]
            yl[b0 + i] += m.oa[k0:k1] @ xloc[p][b0 + m.ocolidx[k0:k1]]
        y[m.nzrows[:m.c.nownedrows]] = yl
    assert np.allclose(y, ywant, rtol=1e-13, atol=1e-13)


def test_vectors(ab):
    n, r, c, v = mg.laplace3d_7pt(4)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
    parts = A.partition(2, _parts("slab", n, 2))
    full = A.vector()
    full.x[:] = np.arange(n)
    for m in parts:
        pv = m.vector()
        assert pv.c.num_nonzeros == m.c.nprows and pv.c.num_ghost_nonzeros == m.c.nghostrows and pv.c.size == n
        assert ab.lib().acgvector_usga(pv.c, full.c) == 0
        assert np.array_equal(pv.x, m.nzrows.astype(float))


def test_solver_refuses_without_device(ab):
    """No CPU fallback: without a usable device init fails with ACG_ERR_CUDA."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    n, r, c, v = mg.poisson1d_3pt(10)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v).dsymv_init(0.0)
    with pytest.raises(ab.AcgError) as e:
        ab.SolverCuda(A)
    assert e.value.code == 4


@pytest.mark.parametrize("name,gen", GENS + [("rmat-long", lambda: mg.rmat_spd(20000, 400000, seed=8)),
                                             ("dense-rows", lambda: mg.random_spd(400, 0.5, 2)),
                                             ("n1", lambda: mg.poisson1d_3pt(1))],
                         ids=[g[0] for g in GENS] + ["rmat-long", "dense-rows", "n1"])
def test_spmv_tile_plan_invariants(name, gen, ab, oracle):
    """The SpMV tile plan (host logic of the CUDA path): every row is in exactly
    one tile or in the long-row list, tiles respect both caps, and every slice
    meets the 16-byte rule of cp.async.bulk (starts/lengths multiples of 4
    elements) while covering the tile's nonzeros."""
    n, r, c, v = gen()
    rowptr = oracle.full_csr(n, r, c, v)[0]
    plan = ab.spmv_plan_host(rowptr)
    lens = np.diff(rowptr)
    G, rows_cap, nnz_cap = plan["lanes"], plan["rows_cap"], plan["nnz_cap"]
    assert G in (1, 2, 4, 8, 16, 32) and rows_cap == 128 // G and nnz_cap % 4 == 0 and plan["stages"] == 2
    covered = np.zeros(n, int)
    covered[plan["longrows"]] += 1
    assert np.all(lens[plan["longrows"]] > nnz_cap)
    prev_end = 0
    for row_begin, nrows, k_al, nnz_al in plan["tiles"]:
        assert 1 <= nrows <= rows_cap and row_begin >= prev_end
        prev_end = row_begin + nrows
        covered[row_begin:row_begin + nrows] += 1
        kb, ke = rowptr[row_begin], rowptr[row_begin + nrows]
        assert ke - kb <= nnz_cap and np.all(lens[row_begin:row_begin + nrows] <= nnz_cap)
        assert k_al % 4 == 0 and nnz_al % 4 == 0 and k_al <= kb < k_al + 4 and k_al + nnz_al >= ke
        assert nnz_al <= nnz_cap + 8          # fits the shared-memory stage (stage_slots in kernels.cu)
    assert np.all(covered == 1)
    if name == "rmat-long":
        assert len(plan["longrows"]) > 0
    if name == "27pt":
        assert G == 4
    if name == "7pt":
        assert G == 1


@pytest.mark.parametrize("kind,nparts", [("slab", 2), ("random", 4), ("cyclic", 3)])
def test_peer_memory_push_addressing(kind, nparts, ab):
    """Host logic of the peer-memory halo exchange (p2p.c): pushing every border
    row through the inverse send map into the recipients' ghost buffers fills
    each ghost slot exactly once with the value of the global row it mirrors."""
    n, r, c, v = mg.stencil3d_27pt(6, 7, 5)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
    parts = A.partition(nparts, _parts(kind, n, nparts))
    halos = [m.halo() for m in parts]
    x = np.random.default_rng(0).standard_normal(n)
    ghost = [np.full(m.c.nghostrows, np.nan) for m in parts]
    writes = [np.zeros(m.c.nghostrows, int) for m in parts]
    for p, m in enumerate(parts):
        h = halos[p]
        # what rank p learns from the all-gather: where its segment starts at each recipient
        rd = [int(halos[q]["rdispls"][list(halos[q]["senders"]).index(p)]) for q in h["recipients"]]
        inv = m.p2p_inverse_map(rd)
        assert inv["bptr"][0] == 0 and inv["bptr"][-1] == len(h["sendbufidx"])
        xl = x[m.nzrows[:m.c.nownedrows]]
        for b in range(m.c.nborderrows):
            assert inv["bptr"][b + 1] > inv["bptr"][b]          # every border row has a recipient
            for e in range(inv["bptr"][b], inv["bptr"][b + 1]):
                q = int(h["recipients"][inv["bq"][e]])
                ghost[q][inv["bdst"][e]] = xl[m.c.borderrowoffset + b]
                writes[q][inv["bdst"][e]] += 1
    for p, m in enumerate(parts):
        assert np.all(writes[p] == 1)
        assert np.array_equal(ghost[p], x[m.nzrows[m.c.nownedrows:]])


@pytest.mark.parametrize("name,gen,full", [
    ("27pt", lambda: mg.stencil3d_27pt(9, 8, 7), True),
    ("7pt", lambda: mg.laplace3d_7pt(8, 9, 10), True),
    ("1d5", lambda: mg.poisson1d_5pt(500), True),
    ("rmat", lambda: mg.rmat_spd(3000, 30000, seed=2), False),
])
def test_row_pattern_dictionary(name, gen, full, ab, oracle):
    """Host logic of the index-free SpMV tiles (compress.c): rebuilding the
    column indices of every matched row from (row, pattern id, pattern table)
    gives back the CSR column indices exactly; stencil matrices match fully
    with a few dozen patterns, a power-law matrix mostly does not."""
    n, r, c, v = gen()
    rowptr, colidx, _ = oracle.full_csr(n, r, c, v)
    d = ab.patterns_host(rowptr, colidx, max_entries=4096)
    assert d["patptr"][0] == 0 and d["patptr"][-1] == len(d["patoff"]) <= 4096
    matched = 0
    for row in range(n):
        pid = int(d["patid"][row])
        if pid == 0xFFFF:
            continue
        matched += 1
        offs = d["patoff"][d["patptr"][pid]:d["patptr"][pid + 1]]
        assert np.array_equal(row + offs, colidx[rowptr[row]:rowptr[row + 1]])
    assert matched == d["nmatched"]
    if full:
        assert matched == n and d["npat"] <= 125
    else:
        assert matched < n
    # partitioned: interior rows keep their patterns, rows touching reordered border rows may not
    if name == "27pt":
        A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
        part = A.partition(2, _parts("slab", n, 2))[0].dsymv_init(0.0)
        no = part.c.nownedrows
        dp = ab.patterns_host(part.frowptr[:no + 1].copy(), part.fcolidx[:part.frowptr[no]].copy())
        assert dp["nmatched"] >= 0.5 * no


@pytest.mark.parametrize("kway", [False, True])
def test_metis_row_partition(kway, ab, oracle):
    """acgsymcsrmatrix_partition_rows (METIS from the CUDA toolkit's static
    archive): valid, balanced, low-cut, reproducible; and it feeds
    acgsymcsrmatrix_partition like any other row->part map."""
    N = 16
    n, r, c, v = mg.stencil3d_27pt(N)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
    try:
        parts, cut = A.partition_rows(8, kway=kway, seed=0)
    except ab.AcgError as e:
        if e.code == 19:
            pytest.skip("library built without METIS")
        raise
    assert parts.min() == 0 and parts.max() == 7
    sizes = np.bincount(parts, minlength=8)
    assert sizes.max() <= 1.05 * n / 8 + 1
    # edge cut as METIS reports it == edges of the pattern whose ends differ
    off = r != c
    assert cut == int(np.sum(parts[r[off]] != parts[c[off]]))
    # a 2x2x2 block split cuts 3 planes; METIS should be within 2x of that
    from acg_b200 import dist as abdist
    blk = abdist.block_partition(N, N, N, 2, 2, 2)
    assert cut <= 2 * int(np.sum(blk[r[off]] != blk[c[off]]))
    again, cut2 = A.partition_rows(8, kway=kway, seed=0)
    assert np.array_equal(parts, again) and cut == cut2
    one, cut1 = A.partition_rows(1)
    assert np.all(one == 0) and cut1 == 0
    subs = A.partition(8, parts)
    assert sum(m.c.nownedrows for m in subs) == n
    assert sum(m.c.ninterfacenzs for m in subs) == 2 * cut


@pytest.mark.parametrize("kind,dims,procs", [
    (27, (8, 8, 8), (2, 2, 2)),
    (27, (7, 9, 5), (2, 1, 3)),
    (27, (6, 6, 6), (1, 1, 2)),
    (7, (9, 7, 8), (3, 2, 2)),
    (7, (6, 6, 6), (1, 1, 1)),
])
def test_stencil_part_matches_partition(kind, dims, procs, ab):
    """acgb200_stencil_part (no global matrix) == partition of the global stencil
    matrix by the same block map, array for array."""
    from acg_b200 import dist as abdist
    nx, ny, nz = dims
    px, py, pz = procs
    n, r, c, v = (mg.stencil3d_27pt if kind == 27 else mg.laplace3d_7pt)(nx, ny, nz)
    A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
    nparts = px * py * pz
    want = A.partition(nparts, abdist.block_partition(nx, ny, nz, px, py, pz)) if nparts > 1 else [A]
    for p in range(nparts):
        m = ab.SymCsrMatrix.stencil_part(kind, nx, ny, nz, px, py, pz, p)
        w = want[p]
        for k in ("nrows", "nprows", "nnzs", "npnzs", "nownedrows", "ninnerrows", "nborderrows", "borderrowoffset",
                  "nghostrows", "ghostrowoffset", "ninnernzs", "ninterfacenzs"):
            assert getattr(m.c, k) == getattr(w.c, k), k
        if nparts > 1:
            assert np.array_equal(m.nzrows, w.nzrows)
        assert np.array_equal(m.rowptr, w.rowptr) and np.array_equal(m.colidx, w.colidx) and np.array_equal(m.a, w.a)
        hm, hw = m.halo(), w.halo()
        for k in hm:
            assert np.array_equal(hm[k], hw[k]), k
        m.dsymv_init(0.0); w.dsymv_init(0.0)
        for k in ("frowptr", "fcolidx", "fa", "orowptr", "ocolidx", "oa"):
            assert np.array_equal(getattr(m, k), getattr(w, k)), k
        m.free()


def test_stencil_part_large_is_cheap(ab):
    """One eighth of the 27-point 448^3 problem (BASELINE config 4) has the sizes
    SURVEY.md section 8 lists -- checked on a scaled-down box with the same formulas."""
    N = 64
    m = ab.SymCsrMatrix.stencil_part(27, N, N, N, 2, 2, 2, 0)
    h = N // 2
    assert m.c.nownedrows == h ** 3
    assert m.c.nghostrows == 3 * h * h + 3 * h + 1          # three faces, three edges, one corner
    assert m.c.nborderrows == h ** 3 - (h - 1) ** 3
    assert len(m.halo()["recipients"]) == 7


@pytest.mark.parametrize("name,gen", [("27pt", lambda: mg.stencil3d_27pt(10, 9, 11)), ("7pt", lambda: mg.laplace3d_7pt(12)),
                                      ("27pt-part", None)], ids=["27pt", "7pt", "27pt-part"])
def test_slices_and_tiles_arithmetic_emulated(name, gen, ab, oracle):
    """Emulation on the CPU of the index arithmetic of slices_fill_kernel + spmv_slices_kernel and of
    spmv_tiles_kernel, from exactly the arrays the device gets (slice descriptors, zero-padded offset
    table, pattern ids; tile descriptors with their aligned slice starts): every row is computed
    exactly once and y = A x."""
    if gen is None:
        from acg_b200 import dist as abdist
        n, r, c, v = mg.stencil3d_27pt(12)
        A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
        part = A.partition(2, abdist.block_partition(12, 12, 12, 1, 1, 2))[1].dsymv_init(0.0)
        no = part.c.nownedrows
        rowptr = part.frowptr[:no + 1].copy(); colidx = part.fcolidx[:rowptr[no]].copy(); vals = part.fa[:rowptr[no]].copy()
        nvec = no
    else:
        n, r, c, v = gen()
        rowptr, colidx, vals = oracle.full_csr(n, r, c, v)
        no = nvec = n
    plan = ab.spmv_plan_host(rowptr, colidx)          # tiles around the covered slices
    sp = ab.slices_host(rowptr, colidx)
    pat = ab.patterns_host(rowptr, colidx)
    assert sp["nslices"] > 0 and plan["slices"] == sp["nslices"] and plan["slice_rows"] == sp["rows"]
    x = np.random.default_rng(3).standard_normal(nvec)
    y = np.zeros(no)
    count = np.zeros(no, dtype=int)
    lpad, table = sp["lpad"], sp["spatoff"]
    # slices_fill_kernel: slice-major values, rows padded with zeros
    sval = np.full(32 * sp["blocks"], np.nan)
    for row0, _, L, vblk in sp["slices"]:
        for lane in range(32):
            kb, ln = rowptr[row0 + lane], rowptr[row0 + lane + 1] - rowptr[row0 + lane]
            for e in range(L):
                sval[32 * vblk + 32 * e + lane] = vals[kb + e] if e < ln else 0.0
    assert not np.isnan(sval).any()
    # spmv_slices_kernel: lane = row, column = row + table[pattern][slot]
    for row0, _, L, vblk in sp["slices"]:
        for lane in range(32):
            row = row0 + lane
            pid = int(sp["patid"][row])
            kb, ln = rowptr[row], rowptr[row + 1] - rowptr[row]
            offs = table[(0 if pid == 0xFFFF else pid) * lpad:][:lpad]
            acc = 0.0
            for e in range(L):
                # exception rows (not in the dictionary): the column comes from the index array, padded slots gather x[row]
                c = (colidx[kb + e] if e < ln else row) if pid == 0xFFFF else row + offs[e]
                acc += sval[32 * vblk + 32 * e + lane] * x[c]
            y[row] = acc
            count[row] += 1
    for row_begin, nrows, k_al, nnz_al in plan["tiles"]:
        # what spmv_issue stages: values / indices slice, row-pointer slice
        vals_s = np.concatenate([vals, np.zeros(16)])[k_al:k_al + nnz_al]
        cols_s = np.concatenate([colidx, np.zeros(16, colidx.dtype)])[k_al:k_al + nnz_al]
        row_al = row_begin & ~3
        nrp = (row_begin + nrows + 1 - row_al + 3) & ~3
        rptr_s = np.concatenate([rowptr, np.full(8, rowptr[-1])])[row_al:row_al + nrp]
        rp = rptr_s[row_begin & 3:]
        for lr in range(nrows):
            row = row_begin + lr
            kb, ke = rp[lr] - k_al, rp[lr + 1] - k_al
            assert 0 <= kb <= ke <= nnz_al
            y[row] = vals_s[kb:ke] @ x[cols_s[kb:ke]] if ke > kb else 0.0
            count[row] += 1
    assert (count == 1).all()
    want = np.zeros(no)
    for i in range(no):
        want[i] = vals[rowptr[i]:rowptr[i + 1]] @ x[colidx[rowptr[i]:rowptr[i + 1]]]
    assert np.allclose(y, want, rtol=1e-14, atol=1e-14)


_FS_HASH = r"""
import hashlib, sys
import numpy as np
import acg_b200 as ab
from acg_b200 import matgen as mg
m = hashlib.sha256()
n, r, c, v = mg.rmat_spd(2048, 20000, seed=5)
A = ab.SymCsrMatrix.init_real_double(n, r, c, v)
mats = [ab.SymCsrMatrix.init_real_double(n, c, r, v).dsymv_init(0.5)]           # lower-triangle input
mats += [p.dsymv_init(0.25) for p in A.partition(3, (np.arange(n) * 31 % 3).astype(np.int32))]
mats += [ab.SymCsrMatrix.stencil_part(27, 11, 12, 13, 2, 1, 2, q).dsymv_init(0.0) for q in range(4)]
for M in mats:
    for k in ("frowptr", "fcolidx", "fa", "orowptr", "ocolidx", "oa"):
        m.update(np.ascontiguousarray(getattr(M, k)).tobytes())
print(m.hexdigest())
"""


def test_full_storage_independent_of_thread_count():
    """The threaded expansion in acgsymcsrmatrix_dsymv_init and the threaded stencil
    generator give byte-identical arrays for any OMP_NUM_THREADS (the entry order
    inside a row fixes the summation order of the SpMV)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    seen = set()
    for nt in ("1", "3", "8"):
        env = dict(os.environ, OMP_NUM_THREADS=nt, PYTHONPATH=root)
        out = subprocess.run([sys.executable, "-c", _FS_HASH], env=env, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        seen.add(out.stdout.strip().splitlines()[-1])
    assert len(seen) == 1, seen


def test_comm_matrix(ab, tmp_path):
    """Communication matrix (cuda/acg-cuda.c:1713-1775): entry (p,q) = border values p
    sends q; symmetric for a structurally symmetric matrix, and equal to what q
    receives from p."""
    from acg_b200 import dist as abdist, mtxio
    n, r, c, v = mg.stencil3d_27pt(8)
    parts = ab.SymCsrMatrix.init_real_double(n, r, c, v).partition(8, abdist.block_partition(8, 8, 8, 2, 2, 2))
    M = np.stack([p.comm_matrix_row(8) for p in parts])
    assert np.array_equal(M, M.T) and np.all(np.diag(M) == 0)
    assert M[0, 1] == 16 and M[0, 3] == 4 and M[0, 7] == 1            # face, edge, corner of a 4^3 block
    for p, m in enumerate(parts):
        h = m.halo()
        for q, cnt in zip(h["senders"], h["recvcounts"]):
            assert M[q, p] == cnt
    path = str(tmp_path / "comm.mtx")
    mtxio.write_comm_matrix(path, M)
    lines = open(path).read().splitlines()
    assert lines[0] == "%%MatrixMarket matrix coordinate integer general" and lines[1] == f"8 8 {np.count_nonzero(M)}"
    assert "1 2 16" in lines                                           # 1-based in the file


def test_grid_partition_matches_python_helpers(ab):
    """acgb200_partition_rows_grid / acgb200_grid_factors (C) == dist.block_partition / grid_factors."""
    import ctypes as C
    from acg_b200 import dist as abdist
    L = ab.lib()
    for nparts in (1, 2, 3, 4, 6, 8, 12, 16, 27, 64):
        px, py, pz = C.c_int(), C.c_int(), C.c_int()
        L.acgb200_grid_factors(nparts, C.byref(px), C.byref(py), C.byref(pz))
        assert (px.value, py.value, pz.value) == abdist.grid_factors(nparts)
    for dims, procs in (((10, 9, 8), (2, 3, 1)), ((7, 7, 7), (3, 3, 3)), ((5, 4, 6), (1, 1, 1))):
        out = np.zeros(dims[0] * dims[1] * dims[2], np.int32)
        assert L.acgb200_partition_rows_grid(*dims, *procs, out) == 0
        assert np.array_equal(out, abdist.block_partition(*dims, *procs))
    assert L.acgb200_partition_rows_grid(4, 4, 4, 5, 1, 1, np.zeros(64, np.int32)) != 0


_RMAT_HASH = r"""
import hashlib
import numpy as np
import acg_b200 as ab
A = ab.SymCsrMatrix.rmat_spd(50000, 400000, seed=9)
m = hashlib.sha256()
for k in ("rowptr", "colidx", "a"):
    m.update(np.ascontiguousarray(getattr(A, k)).tobytes())
print(m.hexdigest())
"""


def test_rmat_generator(ab, oracle):
    """acgb200_rmat_spd (BASELINE config 5): packed upper triangle with sorted, duplicate-free
    rows; diagonal = degree + 1, off-diagonal -1 (every row of the full matrix sums to 1, so
    A is strictly diagonally dominant, hence SPD); heavy-tailed degrees; the same matrix for
    any thread count and a different one for another seed."""
    import subprocess
    import sys
    n = 50000
    A = ab.SymCsrMatrix.rmat_spd(n, 400000, seed=9)
    rp, ci, va = A.rowptr.copy(), A.colidx.copy(), A.a.copy()
    assert A.c.nprows == n and rp[-1] == len(ci)
    for i in (0, 1, 17, n - 1):
        row = ci[rp[i]:rp[i + 1]]
        assert row[0] == i and np.all(np.diff(row) > 0)          # diagonal first, then ascending, no duplicates
    A.dsymv_init(0.0)
    y = oracle.dsymv((A.frowptr.copy(), A.fcolidx.copy(), A.fa.copy()), 1.0, np.ones(n), 0.0, np.zeros(n))
    assert np.allclose(y, 1.0, rtol=0, atol=1e-9)
    deg = np.diff(A.frowptr) - 1
    assert deg.max() > 50 * deg.mean()                             # power law: a few very long rows
    assert 350000 < (len(ci) - n) <= 400000                        # few collisions, self-loops dropped
    B = ab.SymCsrMatrix.rmat_spd(n, 400000, seed=10)
    assert not np.array_equal(B.colidx, ci)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    seen = set()
    for nt in ("1", "5"):
        out = subprocess.run([sys.executable, "-c", _RMAT_HASH], env=dict(os.environ, OMP_NUM_THREADS=nt, PYTHONPATH=root),
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        seen.add(out.stdout.strip().splitlines()[-1])
    assert len(seen) == 1


def test_medium_rows_leave_the_tiles(ab):
    """Option spmv_medium = threshold: rows with threshold < length <= nnz_cap are planned for the
    warp-per-row kernel; tiles, medium rows and long rows partition the rows, tiles keep their
    bounds, and with the option off the plan is what it always was."""
    A = ab.SymCsrMatrix.rmat_spd(60000, 600000, seed=3).dsymv_init(0.0)
    lens = np.diff(A.frowptr)
    base = ab.spmv_plan_host(A.frowptr)
    assert base["nmedium"] == 0
    for thr in (64, 200):
        ab.set_option("spmv_medium", thr)
        try:
            pl = ab.spmv_plan_host(A.frowptr)
        finally:
            ab.set_option("spmv_medium", 0)
        cap = pl["nnz_cap"]
        assert pl["nmedium"] == int(((lens > thr) & (lens <= cap)).sum()) > 0
        assert np.array_equal(pl["longrows"], np.nonzero(lens > cap)[0])
        covered = np.zeros(len(lens), bool)
        for row_begin, nrows, k_al, nnz_al in pl["tiles"]:
            assert not covered[row_begin:row_begin + nrows].any()
            covered[row_begin:row_begin + nrows] = True
            assert lens[row_begin:row_begin + nrows].max() <= thr and nrows <= pl["rows_cap"]
            assert lens[row_begin:row_begin + nrows].sum() <= cap
        assert covered.sum() + pl["nmedium"] + len(pl["longrows"]) == len(lens)
        assert not covered[lens > thr].any()
    again = ab.spmv_plan_host(A.frowptr)
    assert np.array_equal(again["tiles"], base["tiles"])


def test_balanced_rows_partition(ab):
    """dist.balanced_rows_partition: contiguous blocks, every row assigned, nonzeros of the full
    matrix per part within a few percent of each other even for a power-law matrix."""
    from acg_b200 import dist as abdist
    A = ab.SymCsrMatrix.rmat_spd(40000, 400000, seed=6)
    rp = abdist.balanced_rows_partition(A, 5)
    assert rp.min() == 0 and rp.max() == 4 and np.all(np.diff(rp) >= 0)
    full = np.diff(A.dsymv_init(0.0).frowptr)
    per = np.array([full[rp == p].sum() for p in range(5)])
    assert per.sum() == A.c.fnpnzs
    assert per.max() <= 1.05 * per.mean() + full.max()
    rows = np.array([(rp == p).sum() for p in range(5)])
    assert rows.max() > 3 * rows.min()                     # equal work is far from equal row counts here
