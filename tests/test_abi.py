"""The C-ABI boundary: library loads, exports what include/ declares, and its
struct layouts are the reference's (the same probe compiled against
include/acgb200/ prints what it printed compiled against the reference's
headers, tests/golden/reference/struct_layouts.txt)."""
import ctypes
import glob
import os
import re
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
%(includes)s
#define F(s, m) printf(#s "." #m " %%zu\n", offsetof(struct s, m))
int main(void) {
    printf("acgvector %%zu\n", sizeof(struct acgvector));
    printf("acgsymcsrmatrix %%zu\n", sizeof(struct acgsymcsrmatrix));
    printf("acggraph %%zu\n", sizeof(struct acggraph));
    printf("acgsolvercuda %%zu\n", sizeof(struct acgsolvercuda));
    F(acgvector, x); F(acgvector, idx); F(acgvector, num_ghost_nonzeros);
    F(acgsymcsrmatrix, nzrows); F(acgsymcsrmatrix, rowptr); F(acgsymcsrmatrix, nownedrows);
    F(acgsymcsrmatrix, borderrowoffset); F(acgsymcsrmatrix, ghostrowoffset); F(acgsymcsrmatrix, a);
    F(acgsymcsrmatrix, fnpnzs); F(acgsymcsrmatrix, onpnzs); F(acgsymcsrmatrix, frowptr); F(acgsymcsrmatrix, orowptr);
    F(acgsymcsrmatrix, fcolidx); F(acgsymcsrmatrix, ocolidx); F(acgsymcsrmatrix, fa); F(acgsymcsrmatrix, oa);
    F(acggraph, parentnodeidx); F(acggraph, srcnodeptr); F(acggraph, dstnodeidx); F(acggraph, bordernodeoffset);
    F(acggraph, ghostnodeoffset); F(acggraph, nneighbours); F(acggraph, neighbours);
    F(acgsolvercuda, halo); F(acgsolvercuda, haloexchange); F(acgsolvercuda, maxits); F(acgsolvercuda, bnrm2);
    F(acgsolvercuda, rnrm2); F(acgsolvercuda, d_r); F(acgsolvercuda, d_rowptr); F(acgsolvercuda, d_oa);
    F(acgsolvercuda, niterations); F(acgsolvercuda, nflops); F(acgsolvercuda, tsolve); F(acgsolvercuda, tgemv);
    F(acgsolvercuda, Bgemv); F(acgsolvercuda, nhalomsgs);
    printf("ACG_ERR_CUDA %%d\nACG_ERR_NOT_SUPPORTED %%d\nACG_ERR_NVSHMEM_NOT_SUPPORTED %%d\nACG_ERR_NOT_CONVERGED %%d\n",
           ACG_ERR_CUDA, ACG_ERR_NOT_SUPPORTED, ACG_ERR_NVSHMEM_NOT_SUPPORTED, ACG_ERR_NOT_CONVERGED);
    return 0;
}
"""


def _run_probe(includes, flags):
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "probe.c")
        open(src, "w").write(PROBE % dict(includes=includes))
        exe = os.path.join(d, "probe")
        subprocess.run(["/usr/bin/gcc", "-o", exe, src] + flags, check=True)
        return subprocess.run([exe], check=True, capture_output=True, text=True).stdout


def test_library_loads_and_exports_declared_symbols(ab):
    lib = ctypes.CDLL(os.path.join(ROOT, "acg_b200", "libacgb200.so"))
    declared = set()
    for h in glob.glob(os.path.join(ROOT, "include", "acgb200", "*.h")):
        text = open(h).read()
        declared |= set(re.findall(r"ACG_API\s+[\w\s\*]+?\b(acg\w+)\s*\(", text))
        declared |= set(re.findall(r"^const char \*(acgerrcodestr)\(", text, flags=re.M))
    declared -= {"acgcomm_init_mpi", "acgsolvercuda_fwritempi"}      # only with ACG_HAVE_MPI
    assert len(declared) > 45
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert set(ab.api.EXPORTS) <= declared | {"acgerrcodestr"}


def test_error_strings(ab):
    L = ab.lib()
    assert L.acgerrcodestr(0, 0) == b"success"
    assert b"not converged" in L.acgerrcodestr(39, 0)
    assert b"NVSHMEM" in L.acgerrcodestr(16, 0)


def test_struct_layouts_match_reference_headers():
    cuda_inc = "/usr/local/cuda/include"
    mine = _run_probe('#include "acgb200/cgcuda.h"\n#include "acgb200/error.h"',
                      ["-I" + os.path.join(ROOT, "include"), "-I" + cuda_inc])
    with open(os.path.join(ROOT, "tests", "golden", "reference", "struct_layouts.txt")) as f:
        theirs = f.read()
    assert mine == theirs


def test_binding_struct_sizes(ab):
    # api.lib() already asserts ctypes sizes == library sizes; make it explicit here
    L = ab.lib()
    assert L.acgb200_sizeof(b"acgsolvercuda") == ctypes.sizeof(ab.api.acgsolvercuda)
    assert L.acgb200_sizeof(b"acgsymcsrmatrix") == ctypes.sizeof(ab.api.acgsymcsrmatrix)
    assert L.acgb200_have_mpi() == 0


def test_reference_and_product_libraries_do_not_interpose(ab, ref):
    """libacgref.so (the reference) and libacgb200.so export the same names.  Both
    are linked -Bsymbolic and loaded RTLD_LOCAL, so a test process that holds both
    really compares two implementations (an earlier build silently bound the
    reference shim's calls to the product's symbols)."""
    mine, theirs = ab.lib(), ref.lib
    for name in ("acgsymcsrmatrix_init_real_double", "acgsymcsrmatrix_dsymv_init", "acgsymcsrmatrix_partition",
                 "acgvector_alloc", "acgerrcodestr"):
        a = ctypes.cast(getattr(mine, name), ctypes.c_void_p).value
        b = ctypes.cast(getattr(theirs, name), ctypes.c_void_p).value
        assert a != b, name
    theirs.acgerrcodestr.restype = ctypes.c_char_p
    # behavioural fingerprint: the two libraries word this message differently
    assert mine.acgerrcodestr(16, 0) != theirs.acgerrcodestr(16, 0)
    # and the reference shim reaches the reference's code: its init does not
    # bounds-check under NDEBUG, the product's does (ACG_ERR_INDEX_OUT_OF_BOUNDS)
    import numpy as np
    r = np.array([0], np.int32); c = np.array([5], np.int32); v = np.array([1.0])
    A = ab.api.acgsymcsrmatrix()
    assert mine.acgsymcsrmatrix_init_real_double(ctypes.byref(A), 2, 1, 0, r, c, v) == 31
