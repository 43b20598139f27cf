import glob
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_device_count():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


# Order of a run: the parity core first (ABI, oracle pins, host structures, GPU parity through
# the C-ABI, multi-rank), then the callers around it (reference driver, example program, Python
# command line).  Within a file, tests that have not had their first run on hardware yet go last,
# so that under `-x` a problem in a new test cannot hide the verdict of the established ones.
_FILE_ORDER = ["test_abi.py", "test_oracle_pin.py", "test_host_structs.py", "test_mtxfile.py", "test_gpu_parity.py",
               "test_multirank.py", "test_reference_driver.py", "test_example_program.py", "test_driver_py.py"]
_FIRST_RUN_PENDING = ("test_spmv_ragged_rows", "test_device_and_plain_entry_points", "test_power_law_properties",
                      "test_stock_reference_gpu_solver_pins_the_oracle", "test_driver_manufactured_solution",
                      "acg-device", "test_public_blas1_building_blocks")


def _order_key(item):
    fname = os.path.basename(str(item.fspath))
    rank = _FILE_ORDER.index(fname) if fname in _FILE_ORDER else len(_FILE_ORDER)
    pending = any(tag in item.nodeid for tag in _FIRST_RUN_PENDING)
    return (rank, pending)


def pytest_collection_modifyitems(config, items):
    items.sort(key=_order_key)          # stable: definition order is kept inside each group
    # `-m gpu` on a box without a device must fail loudly, not skip silently:
    # only skip when the run did not ask for gpu tests explicitly.
    if _cuda_device_count() > 0:
        return
    if "gpu" in (config.getoption("-m") or "") and "not gpu" not in (config.getoption("-m") or ""):
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    from oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    from oracle import Ref, ref_available
    if not ref_available() and not os.path.isdir("/root/reference/acg"):
        pytest.skip("oracle/_ref not built and no reference tree")
    return Ref()


@pytest.fixture(scope="session")
def ab():
    if os.environ.get("ACGB200_TEST_LIB"):
        # development aid: run the host-structure tests against another build of the same sources
        # (e.g. tests/hostsim built with -fsanitize=address,undefined, under LD_PRELOAD=libasan.so)
        import acg_b200.api as api
        api._LIBPATH = os.environ["ACGB200_TEST_LIB"]
    import acg_b200
    acg_b200.lib()
    return acg_b200


def load_golden(path):
    z = np.load(path)
    return {k: z[k] for k in z.files}


def load_golden_json(name):
    with open(os.path.join(ROOT, "tests", "golden", "reference", name + ".json")) as f:
        return json.load(f)


def digest(a):
    """SHA-256 of an array's dtype, shape and bytes: what tests/golden/reference/*.json store in place
    of arrays that are compared bit for bit, to keep the fixtures small."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()
