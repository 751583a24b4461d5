"""The default-range kernels fold each range's value bounds into its saturation thresholds (csrc/pixel_math.cuh sat_threshold_entry_folded, filled by
init_tables): a value outside the bounds gets a threshold no delta passes, and the value compares are not emitted.  Exhaustive proof on a host build
that the folded compare is exactly "saturation bound holds and value inside its bounds", for every value and delta."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.conftest import ROOT


@pytest.fixture(scope="module")
def fold_host(tmp_path_factory):
    out = tmp_path_factory.mktemp("fold") / "libfoldchk.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", str(out), os.path.join(ROOT, "tests", "host_sat_fold_check.cpp")])
    lib = C.CDLL(str(out))
    lib.fold_check.argtypes = [C.c_longlong, C.c_int, C.c_longlong, C.c_longlong]
    lib.fold_check.restype = C.c_longlong
    lib.fold_check_all_value_bounds.argtypes = [C.c_void_p, C.c_int]
    lib.fold_check_all_value_bounds.restype = C.c_longlong
    return lib


def test_folded_thresholds_every_saturation_bound(fold_host):
    """Every saturation bound from -2 to 300, both directions, with the default ranges' value bounds, with open ones, and with empty ones."""
    for vlo, vhi in ((24, 255), (23, 255), (0, 255), (-1, 256), (100, 180), (0, 0), (255, 255), (200, 100), (-(2 ** 31), 255), (0, -(2 ** 31))):
        for upper in (0, 1):
            for K in range(-2, 301):
                assert fold_host.fold_check(K, upper, vlo, vhi) == 0, (K, upper, vlo, vhi)


def test_folded_thresholds_every_value_bound(fold_host):
    """Every value bound from -1 to 256, lower and upper, against saturation bounds around the edges of the saturation range."""
    ks = np.array([-2, -1, 0, 1, 2, 12, 50, 99, 128, 200, 253, 254, 255, 256, 300], dtype=np.int64)
    assert fold_host.fold_check_all_value_bounds(ks.ctypes.data, len(ks)) == 0
