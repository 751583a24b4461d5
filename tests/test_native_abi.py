"""CPU-side checks of the C-ABI library: it builds, loads, exports what include/trs_b200.h declares, and refuses to
run without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

from tests.conftest import ROOT
from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200 import build as trs_build


def declared_functions():
    text = open(os.path.join(ROOT, "include", "trs_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(trs_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    lib_path = trs_build.build()
    assert os.path.exists(lib_path)
    lib = nat.load()
    names = declared_functions()
    assert len(names) >= 14
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/trs_b200.h but not exported"
    assert sorted(nat.SYMBOLS) == names
    assert lib.trs_version() == 100


def test_struct_layouts_match_the_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "trs_b200.h"\n#include <stddef.h>\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(trs_preproc_params), sizeof(trs_spd_params), sizeof(trs_ctl_params), sizeof(trs_tensor), offsetof(trs_tensor, ndim), offsetof(trs_tensor, shape));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    a, b, c, t, t_ndim, t_shape = map(int, subprocess.check_output([str(exe)]).split())
    assert a == C.sizeof(nat.PreprocParams)
    assert b == C.sizeof(nat.SpdParams)
    assert c == C.sizeof(nat.CtlParams)
    assert t == C.sizeof(nat.Tensor) and t_ndim == nat.Tensor.ndim.offset and t_shape == nat.Tensor.shape.offset


def test_sass_is_sm100a_only():
    out = subprocess.check_output(["cuobjdump", "-lelf", nat.LIB_PATH]).decode()
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_gpu_means_loud_failure_not_fallback():
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that a machine with a GPU checks this too."""
    code = "import pytest\nfrom triton_racer_sim_b200 import _native as nat\nwith pytest.raises(nat.NativeError):\n    nat.Context(0)\n"
    run = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True,
                         timeout=300)
    assert run.returncode == 0, run.stderr[-2000:]


def test_product_does_not_touch_the_oracle():
    pkg = os.path.join(ROOT, "triton-racer-sim_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "trs_oracle" not in text, f
