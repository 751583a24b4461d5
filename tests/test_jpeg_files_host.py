"""The JPEG file families of tests/jpeg_files.py through the host build of the decoder's shared source (jpeg_core.cuh + jpeg_host.h):
optimised Huffman tables, OpenCV's files, segments the parser skips, and the files it refuses.  Pillow's decode is the reference,
bit for bit; test_jpeg_files_gpu.py runs the same bytes through the kernels."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import jpeg_files as J
from tests.conftest import ROOT
from tests.test_jpeg_host import host_decode
from triton_racer_sim_b200 import synth


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("jpgfiles") / "libjpgcheck.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", str(out), os.path.join(ROOT, "tests", "host_jpeg_check.cpp")])
    lib = C.CDLL(str(out))
    lib.jpg_decode_rgb_host.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    return lib


@pytest.mark.parametrize("h,w", J.SIZES)
def test_every_accepted_family_matches_pillow(host_lib, tmp_path, h, w):
    files = J.accepted(tmp_path, h, w)
    assert len(files) == 21
    for name, _, data in files:
        rc, got = host_decode(host_lib, data, h, w)
        assert rc == 0, (name, rc)
        want = J.pil_decode(data)
        assert np.array_equal(got, want), (name, int((got != want).sum()))


def test_optimised_tables_are_not_annex_k(tmp_path):
    """The families really are what they claim: optimised files carry Huffman tables of their own (a one-symbol table at 1x1), the
    ICC profile spans two APP2 segments and the edits add the segments they name."""
    default = J.pil_file(tmp_path, synth.frame_pool(2, 120, 160, seed=1)[1])
    for h, w in ((1, 1), (120, 160)):
        fam = {name: data for name, _, data in J.accepted(tmp_path, h, w)}
        assert J.table_bytes(fam["pil-opt-420-q75"], (0xDB,)) == J.table_bytes(default, (0xDB,))        # quality 75 ...
        assert J.table_bytes(fam["pil-opt-420-q75"], (0xC4,)) != J.table_bytes(default, (0xC4,))        # ... other Huffman tables
        if (h, w) == (1, 1):
            assert 1 in J.huffman_symbol_counts(fam["pil-opt-420-q75"]) and 1 in J.huffman_symbol_counts(fam["cv-opt"])
        assert sum(m == 0xE2 for _, m, _ in J.segments(fam["icc"])) == 2
        assert sum(m == 0xFE for _, m, _ in J.segments(fam["comment"])) == 1
        assert sum(m == 0xDD for _, m, _ in J.segments(fam["dri-0"])) == 1


@pytest.mark.parametrize("h,w", [(1, 1), (7, 9), (120, 160), (240, 320)])
def test_refused_families(host_lib, tmp_path, h, w):
    for name, data in J.refused(tmp_path, synth.frame_pool(2, h, w, seed=h + w)[1]):
        assert host_decode(host_lib, data, h, w)[0] == 111, name                 # 100 + JPG_E_UNSUPPORTED
