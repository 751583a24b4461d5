"""CPU tier of the several-configuration preprocessing (trs_preprocess_configs): the bucketing of the frames by configuration
(csrc/loc_grid.h) and the slice every launch walks (csrc/preproc_list.h), built with g++ under the address and UB sanitizers through
tests/host_preproc_list_check.cpp, against numpy's stable argsort."""
import os
import subprocess

import numpy as np
import pytest

from tests.conftest import ROOT


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = tmp_path_factory.mktemp("plist") / "plist_check"
    build = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-fno-omit-frame-pointer", "-o", str(out), os.path.join(ROOT, "tests", "host_preproc_list_check.cpp")],
                           capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("no sanitizer runtime in this toolchain: " + build.stderr[-200:])
    return out


def _buckets(exe, tmp_path, cfg, k, max_blocks):
    cfg = np.ascontiguousarray(cfg, np.int32)
    src, dst = tmp_path / "in.bin", tmp_path / "out.bin"
    np.concatenate([np.array([len(cfg), k, max_blocks], np.int32), cfg]).tofile(src)
    run = subprocess.run([str(exe), str(src), str(dst)], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, (run.returncode, run.stderr[-2000:])
    raw, out, p = np.fromfile(dst, np.int32), [], 0
    for _ in range(k + 1):
        c = int(raw[p])
        out.append(raw[p + 1:p + 1 + c])
        p += 1 + c
    assert p == len(raw)
    return out


@pytest.mark.parametrize("n,k,max_blocks", [(0, 1, 296), (1, 1, 296), (1, 16, 296), (1000, 2, 1), (1000, 7, 7), (4096, 8, 296),
                                            (65_536, 16, 296), (70_001, 3, 296)])
def test_frame_buckets_are_a_stable_sort_by_configuration(exe, tmp_path, n, k, max_blocks):
    """Bucket c (c < K) lists the frames with configuration c in their batch order, bucket K the frames whose index is outside [0, K)
    (-1, K, INT32_MIN, INT32_MAX): together numpy's stable argsort of the buckets.  Random, sorted, all on one configuration, two
    configurations only (the others empty), and out-of-range indices."""
    rng = np.random.default_rng(n * 31 + k)
    cases = [rng.integers(0, k, n), np.sort(rng.integers(0, k, n)), np.full(n, k - 1), np.where(rng.random(n) < 0.5, 0, k - 1),
             rng.integers(-2, k + 2, n), rng.choice(np.array([-1, k, -2**31, 2**31 - 1, 0]), n)]
    for cfg in cases:
        cfg = cfg.astype(np.int32)
        got = _buckets(exe, tmp_path, cfg, k, max_blocks)
        bucket = np.where((cfg >= 0) & (cfg < k), cfg, k)
        order = np.argsort(bucket, kind="stable")
        assert np.array_equal(np.concatenate(got) if n else np.zeros(0, np.int32), order)
        for c in range(k + 1):
            assert np.array_equal(got[c], np.flatnonzero(bucket == c)), c
