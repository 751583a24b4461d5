"""CPU tier of the multi-track nearest waypoint (trs_set_tracks / trs_locate_tracks): csrc/loc_grid.h built with g++ through
tests/host_locate_tracks_check.cpp.  The per-track tables and the bucketing are checked against numpy, the whole large-batch path (bucketing,
slices of the walk split at track boundaries, the scan of the cars put off) against the oracle per track, and a fuzz of the same path runs under
the sanitizers."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from tests.conftest import ROOT
from triton_racer_sim_b200 import synth

I64P = C.POINTER(C.c_longlong)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("loct") / "libloctchk.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", str(out), os.path.join(ROOT, "tests", "host_locate_tracks_check.cpp")])
    lib = C.CDLL(str(out))
    lib.tracks_build_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.tracks_bucket_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.locate_tracks_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def _cat(tracks):
    return np.ascontiguousarray(np.concatenate(tracks), np.float64), np.array([len(t) for t in tracks], np.int32)


def _tracks(golden_tracks):
    gen, mnt = golden_tracks["wp/generated_track"], golden_tracks["wp/mountain_track"]
    nan_line = gen.copy()
    nan_line[17, 1] = np.nan
    return [gen, mnt, gen + 1.0e6, mnt * 1e-3, gen * 1e3, synth.synthetic_track(10), nan_line]


def _first_occurrences(wp):
    """Indices of the points the reference's strict `<` can select: first occurrences by value (a point with a NaN is always kept)."""
    seen, keep = set(), []
    for i, p in enumerate(wp):
        key = tuple(float(v) + 0.0 for v in p)              # -0.0 == 0.0
        if any(v != v for v in key):
            keep.append(i)
        elif key not in seen:
            seen.add(key)
            keep.append(i)
    return np.array(keep)


def test_per_track_tables_match_numpy(lib, golden_tracks):
    """Every track's distinct points, in order of first occurrence with their original index, one after the other; a grid table for each track
    that can have one and none for a 10-point line or a line with a NaN; the grid tables hold the same points in cell order."""
    tracks = _tracks(golden_tracks)
    wp, n_wp = _cat(tracks)
    k = len(tracks)
    mn, mx = np.zeros(k), np.full(k, 10.0)
    info, sizes = np.zeros((k, 7), np.int64), np.zeros(4, np.int64)
    assert lib.tracks_build_host(wp.ctypes.data, n_wp.ctypes.data, k, mn.ctypes.data, mx.ctypes.data, info.ctypes.data, sizes.ctypes.data, None, None) == 0
    scan, grid = np.zeros((sizes[0], 4)), np.zeros((max(sizes[1], 1), 4))
    assert lib.tracks_build_host(wp.ctypes.data, n_wp.ctypes.data, k, mn.ctypes.data, mx.ctypes.data, info.ctypes.data, sizes.ctypes.data,
                                 scan.ctypes.data, grid.ctypes.data) == 0
    scan_off, grid_off, cell_off = 0, 0, 0
    for t, line in enumerate(tracks):
        keep = _first_occurrences(line)
        n_u = len(keep)
        assert info[t, 0] == n_u and info[t, 1] == scan_off, t
        want = np.concatenate([line[keep], keep[:, None].astype(np.float64)], 1)
        assert np.array_equal(scan[scan_off:scan_off + n_u], want, equal_nan=True), t
        has_grid = len(line) >= 64 and np.isfinite(line).all()
        assert (info[t, 2] >= 0) == has_grid, t
        if has_grid:
            assert info[t, 2] == grid_off and info[t, 3] == cell_off and info[t, 4] == info[t, 5] * info[t, 6], t
            g = grid[grid_off:grid_off + n_u]                   # (x, z, y, index) in cell order: a permutation of the distinct points
            assert np.array_equal(g[np.argsort(g[:, 3])], want[:, [0, 2, 1, 3]]), t
            grid_off += n_u
            cell_off += info[t, 4] + 1
        scan_off += n_u
    assert sizes[0] == scan_off and sizes[1] == grid_off and sizes[2] == cell_off
    assert list(info[:2, 0]) == [917, 1260]                     # the shipped lines' distinct points (DESIGN §4.6)


@pytest.mark.parametrize("n,k,max_blocks", [(1, 1, 4), (1000, 3, 1), (1000, 3, 7), (5000, 8, 296), (70_001, 256, 296), (4096, 2, 16)])
def test_bucketing_is_a_stable_sort_by_track(lib, n, k, max_blocks):
    """The histogram / scan / scatter passes give numpy's stable argsort of the buckets (track, or K for an index outside [0, K)), and the
    bucket starts; with tracks that have no cars, all cars on one track, and random, sorted and out-of-range indices."""
    rng = np.random.default_rng(n + k)
    cases = [rng.integers(0, k, n), np.sort(rng.integers(0, k, n)), np.full(n, k - 1), rng.integers(-2, k + 2, n),
             np.where(rng.random(n) < 0.5, 0, k - 1), rng.integers(-2**31, 2**31 - 1, n)]
    for trk in cases:
        trk = np.ascontiguousarray(trk, np.int32)
        perm, start = np.full(n, -7, np.int32), np.zeros(k + 2, np.int32)
        lib.tracks_bucket_host(trk.ctypes.data, n, k, max_blocks, 256, perm.ctypes.data, start.ctypes.data)
        bucket = np.where((trk >= 0) & (trk < k), trk, k)
        assert np.array_equal(perm, np.argsort(bucket, kind="stable"))
        assert np.array_equal(start, np.concatenate([[0], np.cumsum(np.bincount(bucket, minlength=k + 1))]))


def _locate(lib, tracks, mn, mx, xyz, trk, ctas):
    wp, n_wp = _cat(tracks)
    k, n = len(tracks), len(xyz)
    mn, mx = np.ascontiguousarray(mn, np.float64), np.ascontiguousarray(mx, np.float64)
    xyz, trk = np.ascontiguousarray(xyz, np.float64), np.ascontiguousarray(trk, np.int32)
    idx, seg, stats = np.zeros(n, np.int32), np.zeros(n), np.zeros(3, np.int64)
    assert lib.locate_tracks_host(wp.ctypes.data, n_wp.ctypes.data, k, mn.ctypes.data, mx.ctypes.data, xyz.ctypes.data, trk.ctypes.data, n, ctas,
                                  idx.ctypes.data, seg.ctypes.data, stats.ctypes.data) == 0
    return idx, seg, stats


def test_multi_track_walk_matches_the_oracle_per_track(lib, golden_tracks):
    """Both shipped lines, shifted and scaled copies, a 10-point line and a line with a NaN point in one batch; cars near each line, anywhere
    around it, NaN / infinite, and out-of-range indices; walked by 1 to 296 CTAs, so slices start and end inside tracks."""
    tracks = _tracks(golden_tracks)
    k = len(tracks)
    mn, mx = np.linspace(-2.5, 3.0, k), np.linspace(7.25, 40.0, k)
    rng = np.random.default_rng(5)
    xyz, trk = [], []
    for t, line in enumerate(tracks):
        fin = line[np.isfinite(line).all(1)]
        lo, hi = fin.min(0), fin.max(0)
        ext = max(hi[0] - lo[0], hi[2] - lo[2], 1e-9)
        m = 1500
        near = fin[rng.integers(0, len(fin), m)] + rng.standard_normal((m, 3)) * np.array([1.5, 0.05, 1.5]) * ext / 300
        around = np.stack([rng.uniform(lo[0] - ext / 5, hi[0] + ext / 5, m), rng.uniform(lo[1], hi[1] + 1e-9, m),
                           rng.uniform(lo[2] - ext / 5, hi[2] + ext / 5, m)], 1)
        xyz += [near, around]
        trk += [np.full(2 * m, t)]
    xyz.append(np.array([[np.nan, 1, 1], [1, np.nan, 1], [np.inf, 0, 0], [0, 0, -np.inf], [1e300, 0, 1e300]] * k))
    trk.append(np.repeat(np.arange(k), 5).reshape(k, 5).T.reshape(-1))
    xyz, trk = np.concatenate(xyz), np.concatenate(trk).astype(np.int32)
    perm = rng.permutation(len(xyz))
    xyz, trk = xyz[perm], trk[perm]
    trk[rng.random(len(trk)) < 0.02] = -1
    trk[rng.random(len(trk)) < 0.02] = k
    for ctas in (1, 5, 296):
        idx, seg, stats = _locate(lib, tracks, mn, mx, xyz, trk, ctas)
        assert stats[1] == 5 and stats[0] > 0                    # five tracks with a grid; cars put off to the scan
        bad = (trk < 0) | (trk >= k)
        assert (idx[bad] == -1).all() and np.isnan(seg[bad]).all()
        for t, line in enumerate(tracks):
            sel = trk == t
            with np.errstate(invalid="ignore", over="ignore"):
                want_i, want_s = oracle.locate(line, xyz[sel], mn[t], mx[t])
            assert np.array_equal(idx[sel], want_i), (ctas, t, int((idx[sel] != want_i).sum()))
            assert np.array_equal(seg[sel], want_s), (ctas, t)


def test_multi_track_fuzz_under_the_sanitizers(tmp_path):
    """tests/host_locate_tracks_fuzz.cpp with -fsanitize=address,undefined: 200 random batches of 1-9 centre lines x 600 cars against the
    reference's loop per track — exact indices and segments, no table, cell or bucket index out of bounds."""
    exe = tmp_path / "loct_fuzz"
    build = subprocess.run(["g++", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer", "-o",
                            str(exe), os.path.join(ROOT, "tests", "host_locate_tracks_fuzz.cpp")], capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("no sanitizer runtime in this toolchain: " + build.stderr[-200:])
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0 and run.stdout.strip() == "ok 120000 cars", (run.stdout[-500:], run.stderr[-2000:])
