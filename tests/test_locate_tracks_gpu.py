"""MultiTrackLocationTracker / trs_locate_tracks on the GPU: every car's (idx, segment) is bit for bit what the single-track LocationTracker of its
own track returns, and what the oracle returns, on every path (warp per car, bucketing + grid walk + warp per car for the cars put off, bucketing
+ thread-per-car scan), at sizes on both sides of the crossover."""
import numpy as np
import pytest
import torch

import oracle
from triton_racer_sim_b200 import LocationTracker, MultiTrackLocationTracker, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def tracks(golden_tracks):
    gen, mnt = golden_tracks["wp/generated_track"], golden_tracks["wp/mountain_track"]
    nan_line = gen.copy()
    nan_line[17, 1] = np.nan
    lines = [gen, mnt, gen + 1.0e6, mnt * 1e-3, gen * 1e3, synth.synthetic_track(10), nan_line]
    k = len(lines)
    return lines, np.linspace(-2.5, 3.0, k), np.linspace(7.25, 40.0, k)


def _cars(line, rng, n):
    """Near the line, anywhere around it (many rings: put off to the scan), on its points, on cell corners, around the 100 limit."""
    fin = line[np.isfinite(line).all(1)]
    lo, hi = fin.min(0), fin.max(0)
    ext = max(hi[0] - lo[0], hi[2] - lo[2])
    c = 2.0 ** np.ceil(np.log2(ext / 32.0))
    s = ext / 300
    m = n // 5
    return np.concatenate([
        fin[rng.integers(0, len(fin), m)] + rng.standard_normal((m, 3)) * np.array([1.5, 0.05, 1.5]) * s,
        np.stack([rng.uniform(lo[0] - 20 * s, hi[0] + 20 * s, m), rng.uniform(lo[1], hi[1] + 1e-9, m), rng.uniform(lo[2] - 20 * s, hi[2] + 20 * s, m)], 1),
        fin[rng.integers(0, len(fin), m)],
        np.stack([c * rng.integers(np.floor(lo[0] / c) - 2, np.floor(hi[0] / c) + 3, m), rng.uniform(lo[1], hi[1] + 1e-9, m),
                  c * rng.integers(np.floor(lo[2] / c) - 2, np.floor(hi[2] / c) + 3, m)], 1),
        np.stack([lo[0] - rng.uniform(95, 105, n - 4 * m), rng.uniform(lo[1], hi[1] + 1e-9, n - 4 * m), rng.uniform(lo[2], hi[2] + 1e-9, n - 4 * m)], 1)])


def _batch(lines, rng, n, assign, used=None):
    """n cars over the tracks in `used` (default all): `assign` = random | sorted | one; NaN / infinite cars on every track."""
    used = list(range(len(lines))) if used is None else used
    if assign == "one":
        trk = np.full(n, used[0])
    else:
        trk = np.array(used)[rng.integers(0, len(used), n)]
        if assign == "sorted":
            trk = np.sort(trk)
    xyz = np.empty((n, 3))
    for t in set(trk.tolist()):
        sel = np.nonzero(trk == t)[0]
        xyz[sel] = _cars(lines[t], rng, len(sel))[rng.permutation(len(sel))]
    special = np.array([[np.nan, 1, 1], [1, np.nan, 1], [1, 1, np.nan], [np.inf, 0, 0], [0, 0, -np.inf], [1e300, 1e300, 1e300]])
    if n >= 100:
        xyz[:6] = special
    return np.ascontiguousarray(xyz), np.ascontiguousarray(trk, np.int32)


def _check(mt, singles, lines, mn, mx, xyz, trk, what):
    idx, seg = mt.locate_device(torch.from_numpy(xyz).to(DEV), torch.from_numpy(trk).to(DEV))
    idx, seg = idx.cpu().numpy(), seg.cpu().numpy()
    k = len(lines)
    bad = (trk < 0) | (trk >= k)
    assert (idx[bad] == -1).all() and np.isnan(seg[bad]).all(), what
    for t in range(k):
        sel = np.nonzero(trk == t)[0]
        if not len(sel):
            continue
        si, ss = singles[t].locate_device(torch.from_numpy(xyz[sel]).to(DEV))
        with np.errstate(invalid="ignore", over="ignore"):
            oi, os_ = oracle.locate(lines[t], xyz[sel], mn[t], mx[t])
        assert np.array_equal(oi, si.cpu().numpy()) and np.array_equal(os_, ss.cpu().numpy()), (what, t, "single-track tracker vs oracle")
        assert np.array_equal(idx[sel], oi), f"{what} track {t}: {int((idx[sel] != oi).sum())} of {len(sel)} indices differ"
        assert np.array_equal(seg[sel].view(np.int64), os_.view(np.int64)), f"{what} track {t}: segments differ"


@pytest.mark.timeout(600)
@pytest.mark.parametrize("which", ["auto", "warp", "thread", "grid"])
def test_every_car_gets_its_own_tracks_answer(tracks, monkeypatch, which):
    lines, mn, mx = tracks
    if which != "auto":
        monkeypatch.setenv("TRS_LOCATE", which)
    mt = MultiTrackLocationTracker(lines, mn, mx, device=0)
    monkeypatch.delenv("TRS_LOCATE", raising=False)
    singles = [LocationTracker(line, mn[t], mx[t], device=0) for t, line in enumerate(lines)]
    cross = mt.ctx.sm_count * 256
    rng = np.random.default_rng(["auto", "warp", "thread", "grid"].index(which))
    cases = [(1, "random", None), (1000, "random", None), (cross - 1, "random", None), (cross, "random", None), (cross, "sorted", None),
             (cross + 777, "one", [3]), (cross, "random", [1, 5]), (cross, "random", [6, 2, 0]), (200_000, "random", None)]
    for n, assign, used in cases:
        xyz, trk = _batch(lines, rng, n, assign, used)
        _check(mt, singles, lines, mn, mx, xyz, trk, f"{which} n={n} {assign} {used}")
    # out-of-range indices on both sides of the crossover
    for n in (999, cross + 5):
        xyz, trk = _batch(lines, rng, n, "random")
        trk[rng.random(n) < 0.05] = -1
        trk[rng.random(n) < 0.05] = len(lines) + rng.integers(0, 1000)
        trk[:3] = [-2**31, 2**31 - 1, len(lines)]
        _check(mt, singles, lines, mn, mx, xyz, trk, f"{which} n={n} out of range")
    # n = 0
    idx, seg = mt.locate_device(torch.empty((0, 3), dtype=torch.float64, device=DEV), torch.empty(0, dtype=torch.int32, device=DEV))
    assert idx.shape == (0,) and seg.shape == (0,)
    mt.onShutdown()
    for s in singles:
        s.onShutdown()


def test_single_track_trackers_of_different_tracks_coexist(golden_tracks):
    """One LocationTracker per track in one process (the reference's way, and the baseline these tests compare with): a tracker with a larger grid
    table built before one with a smaller table still runs its grid walk (the kernel's shared-memory limit is not the last table's size)."""
    big, small = golden_tracks["wp/mountain_track"], golden_tracks["wp/generated_track"]
    trk_big = LocationTracker(big, device=0)
    trk_small = LocationTracker(small, device=0)
    n = trk_big.ctx.sm_count * 256 + 1000                        # the grid walk's side of the crossover
    for wp, trk in ((big, trk_big), (small, trk_small)):
        xyz = synth.car_states(wp, n, seed=12)[0]
        idx, seg = trk.locate_device(torch.from_numpy(xyz).to(DEV))
        want_i, want_s = oracle.locate(wp, xyz)
        assert np.array_equal(idx.cpu().numpy(), want_i) and np.array_equal(seg.cpu().numpy(), want_s)
    trk_big.onShutdown()
    trk_small.onShutdown()


@pytest.mark.parametrize("which", ["auto", "warp", "thread", "grid"])
def test_one_track_equals_trs_locate(golden_tracks, monkeypatch, which):
    """K = 1 gives trs_locate's answers exactly, on the reference's own states and on large batches."""
    if which != "auto":
        monkeypatch.setenv("TRS_LOCATE", which)
    for name in ("generated_track", "mountain_track"):
        wp = golden_tracks[f"wp/{name}"]
        mt = MultiTrackLocationTracker([wp], device=0)
        single = LocationTracker(wp, device=0)
        for xyz in (golden_tracks[f"xyz/{name}"], synth.car_states(wp, 100_000, seed=31)[0]):
            d = torch.from_numpy(np.ascontiguousarray(xyz)).to(DEV)
            i1, s1 = mt.locate_device(d, torch.zeros(len(xyz), dtype=torch.int32, device=DEV))
            i0, s0 = single.locate_device(d)
            assert torch.equal(i1, i0) and torch.equal(s1.view(torch.int64), s0.view(torch.int64)), (which, name, len(xyz))
        assert np.array_equal(mt.locate_device(torch.from_numpy(golden_tracks[f"xyz/{name}"]).to(DEV),
                                               torch.zeros(len(golden_tracks[f"xyz/{name}"]), dtype=torch.int32, device=DEV))[0].cpu().numpy(),
                              golden_tracks[f"idx/{name}"])
        mt.onShutdown()
        single.onShutdown()


def test_host_forms_and_argument_checks(tracks):
    lines, mn, mx = tracks
    mt = MultiTrackLocationTracker(lines, mn, mx, device=0)
    k = len(lines)
    rng = np.random.default_rng(3)
    xyz, trk = _batch(lines, rng, 500, "random")
    # numpy and python scalars in, the reference's types out
    seg, = mt.step(xyz[:, 0].copy(), xyz[:, 1].copy(), xyz[:, 2].copy(), trk)
    assert isinstance(seg, np.ndarray)
    for t in range(k):
        sel = trk == t
        with np.errstate(invalid="ignore", over="ignore"):
            assert np.array_equal(seg[sel], oracle.locate(lines[t], xyz[sel], mn[t], mx[t])[1], equal_nan=True), t
    s, = mt.step(float(xyz[7, 0]), float(xyz[7, 1]), float(xyz[7, 2]), int(trk[7]))
    assert isinstance(s, float) and s == oracle.locate(lines[trk[7]], xyz[7:8], mn[trk[7]], mx[trk[7]])[1][0]
    seg_t, = mt.step(*[torch.from_numpy(xyz[:, j].copy()).to(DEV) for j in range(3)], torch.from_numpy(trk).to(DEV))
    assert np.array_equal(seg_t.cpu().numpy(), seg, equal_nan=True)
    # out-of-range indices raise from the host forms
    for bad in (-1, k):
        with pytest.raises(ValueError):
            mt.step(xyz[:, 0].copy(), xyz[:, 1].copy(), xyz[:, 2].copy(), np.where(np.arange(500) == 9, bad, trk))
        with pytest.raises(ValueError):
            mt.step(1.0, 2.0, 3.0, bad)
    # the track tensor: dtype, device, shape
    d = torch.from_numpy(xyz).to(DEV)
    t32 = torch.from_numpy(trk).to(DEV)
    for t in (t32.to(torch.int64), t32.to(torch.float32), t32.cpu(), t32[:-1], t32[:, None], torch.cat([t32, t32])[::2]):
        with pytest.raises(ValueError):
            mt.locate_device(d, t)
    # track lists and segment ranges
    with pytest.raises(ValueError):
        MultiTrackLocationTracker([], device=0)
    with pytest.raises(ValueError):
        MultiTrackLocationTracker([lines[0]] * 257, device=0)
    with pytest.raises(ValueError):
        MultiTrackLocationTracker(lines[:2], [0, 1, 2], device=0)
    with pytest.raises(ValueError):
        MultiTrackLocationTracker([lines[0], np.zeros((0, 3))], device=0)
    # the context survived all of that
    _check(mt, [LocationTracker(line, mn[t], mx[t], device=0) for t, line in enumerate(lines)], lines, mn, mx, xyz, trk, "after the errors")
    mt.onShutdown()
    # 256 tracks are accepted
    many = MultiTrackLocationTracker([lines[0] + 1000.0 * i for i in range(256)], device=0)
    trk = rng.integers(0, 256, 60_000).astype(np.int32)
    xyz = lines[0][rng.integers(0, len(lines[0]), 60_000)] + 1000.0 * trk[:, None] + rng.standard_normal((60_000, 3))
    idx, _ = many.locate_device(torch.from_numpy(xyz).to(DEV), torch.from_numpy(trk).to(DEV))
    assert np.array_equal(idx.cpu().numpy(), oracle.locate(lines[0], xyz - 1000.0 * trk[:, None])[0])
    many.onShutdown()


@pytest.mark.parametrize("n", [5000, 120_000])
def test_queues_behind_the_callers_stream_and_captures_in_a_graph(tracks, n):
    """The call reads its inputs in the caller's stream order (inputs written behind a long spin on a side stream are seen), synchronises nothing
    and allocates nothing after the first call of a size: it can be captured in a CUDA graph and replayed on new inputs."""
    lines, mn, mx = tracks
    mt = MultiTrackLocationTracker(lines, mn, mx, device=0)
    rng = np.random.default_rng(n)
    a_xyz, a_trk = _batch(lines, rng, n, "random")
    b_xyz, b_trk = _batch(lines, rng, n, "sorted")
    xyz = torch.from_numpy(a_xyz).to(DEV)
    trk = torch.from_numpy(a_trk).to(DEV)
    want_a = mt.locate_device(xyz, trk)
    torch.cuda.synchronize()
    want_a = [t.clone() for t in want_a]
    b_xyz_dev, b_trk_dev = torch.from_numpy(b_xyz).to(DEV), torch.from_numpy(b_trk).to(DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                           # ~0.1 s of spinning, then the new inputs, then the call
        xyz.copy_(b_xyz_dev)
        trk.copy_(b_trk_dev)
        got_b = mt.locate_device(xyz, trk)
    side.synchronize()
    ref = [LocationTracker(line, mn[t], mx[t], device=0) for t, line in enumerate(lines)]
    _check(mt, ref, lines, mn, mx, b_xyz, b_trk, f"n={n} side stream")
    want_b = mt.locate_device(xyz, trk)
    torch.cuda.synchronize()
    assert torch.equal(got_b[0], want_b[0]) and torch.equal(got_b[1].view(torch.int64), want_b[1].view(torch.int64))
    # a graph of the call at this size, replayed on the first batch again
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gi, gs = mt.locate_device(xyz, trk)
    xyz.copy_(torch.from_numpy(a_xyz).to(DEV))
    trk.copy_(torch.from_numpy(a_trk).to(DEV))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(gi, want_a[0]) and torch.equal(gs.view(torch.int64), want_a[1].view(torch.int64))
    mt.onShutdown()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_leaves_the_callers_current_device_alone(tracks):
    lines, mn, mx = tracks
    torch.cuda.set_device(0)
    mt = MultiTrackLocationTracker(lines, mn, mx, device=1)
    assert torch.cuda.current_device() == 0
    rng = np.random.default_rng(4)
    for n in (2000, 80_000):
        xyz, trk = _batch(lines, rng, n, "random")
        idx, _ = mt.locate_device(torch.from_numpy(xyz).to("cuda:1"), torch.from_numpy(trk).to("cuda:1"))
        assert torch.cuda.current_device() == 0
        idx = idx.cpu().numpy()
        for t in range(len(lines)):
            sel = trk == t
            with np.errstate(invalid="ignore", over="ignore"):
                assert np.array_equal(idx[sel], oracle.locate(lines[t], xyz[sel])[0]), (n, t)
    mt.onShutdown()
    assert torch.cuda.current_device() == 0
