"""Parity of the CUDA path (through the C ABI / Component classes) against the oracle and the reference's golden
vectors.  Bit-exact for uint8 frames, masks and waypoint indices; float32 normalised tensors are compared exactly
too (they are correctly rounded divisions); speed-control outputs within 1e-5 relative (north_star tolerance)."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from tests.helpers import cfg_for, golden_pairs, speed_cases
from triton_racer_sim_b200 import FrameNormalise, ImgPreprocessing, LocationTracker, SpeedControl, synth
from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200.config import full_house_config

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5          # BASELINE.json north_star: "within 1e-5 relative for normalised float tensors and PID outputs"


def run_device(cfg, frames, want_f32=True):
    comp = ImgPreprocessing(cfg, device=0, normalised_key='cam/normalised_img' if want_f32 else None)
    u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV))
    torch.cuda.synchronize()
    comp.onShutdown()
    return u8.cpu().numpy(), (f32.cpu().numpy() if f32 is not None else None)


def describe(got, want):
    bad = np.argwhere(got != want)
    return f"{len(bad)} of {got.size} differ; first at {bad[:5].tolist()}"


def test_library_is_the_cuda_one():
    assert torch.cuda.is_available()
    ctx = nat.Context(0)
    assert ctx.cc[0] >= 10 and ctx.sm_count > 0
    ctx.close()


def test_golden_images_device_path(golden_images):
    count = 0
    for sname, cname, cfg, frames, expected in golden_pairs(golden_images):
        got, f32 = run_device(cfg, frames)
        assert np.array_equal(got, expected), f"{sname}/{cname}: {describe(got, expected)}"
        assert np.array_equal(f32, oracle.normalise(expected)), f"{sname}/{cname} f32"
        count += 1
    assert count >= 30


def test_golden_images_host_path(golden_images):
    for sname, cname, cfg, frames, expected in golden_pairs(golden_images):
        if cname not in ("full_house", "exotic"):
            continue
        comp = ImgPreprocessing(cfg, device=0, normalised_key='cam/normalised_img', collect_stats=True)
        u8, f32 = comp.step(frames)
        assert np.array_equal(u8, expected), f"{sname}/{cname}: {describe(u8, expected)}"
        assert np.array_equal(f32, oracle.normalise(expected))
        assert comp.last_stats["frames"] == frames.shape[0]
        comp.onShutdown()


def test_canny_stage_taps_match_oracle(golden_images):
    """Intermediate planes (selected-channel magnitude, NMS map) for single frames, incl. odd sizes."""
    cfg = full_house_config()
    comp = ImgPreprocessing(cfg, device=0)
    for sname in ("f120", "f240", "odd_7x9", "odd_33x50", "odd_121x163", "odd_64x96"):
        for img in golden_images[f"in/{sname}"][:4]:
            h, w, _ = img.shape
            _, mag, mp = oracle.canny3(img, 60, 100, taps=True)
            d_img = torch.from_numpy(img).to(DEV)
            d_mag = torch.zeros((h, w), dtype=torch.int16, device=DEV)
            d_map = torch.zeros((h, w), dtype=torch.uint8, device=DEV)
            nat.check(comp.ctx.lib.trs_debug_canny_stages(comp.ctx.handle, C.c_void_p(d_img.data_ptr()), h, w, C.c_void_p(d_mag.data_ptr()),
                                                          C.c_void_p(d_map.data_ptr()), None), "debug")
            torch.cuda.synchronize()
            got_mag = d_mag.cpu().numpy().view(np.uint16)
            assert np.array_equal(got_mag, mag), f"{sname} mag: {describe(got_mag, mag)}"
            assert np.array_equal(d_map.cpu().numpy(), mp), f"{sname} map: {describe(d_map.cpu().numpy(), mp)}"
    comp.onShutdown()


@pytest.mark.parametrize("h,w,n", [(120, 160, 96), (240, 320, 24), (17, 23, 5), (41, 64, 7), (119, 8, 3), (1, 40, 2), (40, 1, 2),
                                   (480, 640, 3), (130, 2000, 2),
                                   # banded kernel: uneven last band, eight segments per band (w = 160), nine warps (w = 96), two bands only
                                   (241, 320, 5), (480, 160, 5), (300, 96, 5), (150, 320, 5), (3, 320, 2), (1000, 32, 3)])
def test_fresh_frames_against_oracle(h, w, n):
    frames = synth.frame_pool(n, h, w, seed=1000 + h + w)
    for over in (dict(), dict(preprocessing_dynamic_brightness_enabled=True, preprocessing_contrast_enhancement_ratio=1.6,
                              preprocessing_contrast_enhancement_offset=90, preprocessing_edge_detection_threshold_a=33.3,
                              preprocessing_edge_detection_threshold_b=210)):
        cfg = full_house_config(**over)
        want = oracle.process_batch(frames, cfg)
        got, f32 = run_device(cfg, frames)
        assert np.array_equal(got, want), describe(got, want)
        assert np.array_equal(f32, oracle.normalise(want))


@pytest.mark.parametrize("h,w,n", [(240, 320, 16), (120, 160, 32), (480, 160, 4), (200, 96, 6)])
def test_every_golden_configuration_on_fresh_frames(golden_images, h, w, n):
    """All seven reference-generated configurations (colour only, edge only, no filter, dynamic brightness + contrast, three ranges with
    repeated destination channels, ...) on fresh frames at the second resolution and at sizes that need row bands: the banded kernel applies
    the brightness / contrast table per band (the dynamic one from rows 40..118 of the frame in global memory) and re-reads the frame for
    channels that keep the adjusted pixel; the no-filter configurations take the streaming kernel."""
    from tests.helpers import image_cases
    q = max(1, n // 4)
    frames = synth.expand_numpy(synth.frame_pool(q, h, w, seed=77 + h + w), n, start=13 * q)      # four brightness shifts of q frames each
    for cname, over in image_cases(golden_images).items():
        cfg = cfg_for(over)
        want = oracle.process_batch(frames, cfg)
        got, f32 = run_device(cfg, frames)
        assert np.array_equal(got, want), f"{cname} {h}x{w}: {describe(got, want)}"
        assert np.array_equal(f32, oracle.normalise(want)), f"{cname} {h}x{w} f32"


def test_adversarial_hysteresis_chains():
    """Serpentine weak chains hanging off a single strong pixel: the worst case for iterative flood fill."""
    h, w = 120, 160
    frames = []
    for period in (4, 6, 10):
        img = np.full((h, w, 3), 90, np.uint8)
        for y in range(4, h - 4, period):
            img[y, 4:w - 4] = 112
            x = (w - 5) if (y // period) % 2 == 0 else 4
            img[y:y + period, x] = 112
        img[4, 4:8] = 255
        frames.append(img)
    frames = np.stack(frames)
    cfg = full_house_config(preprocessing_edge_detection_threshold_a=30, preprocessing_edge_detection_threshold_b=200)
    want = oracle.process_batch(frames, cfg)
    got, _ = run_device(cfg, frames, want_f32=False)
    assert np.array_equal(got, want), describe(got, want)
    assert want[..., 2].sum() > 0


def test_component_drop_in_single_frame_and_none():
    cfg = full_house_config()
    comp = ImgPreprocessing(cfg, device=0)
    assert comp.step_inputs == ['cam/img'] and comp.step_outputs == ['cam/processed_img']
    assert comp.getName() == 'Image Preprocessing'
    assert comp.step(None) == (None,)
    img = synth.frame_pool(1, 120, 160, seed=77)[0]
    keep = img.copy()
    out, = comp.step(img)
    assert isinstance(out, np.ndarray) and out.shape == (120, 160, 3) and out.dtype == np.uint8
    assert np.array_equal(img, keep)                                  # the caller's frame is never modified
    assert np.array_equal(out, oracle.process_frame(img, cfg))
    t_out, = comp.step(torch.from_numpy(img).to(DEV))
    assert t_out.is_cuda and np.array_equal(t_out.cpu().numpy(), out)
    comp.onShutdown()
    lag = ImgPreprocessing(cfg, device=0, emulate_latency=True)       # the reference's one-tick lag (img_preprocessing.py:18-21)
    assert lag.step(img) == (None,)
    second, = lag.step(np.zeros_like(img))
    assert np.array_equal(second, out)
    lag.onShutdown()


def test_bad_arguments_raise():
    with pytest.raises(ValueError):
        ImgPreprocessing(full_house_config(preprocessing_color_filter_destination_channels=[0, 5]), device=0)
    with pytest.raises(AssertionError):
        ImgPreprocessing(full_house_config(preprocessing_color_filter_destination_channels=[0]), device=0)
    comp = ImgPreprocessing(full_house_config(), device=0)
    with pytest.raises(ValueError):
        comp.process_device(torch.zeros((2, 8, 8, 4), dtype=torch.uint8, device=DEV))
    empty_u8, _ = comp.process_device(torch.zeros((0, 120, 160, 3), dtype=torch.uint8, device=DEV))
    assert empty_u8.shape[0] == 0
    comp.onShutdown()
    with pytest.raises(FileNotFoundError):
        LocationTracker('/nonexistent/track.json', device=0)


def oracle_counts(frames, cfg, want):
    """The counters trs_preprocess must report for `frames` (TRS_STAT_*), from the oracle.  A colour range whose output channel a
    later range or the edge layer overwrites never reaches the output and counts 0; strong / cand count the NMS map's 2s and
    non-zeros, taken on the frame after its brightness / contrast table; the ROI sum covers rows 40..118 when the table is dynamic."""
    p = oracle.params_from_cfg(cfg)
    c = dict(frames=len(frames), mask0=0, mask1=0, mask2=0, mask3=0, edge=0, strong=0, cand=0, roi_sum=0)
    layers = [(f"mask{i}", p.color_dest[i] % 3) for i in range(p.n_hsv if p.color_filter_enabled else 0)]
    layers += [("edge", p.edge_dest % 3)] if p.edge_enabled else []
    for k, (name, ch) in enumerate(layers):
        if all(later != ch for _, later in layers[k + 1:]):
            c[name] = int((want[..., ch] == 255).sum())
    if p.edge_enabled:
        for img in frames:
            lut, _ = oracle.brightness_lut(img, cfg)
            _, _, mp = oracle.canny3(lut[img], p.canny_a, p.canny_b, taps=True)
            c["strong"] += int((mp == 2).sum())
            c["cand"] += int((mp >= 1).sum())
    if p.dynamic_brightness:
        c["roi_sum"] = int(frames[:, 40:119].astype(np.uint64).sum())
    return c


# (switch, h, w, configuration, frames, CTAs per SM at most): every kernel launch_preprocess picks (trs_api.cu:302-437), with at least
# five frames per CTA.  The grid is SMs x CTAs per SM: two for the resident / banded / store-warp kernels (trs_api.cu:374) and for
# k_preprocess_bsw (384 threads at <= 80 registers: 65,536 registers hold two), eight for k_adjust_stream (trs_api.cu:308), and at most
# 2,048 / 512 threads = four for the generic kernel (trs_api.cu:432).
STAT_KERNELS = {
    "store_warp_120x160": (None, 120, 160, "full_house", 1500, 2),
    "banded_store_warp_240x320": (None, 240, 320, "full_house", 1500, 2),
    "resident_no_store_warp": ("TRS_NO_STORE_WARP", 120, 160, "full_house", 1500, 2),
    "banded_no_store_warp": ("TRS_NO_STORE_WARP", 240, 320, "full_house", 1500, 2),
    "table_dyn_contrast": (None, 120, 160, "dyn_contrast", 1500, 2),
    "table_exotic": (None, 120, 160, "exotic", 1500, 2),
    "no_filter_adjust_stream": (None, 120, 160, "adjust_dynamic", 5920, 8),
    "generic_122x166": ("TRS_FORCE_GENERIC", 122, 166, "full_house", 2960, 4),
    "generic_7x9": (None, 7, 9, "exotic", 2960, 4),
}


@pytest.mark.timeout(600)
def test_statistics_match_oracle_counts(golden_images, monkeypatch):
    """Every counter but the sweeps and the timers against the oracle, for every kernel: the kernels count strong and candidate
    pixels in different places (before the hysteresis in the banded store-warp kernel, from the finished planes in the store
    warps, in the suppression loop of the generic kernel).  All kernels are checked before the test fails, and the message names
    each one that disagrees."""
    from tests.helpers import image_cases
    ctx = nat.Context(0)
    sms = ctx.sm_count
    ctx.close()
    cases = image_cases(golden_images)
    extra = dict(adjust_dynamic=dict(preprocessing_dynamic_brightness_enabled=True, preprocessing_contrast_enhancement_ratio=1.25,
                                     preprocessing_brightness_baseline=380))
    failures = []
    for name, (env, h, w, cname, n, per_sm) in STAT_KERNELS.items():
        assert n >= 5 * sms * per_sm, f"{name}: {n} frames on up to {sms * per_sm} CTAs is fewer than five frames per CTA"
        for switch in ("TRS_NO_STORE_WARP", "TRS_FORCE_GENERIC"):
            monkeypatch.delenv(switch, raising=False)
        if env:
            monkeypatch.setenv(env, "1")                     # read when the component's context is created
        cfg = cfg_for(cases[cname] if cname in cases else extra[cname])
        frames = synth.expand_numpy(synth.frame_pool(64, h, w, seed=5), n, start=11)
        want = oracle.process_batch(frames, cfg)
        comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
        got, _ = comp.process_device(torch.from_numpy(frames).to(DEV), want_f32=False)
        st = comp.stats()
        comp.onShutdown()
        got = got.cpu().numpy()
        if not np.array_equal(got, want):
            failures.append(f"{name}: output {describe(got, want)}")
            continue
        want_st = oracle_counts(frames, cfg, want)
        bad = [f"{k} {st[k]} != {v}" for k, v in want_st.items() if st[k] != v]
        if bad:
            failures.append(f"{name}: " + ", ".join(bad))
    assert not failures, "\n".join(failures)


def test_normalise_and_crop_resize():
    frames = synth.frame_pool(6, 240, 320, seed=3)
    d = torch.from_numpy(frames).to(DEV)
    ident = FrameNormalise(device=0)
    out, = ident.step(d)
    assert np.array_equal(out.cpu().numpy(), oracle.normalise(frames))
    all_bytes = np.arange(256, dtype=np.uint8).repeat(3 * 5).reshape(1, 5, 256, 3)      # every byte value, true division
    assert np.array_equal(ident.step(all_bytes)[0], oracle.normalise(all_bytes))
    ident.onShutdown()
    cam = FrameNormalise(device=0, out_hw=(120, 160))                                   # camera.py:36 case: 320x240 -> 160x120
    u8_want, f32_want = oracle.crop_resize(frames, (0, 240, 0, 320), (120, 160))
    f32, u8 = cam.normalise_device(d, want_u8=True)
    assert np.array_equal(u8.cpu().numpy(), u8_want) and np.array_equal(f32.cpu().numpy(), f32_want)
    assert np.array_equal(u8_want, frames[:, ::2, ::2])
    cam.onShutdown()
    for roi, out_hw in (((40, 119, 0, 320), None), ((10, 230, 17, 301), (77, 131)), ((0, 240, 0, 320), (300, 333)), ((3, 200, 8, 311), (300, 332)),
                        ((0, 240, 0, 320), (60, 80))):
        comp = FrameNormalise(device=0, roi=roi, out_hw=out_hw)
        ho, wo = out_hw if out_hw else (roi[1] - roi[0], roi[3] - roi[2])
        u8_want, f32_want = oracle.crop_resize(frames, roi, (ho, wo))
        f32, u8 = comp.normalise_device(d, want_u8=True)
        assert np.array_equal(u8.cpu().numpy(), u8_want) and np.array_equal(f32.cpu().numpy(), f32_want)
        comp.onShutdown()
    # source rows that are not a multiple of 16 bytes (322 x 3 = 966): the byte-gather kernel instead of the row-staged one
    wide = synth.frame_pool(4, 100, 322, seed=5)
    for roi, out_hw in (((0, 100, 0, 322), (50, 160)), ((5, 90, 3, 300), (64, 100))):
        comp = FrameNormalise(device=0, roi=roi, out_hw=out_hw)
        u8_want, f32_want = oracle.crop_resize(wide, roi, out_hw)
        f32, u8 = comp.normalise_device(torch.from_numpy(wide).to(DEV), want_u8=True)
        assert np.array_equal(u8.cpu().numpy(), u8_want) and np.array_equal(f32.cpu().numpy(), f32_want)
        comp.onShutdown()
    odd = synth.frame_pool(3, 7, 9, seed=1)                                              # 189 bytes per frame: unaligned tail path
    comp = FrameNormalise(device=0)
    assert np.array_equal(comp.step(odd)[0], oracle.normalise(odd))
    comp.onShutdown()


def test_locate_golden_tracks(golden_tracks):
    for name in ("generated_track", "mountain_track"):
        wp, xyz = golden_tracks[f"wp/{name}"], golden_tracks[f"xyz/{name}"]
        trk = LocationTracker(wp, 0, 10, device=0)
        idx, seg = trk.locate_device(torch.from_numpy(xyz).to(DEV))
        assert np.array_equal(idx.cpu().numpy(), golden_tracks[f"idx/{name}"])
        assert np.array_equal(seg.cpu().numpy(), golden_tracks[f"seg/{name}/0_10"])
        # N = 1 python floats, like Car would pass them
        s, = trk.step(float(xyz[5, 0]), float(xyz[5, 1]), float(xyz[5, 2]))
        assert isinstance(s, float) and s == golden_tracks[f"seg/{name}/0_10"][5]
        trk.onShutdown()
        trk2 = LocationTracker(wp, -2.5, 7.25, device=0)
        seg2, = trk2.step(torch.from_numpy(xyz[:, 0].copy()).to(DEV), torch.from_numpy(xyz[:, 1].copy()).to(DEV), torch.from_numpy(xyz[:, 2].copy()).to(DEV))
        assert np.array_equal(seg2.cpu().numpy(), golden_tracks[f"seg/{name}/m2p5_7p25"])
        trk2.onShutdown()


@pytest.mark.parametrize("which", ["warp", "thread", "grid"])
def test_locate_both_kernels_on_the_golden_states(golden_tracks, monkeypatch, which):
    """The warp-per-car kernel (shuffle reduction on (distance, index); default for small batches), the thread-per-car scan and the grid walk
    (default for large batches) on the reference's own outputs, ties and > 100 sentinel cases included."""
    monkeypatch.setenv("TRS_LOCATE", which)
    for name in ("generated_track", "mountain_track"):
        wp, xyz = golden_tracks[f"wp/{name}"], golden_tracks[f"xyz/{name}"]
        trk = LocationTracker(wp, 0, 10, device=0)
        idx, seg = trk.locate_device(torch.from_numpy(xyz).to(DEV))
        assert np.array_equal(idx.cpu().numpy(), golden_tracks[f"idx/{name}"]), which
        assert np.array_equal(seg.cpu().numpy(), golden_tracks[f"seg/{name}/0_10"]), which
        xyz2, _, _, _ = synth.car_states(wp, 30_000, seed=23)
        idx2, seg2 = trk.locate_device(torch.from_numpy(xyz2).to(DEV))
        iw, sw_ = oracle.locate(wp, xyz2)
        assert np.array_equal(idx2.cpu().numpy(), iw) and np.array_equal(seg2.cpu().numpy(), sw_), which
        trk.onShutdown()


def test_locate_large_batch_against_oracle(golden_tracks):
    for name, n in (("generated_track", 200_000), ("mountain_track", 100_000)):
        wp = golden_tracks[f"wp/{name}"]
        xyz, _, _, _ = synth.car_states(wp, n, seed=17)
        idx_want, seg_want = oracle.locate(wp, xyz)
        trk = LocationTracker(wp, device=0)
        idx, seg = trk.locate_device(torch.from_numpy(xyz).to(DEV))
        assert np.array_equal(idx.cpu().numpy(), idx_want)
        assert np.array_equal(seg.cpu().numpy(), seg_want)
        assert (idx_want == 0).sum() >= n // 200                      # the > 100 sentinel cases are present
        trk.onShutdown()
    # more waypoints than one shared-memory tile
    wp = synth.synthetic_track(5000)
    xyz, _, _, _ = synth.car_states(wp, 5000, seed=3)
    trk = LocationTracker(wp, device=0)
    idx, _ = trk.locate_device(torch.from_numpy(xyz).to(DEV))
    assert np.array_equal(idx.cpu().numpy(), oracle.locate(wp, xyz)[0])
    trk.onShutdown()


@pytest.mark.timeout(300)
def test_locate_grid_walk_on_adversarial_cars(golden_tracks, monkeypatch):
    """The grid walk must return the reference's first-index argmin for every car, not only for cars near the centre line: cars exactly on cell
    corners and edges (cell sides are powers of two), on the points themselves and on repeated points, in the middle of the loop (many rings:
    put off to the warp-per-car kernel), outside the bounding box just inside and just outside the 100 limit, with NaN / infinite coordinates;
    a centre line far from the origin, one scaled to millimetres and one to kilometres (other cell sizes), and one too small for a grid."""
    monkeypatch.setenv("TRS_LOCATE", "grid")
    rng = np.random.default_rng(99)
    for name in ("generated_track", "mountain_track"):
        base = golden_tracks[f"wp/{name}"]
        for scale, shift in ((1.0, 0.0), (1.0, 1.0e6), (1e-3, 0.0), (1e3, -5.0e4)):
            wp = base * scale + shift
            lo, hi = wp.min(0), wp.max(0)
            ext = max(hi[0] - lo[0], hi[2] - lo[2])
            c = 2.0 ** np.ceil(np.log2(ext / 32.0))                  # the library's cell side
            n = 6000
            cars = [wp[rng.integers(0, len(wp), n)] + rng.standard_normal((n, 3)) * np.array([1.5, 0.05, 1.5]) * scale,           # near the line
                    wp[rng.integers(0, len(wp), 500)],                                                                           # on points
                    np.stack([rng.uniform(lo[0] - 20 * scale, hi[0] + 20 * scale, n), rng.uniform(lo[1], hi[1], n),
                              rng.uniform(lo[2] - 20 * scale, hi[2] + 20 * scale, n)], 1),                                       # anywhere around
                    np.stack([c * rng.integers(np.floor(lo[0] / c) - 2, np.floor(hi[0] / c) + 3, 2000), rng.uniform(lo[1], hi[1], 2000),
                              c * rng.integers(np.floor(lo[2] / c) - 2, np.floor(hi[2] / c) + 3, 2000)], 1),                     # cell corners
                    np.stack([c * rng.integers(np.floor(lo[0] / c), np.floor(hi[0] / c) + 1, 2000), rng.uniform(lo[1], hi[1], 2000),
                              rng.uniform(lo[2], hi[2], 2000)], 1),                                                               # cell edges
                    np.stack([lo[0] - rng.uniform(95, 105, 1000), rng.uniform(lo[1], hi[1], 1000), rng.uniform(lo[2], hi[2], 1000)], 1),   # around the limit
                    np.array([[np.nan, 1, 1], [1, np.nan, 1], [1, 1, np.nan], [np.inf, 0, 0], [0, 0, -np.inf], [1e300, 1e300, 1e300]])]
            xyz = np.ascontiguousarray(np.concatenate(cars))
            with np.errstate(invalid="ignore"):
                iw, sw_ = oracle.locate(wp, xyz)
            trk = LocationTracker(wp, device=0)
            idx, seg = trk.locate_device(torch.from_numpy(xyz).to(DEV))
            got = idx.cpu().numpy()
            assert np.array_equal(got, iw), f"{name} x{scale} +{shift}: {int((got != iw).sum())} of {len(iw)} differ, first {np.nonzero(got != iw)[0][:5]}"
            assert np.array_equal(seg.cpu().numpy(), sw_)
            trk.onShutdown()
    # a nearest point at a distance of exactly 100 inside the bounding box: the reference's strict `<` against its starting minimum keeps index 0
    wp = np.array([[i, 0, 0] for i in range(40)] + [[1000 + i, 0, 1000] for i in range(40)], np.float64)
    xyz = np.array([[89, 0, 50], [89, 0, 49.999], [89, 0, 50.001], [88, 1, 50], [1000, -50, 950], [1039, 0, 1100]], np.float64)
    want = oracle.locate(wp, xyz)[0]
    assert list(want) == [0, 39, 0, 0, 0, 0]
    for which in ("grid", "warp", "thread"):
        monkeypatch.setenv("TRS_LOCATE", which)
        trk = LocationTracker(wp, device=0)
        assert np.array_equal(trk.locate_device(torch.from_numpy(xyz).to(DEV))[0].cpu().numpy(), want), which
        trk.onShutdown()
    monkeypatch.setenv("TRS_LOCATE", "grid")
    wp = synth.synthetic_track(40)                               # fewer than 64 points: no grid, the scanning kernel answers
    xyz, _, _, _ = synth.car_states(wp, 3000, seed=8)
    trk = LocationTracker(wp, device=0)
    assert np.array_equal(trk.locate_device(torch.from_numpy(xyz).to(DEV))[0].cpu().numpy(), oracle.locate(wp, xyz)[0])
    trk.onShutdown()


def test_speed_control_golden(golden_speed):
    cur, ms, st = golden_speed["cur"], golden_speed["model_spd"], golden_speed["model_steer"]
    for cname, over in speed_cases(golden_speed).items():
        cfg = cfg_for(over)
        comp = SpeedControl(cfg, device=0)
        s, t, b, feat = comp.control_device(torch.from_numpy(cur).to(DEV), torch.from_numpy(st).to(DEV), torch.from_numpy(ms).to(DEV), want_feature=True)
        want = golden_speed[f"out/{cname}"]
        s, t, b = s.cpu().numpy(), t.cpu().numpy(), b.cpu().numpy()
        assert np.array_equal(s, want[:, 0]), cname
        # the law is discontinuous at the dead-bands (-0.2, 0 for throttle; 0.4 for brake): the float32 speed gap is computed
        # identically, so only atan's last ulp can move a state across; require equality of the zeroing decision away from the edges
        for got, ref in ((t, want[:, 1]), (b, want[:, 2])):
            differs = ~(np.abs(got - ref) <= RTOL * np.abs(ref))
            assert differs.sum() == 0, f"{cname}: {differs.sum()} states outside {RTOL} relative"
        assert np.array_equal(feat.cpu().numpy(), golden_speed["feature"])
        out = comp.step(float(cur[3]), float(st[3]), float(ms[3]))
        assert all(isinstance(v, float) for v in out) and abs(out[1] - want[3, 1]) <= RTOL * abs(want[3, 1])
        assert comp.step(None, None, None) == (0.0, 0.0, 0.0)
        comp.onShutdown()
        # the same states under NumPy 1.x scalar promotion (float64 speed gap; ADVICE r1): its own golden set
        comp1 = SpeedControl(dict(cfg, spd_ctl_numpy_legacy_promotion=True), device=0)
        s1, t1, b1, _ = comp1.control_device(torch.from_numpy(cur).to(DEV), torch.from_numpy(st).to(DEV), torch.from_numpy(ms).to(DEV))
        want1 = golden_speed[f"out_numpy1/{cname}"]
        assert np.array_equal(s1.cpu().numpy(), want1[:, 0]), cname
        for got, ref in ((t1.cpu().numpy(), want1[:, 1]), (b1.cpu().numpy(), want1[:, 2])):
            assert (~(np.abs(got - ref) <= RTOL * np.abs(ref))).sum() == 0, f"{cname} (numpy 1 promotion)"
        comp1.onShutdown()


def test_full_size_properties():
    """BASELINE-size batch (65,536 x 120x160): shard invariance, idempotence of masks, counters — no CPU oracle needed."""
    cfg = full_house_config()
    pool = torch.from_numpy(synth.frame_pool(256, 120, 160)).to(DEV)
    n = 65536
    frames = synth.expand_torch(pool, n)
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32 = comp.process_device(frames, want_f32=True)
    st = comp.stats()
    assert st["frames"] == n
    # (1) every output byte is 0 or 255 and the float tensor is exactly u8/255
    assert bool(((u8 == 0) | (u8 == 255)).all())
    assert bool((f32 == u8.to(torch.float32) / 255).all())
    # (2) counters agree with the written planes
    assert st["mask0"] == int((u8[..., 0] == 255).sum()) and st["mask1"] == int((u8[..., 1] == 255).sum())
    assert st["edge"] == int((u8[..., 2] == 255).sum()) and st["edge"] <= st["cand"] and st["strong"] <= st["edge"]
    # (3) a re-run of any sub-range gives the same bytes (shard invariance: rank r of 8 computes rows [r*N/8,(r+1)*N/8))
    lo, hi = 5 * n // 8, 6 * n // 8
    part, _ = comp.process_device(frames[lo:hi], want_f32=False)
    assert torch.equal(part, u8[lo:hi])
    # (4) EVERY distinct frame against the CPU oracle: frame i = pool[i % 256] + offset((i // 256) % 32), so the first 8,192 frames are all the
    # distinct ones and each later block of 8,192 must repeat them bit for bit (which covers all 65,536)
    distinct = 256 * 32
    want = oracle.process_batch(frames[:distinct].cpu().numpy(), cfg)
    assert np.array_equal(u8[:distinct].cpu().numpy(), want)
    for k in range(1, n // distinct):
        assert torch.equal(u8[k * distinct:(k + 1) * distinct], u8[:distinct]), f"block {k} differs from block 0"
        assert torch.equal(f32[k * distinct:(k + 1) * distinct], f32[:distinct])
    comp.onShutdown()


@pytest.mark.parametrize("want_f32", [False, True])
def test_full_size_properties_240x320(want_f32):
    """The second resolution (BASELINE.json configs[2]: full-house mask at 240x320; and the full chain with the f32 tensor) through the
    same properties on 8,192 frames: outputs are masks, the float tensor is exactly u8 / 255, counters agree with the written planes, a
    shard of the batch reproduces the whole, and every distinct frame (64 x 32 = 2,048) equals the oracle."""
    cfg = full_house_config()
    pool = torch.from_numpy(synth.frame_pool(64, 240, 320)).to(DEV)
    n = 8192
    frames = synth.expand_torch(pool, n)
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32 = comp.process_device(frames, want_f32=want_f32)
    st = comp.stats()
    assert st["frames"] == n
    assert bool(((u8 == 0) | (u8 == 255)).all())
    if want_f32:
        assert bool((f32 == u8.to(torch.float32) / 255).all())
    assert st["mask0"] == int((u8[..., 0] == 255).sum()) and st["mask1"] == int((u8[..., 1] == 255).sum())
    assert st["edge"] == int((u8[..., 2] == 255).sum()) and st["edge"] <= st["cand"] and st["strong"] <= st["edge"]
    lo, hi = 3 * n // 8, 4 * n // 8
    part, _ = comp.process_device(frames[lo:hi], want_f32=False)
    assert torch.equal(part, u8[lo:hi])
    distinct = 64 * 32
    want = oracle.process_batch(frames[:distinct].cpu().numpy(), cfg)
    assert np.array_equal(u8[:distinct].cpu().numpy(), want)
    for k in range(1, n // distinct):
        assert torch.equal(u8[k * distinct:(k + 1) * distinct], u8[:distinct]), f"block {k} differs from block 0"
    comp.onShutdown()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("h,w,n", [(240, 320, 1536), (120, 160, 3072)])
@pytest.mark.parametrize("cname", ["dyn_contrast", "exotic", "static_contrast", "edge_only", "colour_only", "adjust_only", "adjust_dynamic"])
def test_non_default_configurations_many_frames_per_cta(golden_images, cname, h, w, n):
    """Every kernel keeps a CTA busy with frame after frame, and the hand-over between its warps (plane sets by frame parity, the tail copy,
    the per-frame brightness table, the alternating ROI accumulators) only shows with several frames per CTA: five to eleven frames per CTA
    here, at both resolutions, for the configurations with a brightness / contrast table (static, or rebuilt per frame from rows 40..118),
    run-time colour ranges, and channels that keep the adjusted pixel.  Every frame against the oracle, the ROI statistic against a direct
    sum.  (A store-warp kernel that deadlocked with a table and more than two frames per CTA went unnoticed by the small-batch tests.)"""
    from tests.helpers import image_cases
    extra = {"static_contrast": dict(preprocessing_color_filter_enabled=True, preprocessing_edge_detection_enabled=True,
                                     preprocessing_contrast_enhancement_ratio=1.6, preprocessing_contrast_enhancement_offset=90),
             "adjust_dynamic": dict(preprocessing_dynamic_brightness_enabled=True, preprocessing_contrast_enhancement_ratio=1.25,
                                    preprocessing_brightness_baseline=380)}      # no filter: the streaming kernel with a table per frame
    cases = image_cases(golden_images)
    over = cases[cname] if cname in cases else extra[cname]
    cfg = cfg_for(over)
    frames = synth.expand_numpy(synth.frame_pool(96, h, w, seed=411), n, start=7)      # brightness shifts of 96 frames
    want = oracle.process_batch(frames, cfg)
    comp = ImgPreprocessing(cfg, device=0, normalised_key='cam/normalised_img', collect_stats=True)
    u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV))
    st = comp.stats()
    got = u8.cpu().numpy()
    assert np.array_equal(got, want), f"{cname}: {describe(got, want)}"
    assert np.array_equal(f32.cpu().numpy(), oracle.normalise(want))
    assert st["frames"] == n
    if cfg["preprocessing_dynamic_brightness_enabled"]:
        assert st["roi_sum"] == int(frames[:, 40:119].astype(np.uint64).sum())
    comp.onShutdown()


@pytest.mark.parametrize("hsvs", [
    None,                                                                     # the reference's defaults (core/config.py:23)
    [[[0, 0, 130], [180, 70, 255]], [[25, 100.5, 155], [43, 255, 255]]],       # same live bounds, other saturation thresholds
    [[[0, 0, 0], [180, 0, 255]], [[0, 255, 1], [179, 255, 255]]],              # saturation pinned to 0 / to 255
    [[[0, 0, 130], [180, -3, 255]], [[25, 254.5, 155], [43, 255, 255]]],       # an empty range, a half-to-even bound
])
def test_every_colour_through_the_masks(hsvs):
    """All 2^24 colours (874 frames of 120x160) through the fused kernels: the colour-mask channels of every frame must equal
    the oracle bit for bit (this pins the saturation-threshold tables of the specialised kernels)."""
    n_px = 1 << 24
    per = 120 * 160
    n = (n_px + per - 1) // per
    c = np.arange(n * per, dtype=np.uint32) % n_px
    frames = np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], axis=-1).astype(np.uint8).reshape(n, 120, 160, 3)
    over = {} if hsvs is None else dict(preprocessing_color_filter_hsvs=hsvs)
    cfg = full_house_config(**over)
    want = oracle.process_batch(frames, cfg)
    for env in (None, "TRS_NO_STORE_WARP"):
        if env:
            import os
            os.environ[env] = "1"
        try:
            got, _ = run_device(cfg, frames, want_f32=False)
        finally:
            if env:
                del os.environ[env]
        assert np.array_equal(got, want), f"{env}: {describe(got, want)}"


@pytest.mark.parametrize("env", ["TRS_FORCE_GENERIC", "TRS_NO_STORE_WARP"])
def test_other_kernels_still_match(golden_images, monkeypatch, env):
    """The store-warp kernel takes 120x160 full-house frames by default; force the resident kernel without store warps
    (TRS_NO_STORE_WARP) and the generic banded kernel (TRS_FORCE_GENERIC) on the same data."""
    monkeypatch.setenv(env, "1")
    for sname, cname, cfg, frames, expected in golden_pairs(golden_images):
        if sname not in ("f120", "f240") or cname not in ("full_house", "exotic", "edge_only"):
            continue
        got, f32 = run_device(cfg, frames)
        assert np.array_equal(got, expected), f"{sname}/{cname}: {describe(got, expected)}"
        assert np.array_equal(f32, oracle.normalise(expected))


@pytest.mark.timeout(300)
@pytest.mark.parametrize("env,h,w,n", [
    (None, 96, 128, 2400),                      # store-warp kernel, run-time geometry (not the 120x160 instantiation)
    (None, 64, 96, 2400),                       # three strip groups per row
    ("TRS_NO_STORE_WARP", 120, 160, 2400),      # resident kernel without store warps
    ("TRS_NO_STORE_WARP", 240, 320, 1200),      # banded kernel (every configuration; the default one normally takes the banded store-warp kernel)
    ("TRS_FORCE_GENERIC", 122, 166, 1500),      # generic kernel (width not a multiple of 32)
    ("TRS_FORCE_GENERIC", 120, 160, 1500),
])
def test_every_kernel_variant_with_many_frames_per_cta(golden_images, monkeypatch, env, h, w, n):
    """The hand-over protocols between the warps of a CTA (and the prefetch of the next frame) are only exercised when a CTA runs several
    frames back to back: four to eight frames per CTA through every kernel variant, four configurations each, every frame against the oracle."""
    from tests.helpers import image_cases
    if env:
        monkeypatch.setenv(env, "1")
    frames = synth.expand_numpy(synth.frame_pool(64, h, w, seed=97 + h), n, start=5)
    cases = image_cases(golden_images)
    for cname in ("full_house", "dyn_contrast", "exotic", "edge_only"):
        cfg = cfg_for(cases[cname])
        want = oracle.process_batch(frames, cfg)
        got, _ = run_device(cfg, frames, want_f32=False)
        assert np.array_equal(got, want), f"{env} {h}x{w} {cname}: {describe(got, want)}"


# ---- per-car control post-processing (SURVEY.md 8(f) rank 3): bit-exact f64 selects / divisions -----------------------------------
def _control_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "control.npz"))


def test_control_mux_reference_sequences():
    """The reference's own ControlMultiplexer, run in real time with its lock threads, replayed through the kernel with the recorded
    clock: every step of every sequence must give the same three floats (N = 1 API with DriveMode-like strings)."""
    import json

    from triton_racer_sim_b200 import ControlMultiplexer
    g = _control_golden()
    names = ['human', 'ai_steering', 'ai']
    for cname, over in json.loads(bytes(g["mux_cases_json"]).decode()).items():
        for si in range(3):
            rows = g[f"mux/{cname}/{si}"]
            mux = ControlMultiplexer(over, device=0)
            for r in rows:
                out = mux.step(names[int(r[1])], *[float(v) for v in r[2:8]], now=float(r[0]))
                assert isinstance(out[0], float) and list(out) == list(r[8:11]), f"{cname}/{si} at t={r[0]:.3f}"
            mux.onShutdown()


def test_control_mux_batch_against_oracle():
    from oracle import control as oc
    from triton_racer_sim_b200 import ControlMultiplexer
    from triton_racer_sim_b200.config import default_config
    rng = np.random.default_rng(5)
    n = 50_000
    over = dict(ai_launch_boost_throttle_enabled=True, ai_launch_boost_throttle_value=0.9, ai_launch_boost_throttle_duration=0.35,
                ai_launch_lock_steering_enabled=True, ai_launch_lock_steering_value=0.1, ai_launch_lock_steering_duration=0.12)
    cfg = default_config(**over)
    mux = ControlMultiplexer(over, device=0)
    last, launch = np.zeros(n, np.int32), np.full((oc.LAUNCH_SLOTS, n), oc.NEVER)
    now = 100.0
    for step in range(40):
        now += float(rng.uniform(0.01, 0.09))
        mode = rng.integers(0, 3, n).astype(np.int32)
        vals = rng.uniform(-1, 1, (6, n))
        want = oc.control_mux(mode, vals[0:3], vals[3:6], now, last, launch, cfg)
        got = mux.step(torch.from_numpy(mode).to(DEV), *[torch.from_numpy(v.copy()).to(DEV) for v in vals], now=now)
        assert np.array_equal(torch.stack(got).cpu().numpy(), want), f"step {step}"
    assert np.array_equal(mux.launch_times.cpu().numpy(), launch) and np.array_equal(mux.last_mode.cpu().numpy(), last)
    mux.onShutdown()


def test_driver_assistance_and_pwm_map():
    from oracle import control as oc
    from triton_racer_sim_b200 import DriverAssistance, three_segment_map
    from triton_racer_sim_b200.config import default_config
    g = _control_golden()
    st, th, br, sp = g["assist/in"]
    for mode in ("steering", "speed"):
        for k in (5, 2.5):
            da = DriverAssistance(dict(drive_assist_limit_mode=mode, drive_assist_limit_k=k), device=0)
            got = da.step(*[torch.from_numpy(a.copy()).to(DEV) for a in (st, th, br, sp)])
            assert np.array_equal(torch.stack(got).cpu().numpy(), g[f"assist/{mode}/{k}"]), f"{mode}/{k}"
            assert da.step(0.5, None, 0.0, 3.0) == (0.5, None, 0.0)                                  # driver_assistance.py:15
            one = da.step(float(st[7]), float(th[7]), float(br[7]), float(sp[7]))
            assert list(one) == list(g[f"assist/{mode}/{k}"][:, 7])
            da.onShutdown()
    rng = np.random.default_rng(9)
    big = [rng.uniform(-2, 2, 200_000), rng.uniform(-1, 1, 200_000), rng.uniform(0, 1, 200_000), rng.uniform(-5, 30, 200_000)]
    for mode in ("steering", "speed"):
        cfg = default_config(drive_assist_limit_mode=mode, drive_assist_limit_k=3.7)
        da = DriverAssistance(cfg, device=0)
        got = da.step(*[torch.from_numpy(a).to(DEV) for a in big])
        assert np.array_equal(torch.stack(got).cpu().numpy(), np.stack(oc.driver_assist(*big, cfg)))
        da.onShutdown()
    v = g["pwm/in"]
    for name in ("steering", "throttle", "odd"):
        a, b, c = g[f"pwm/{name}/map"]
        assert np.array_equal(three_segment_map(torch.from_numpy(v.copy()).to(DEV), a, b, c).cpu().numpy(), g[f"pwm/{name}"]), name
    assert three_segment_map(-0.5, 430, 350, 300) == 350 + (350 - 430) * -0.5


# ---- robustness of the boundary (round-1 advisor findings) ------------------------------------------------------------------------
def test_device_methods_validate_their_tensors():
    """A CPU tensor, a wrong dtype or a wrong shape must raise in Python: handed to the library they would become an illegal-address
    fault that poisons the CUDA context."""
    from triton_racer_sim_b200 import ControlMultiplexer
    frames = torch.from_numpy(synth.frame_pool(2, 120, 160)).to(DEV)
    comp = ImgPreprocessing(full_house_config(), device=0)
    with pytest.raises(ValueError):
        comp.process_device(frames.cpu())
    with pytest.raises(ValueError):
        comp.process_device(frames, out_u8=torch.empty(frames.shape, dtype=torch.uint8))                 # output on the CPU
    with pytest.raises(ValueError):
        comp.process_device(frames, out_f32=torch.empty((1, 120, 160, 3), dtype=torch.float32, device=DEV), want_f32=True)
    with pytest.raises(ValueError):
        comp.process_host(frames.cpu().numpy(), keep_f32_dev=torch.empty(frames.shape, dtype=torch.float32))
    comp.onShutdown()
    norm = FrameNormalise(device=0)
    with pytest.raises(ValueError):
        norm.normalise_device(frames.cpu())
    norm.onShutdown()
    trk = LocationTracker(synth.synthetic_track(50), device=0)
    with pytest.raises(ValueError):
        trk.locate_device(torch.zeros((4, 3), dtype=torch.float64))
    with pytest.raises(ValueError):
        trk.locate_device(torch.zeros((4, 3), dtype=torch.float32, device=DEV))
    trk.onShutdown()
    spd = SpeedControl({}, device=0)
    with pytest.raises(ValueError):
        spd.control_device(torch.zeros(4, dtype=torch.float64), torch.zeros(4), torch.zeros(4))
    with pytest.raises(ValueError):
        spd.control_device(torch.zeros(4, dtype=torch.float64, device=DEV), torch.zeros(3, device=DEV), torch.zeros(4, device=DEV))
    spd.onShutdown()
    mux = ControlMultiplexer({}, device=0)
    with pytest.raises(ValueError):
        mux.mux_device(torch.zeros(4, dtype=torch.int32, device=DEV), torch.zeros((3, 4), dtype=torch.float64), torch.zeros((3, 4), dtype=torch.float64, device=DEV), 0.0)
    with pytest.raises(ValueError):
        mux.mux_device(torch.zeros(4, dtype=torch.int32, device=DEV), torch.zeros((3, 5), dtype=torch.float64, device=DEV),
                       torch.zeros((3, 4), dtype=torch.float64, device=DEV), 0.0)
    mux.onShutdown()
    # the context survived all of that
    comp = ImgPreprocessing(full_house_config(), device=0)
    u8, _ = comp.process_device(frames)
    assert np.array_equal(u8.cpu().numpy(), oracle.process_batch(frames.cpu().numpy(), full_house_config()))
    comp.onShutdown()


def test_host_pipeline_waits_for_work_on_the_callers_stream():
    """trs_preprocess_host writes keep_f32_dev from internal streams: a consumer of the previous step's tensor that is still queued on the
    caller's stream (here: a long spin, then a clone) must see the OLD contents."""
    cfg = full_house_config()
    a = synth.frame_pool(64, 120, 160, seed=5)
    b = synth.frame_pool(64, 120, 160, seed=6)
    comp = ImgPreprocessing(cfg, device=0)
    keep = torch.zeros((64, 120, 160, 3), dtype=torch.float32, device=DEV)
    ua, _ = comp.process_host(a, keep_f32_dev=keep)
    want_a = oracle.normalise(oracle.process_batch(a, cfg))
    assert np.array_equal(keep.cpu().numpy(), want_a)
    torch.cuda._sleep(400_000_000)                       # ~0.2 s of spinning on the current stream ...
    snap = keep.clone()                                  # ... then the consumer of step A's tensor
    ub, _ = comp.process_host(b, keep_f32_dev=keep)      # step B must not overwrite `keep` before the clone has run
    torch.cuda.synchronize()
    assert np.array_equal(snap.cpu().numpy(), want_a), "the host pipeline overwrote keep_f32_dev while the caller's stream was still reading it"
    assert np.array_equal(keep.cpu().numpy(), oracle.normalise(oracle.process_batch(b, cfg)))
    comp.onShutdown()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_calls_leave_the_callers_current_device_alone(golden_tracks):
    """A component bound to cuda:1 while torch's current device is cuda:0: every entry point must run on its own device and put the
    caller's device back (PyTorch derives its current device from cudaGetDevice)."""
    cfg = full_house_config()
    frames = synth.frame_pool(8, 120, 160, seed=3)
    torch.cuda.set_device(0)
    comp = ImgPreprocessing(cfg, device=1, normalised_key='cam/normalised_img')
    assert torch.cuda.current_device() == 0
    u8, f32 = comp.process_device(torch.from_numpy(frames).to("cuda:1"))
    assert torch.cuda.current_device() == 0
    probe = torch.empty(4, device="cuda")                # a device-less allocation after the call lands on the caller's device
    assert probe.device.index == 0
    torch.cuda.synchronize(1)
    want = oracle.process_batch(frames, cfg)
    assert np.array_equal(u8.cpu().numpy(), want) and np.array_equal(f32.cpu().numpy(), oracle.normalise(want))
    h8, _ = comp.process_host(frames)
    assert torch.cuda.current_device() == 0 and np.array_equal(h8, want)
    comp.onShutdown()
    wp, xyz = golden_tracks["wp/generated_track"], golden_tracks["xyz/generated_track"]
    trk = LocationTracker(wp, 0, 10, device=1)
    idx, _ = trk.locate_device(torch.from_numpy(xyz).to("cuda:1"))
    assert torch.cuda.current_device() == 0
    assert np.array_equal(idx.cpu().numpy(), golden_tracks["idx/generated_track"])
    trk.onShutdown()
    assert torch.cuda.current_device() == 0
