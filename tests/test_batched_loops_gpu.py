"""The batched paths at sizes where every loop makes several trips: the host pipeline over many chunks and streams, the crop / resize
kernels over many rows per CTA, and the streaming normalise over several unrolled trips.

The other tests run these paths at sizes where each loop makes one trip (a few golden frames are one chunk on one stream; a few
thousand output rows give every resize CTA one row), so a defect that only shows from the second chunk, row or trip on passes them.
Each test here states the trips it claims, computed from the SM count and the launch rules restated from csrc/trs_api.cu, and fails
with that precondition's message if a change to a grid cap or a chunk size makes it test less.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from tests.helpers import cfg_for, image_cases
from triton_racer_sim_b200 import FrameNormalise, ImgPreprocessing, synth
from triton_racer_sim_b200 import _native as nat

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
DEV = "cuda:0"
HOST_STREAMS = 3                      # trs_api.cu:65
DEFAULT_CHUNK_BYTES = 48 << 20        # trs_api.cu:74 (TrsSwitches::host_chunk_bytes)
RESIZE_DEPTH = 8                      # misc_kernels.cuh:103: rows in flight per CTA in k_crop_resize_rows
NO_COUNT = ("hyst_sweeps",)           # per-frame sweep counts are a property of the schedule, not of the result


@pytest.fixture(scope="module")
def sm_count():
    ctx = nat.Context(0)
    n = ctx.sm_count
    ctx.close()
    return n


def describe(got, want):
    bad = np.argwhere(got != want)
    return f"{len(bad)} of {got.size} differ; first at {bad[:5].tolist()}"


def counters(st):
    return {k: v for k, v in st.items() if not k.startswith("t_") and k not in NO_COUNT}


# ---- host pipeline (trs_preprocess_host) ------------------------------------------------------------------------------------------
def host_chunks(n, h, w, chunk_bytes):
    """Frames per chunk and the number of chunks, as trs_preprocess_host (trs_api.cu:1102-1106) cuts a batch."""
    fb = h * w * 3
    chunk = min(max(1, chunk_bytes // fb), n)
    chunk = (chunk + 3) & ~3
    return chunk, -(-n // chunk)


def assert_many_chunks(n, h, w, chunk_bytes=1 << 20):
    chunk, chunks = host_chunks(n, h, w, chunk_bytes)
    assert chunks >= 7 and n % chunk != 0, \
        f"{n} frames of {h}x{w} make {chunks} chunks of {chunk} frames (last {n % chunk}): the test needs >= 7 chunks and a ragged last one"
    assert chunks >= 2 * HOST_STREAMS, f"{chunks} chunks: every one of the {HOST_STREAMS} staging sets must serve at least two"
    return chunk, chunks


def device_reference(cfg, frames, want_f32=True):
    """process_device on the same frames: (u8, f32 or None, counters)."""
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV), want_f32=want_f32)
    st = comp.stats()
    out = u8.cpu().numpy(), (f32.cpu().numpy() if f32 is not None else None), counters(st)
    comp.onShutdown()
    return out


def pinned_like(shape, dtype):
    return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()


# (switch, h, w, configuration, frames): every kernel launch_preprocess can pick (trs_api.cu:302-437)
HOST_KERNELS = {
    "store_warp_120x160": (None, 120, 160, "full_house", 150),
    "banded_store_warp_240x320": (None, 240, 320, "full_house", 30),
    "resident_no_store_warp": ("TRS_NO_STORE_WARP", 120, 160, "full_house", 150),
    "banded_no_store_warp": ("TRS_NO_STORE_WARP", 240, 320, "full_house", 30),
    "table_dyn_contrast": (None, 120, 160, "dyn_contrast", 150),
    "no_filter_adjust_stream": (None, 120, 160, "adjust_dynamic", 150),
    "generic_122x166": ("TRS_FORCE_GENERIC", 122, 166, "full_house", 150),
    "generic_7x9": (None, 7, 9, "exotic", 40_000),            # fb % 4 != 0: chunk bases are only 4-frame aligned
}
EXTRA_CFG = {"adjust_dynamic": dict(preprocessing_dynamic_brightness_enabled=True, preprocessing_contrast_enhancement_ratio=1.25,
                                    preprocessing_brightness_baseline=380)}


def kernel_case(golden_images, monkeypatch, name):
    env, h, w, cname, n = HOST_KERNELS[name]
    if env:
        monkeypatch.setenv(env, "1")
    cases = image_cases(golden_images)
    cfg = cfg_for(cases[cname] if cname in cases else EXTRA_CFG[cname])
    return cfg, h, w, n


@pytest.mark.parametrize("name", list(HOST_KERNELS))
def test_host_pipeline_many_chunks_every_kernel(golden_images, monkeypatch, name):
    """u8 + host f32 from pageable memory, 1 MB chunks: >= 7 chunks over the three streams, the last one ragged."""
    cfg, h, w, n = kernel_case(golden_images, monkeypatch, name)
    monkeypatch.setenv("TRS_HOST_CHUNK_MB", "1")                # read when the context is created
    assert_many_chunks(n, h, w)
    frames = synth.expand_numpy(synth.frame_pool(64, h, w, seed=31 + h + w), n, start=3)
    want_u8, want_f32, want_st = device_reference(cfg, frames)
    assert np.array_equal(want_u8, oracle.process_batch(frames, cfg)), f"{name}: the device path differs from the oracle"
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32 = comp.process_host(frames, out_f32=np.empty(frames.shape, np.float32))
    assert np.array_equal(u8, want_u8), f"{name} u8: {describe(u8, want_u8)}"
    assert np.array_equal(f32, want_f32), f"{name} f32: {describe(f32, want_f32)}"
    assert counters(comp.last_stats) == want_st, f"{name}: {counters(comp.last_stats)} != {want_st}"
    comp.onShutdown()


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("form", ["u8", "u8_host_f32", "u8_keep_f32_dev", "host_f32", "stats"])
def test_host_pipeline_many_chunks_every_output_form(monkeypatch, form, pinned):
    """Every output form of trs_preprocess_host on the 120x160 store-warp kernel, from pageable and from pinned buffers."""
    monkeypatch.setenv("TRS_HOST_CHUNK_MB", "1")
    h, w, n = 120, 160, 153
    assert_many_chunks(n, h, w)
    cfg = cfg_for(dict(preprocessing_color_filter_enabled=True, preprocessing_edge_detection_enabled=True))
    src = synth.expand_numpy(synth.frame_pool(64, h, w, seed=8), n, start=40)
    want_u8, want_f32, want_st = device_reference(cfg, src)
    frames = pinned_like(src.shape, torch.uint8) if pinned else src.copy()
    frames[...] = src
    alloc = (lambda s, dt: pinned_like(s, {np.uint8: torch.uint8, np.float32: torch.float32}[dt])) if pinned else (lambda s, dt: np.empty(s, dt))
    out_u8 = alloc(src.shape, np.uint8) if form.startswith("u8") else None
    out_f32 = alloc(src.shape, np.float32) if form in ("u8_host_f32", "host_f32") else None
    keep = torch.full(src.shape, -1.0, dtype=torch.float32, device=DEV) if form == "u8_keep_f32_dev" else None
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32 = comp.process_host(frames, out_u8=out_u8, out_f32=out_f32, keep_f32_dev=keep, want_u8=out_u8 is not None)
    if out_u8 is not None:
        assert np.array_equal(u8, want_u8), f"{form} u8: {describe(u8, want_u8)}"
    if out_f32 is not None:
        assert np.array_equal(f32, want_f32), f"{form} f32: {describe(f32, want_f32)}"
    if keep is not None:
        k = keep.cpu().numpy()
        assert np.array_equal(k, want_f32), f"{form} keep_f32_dev: {describe(k, want_f32)}"
    assert counters(comp.last_stats) == want_st, f"{form}: {counters(comp.last_stats)} != {want_st}"
    assert np.array_equal(frames, src), "the input buffer was written"
    comp.onShutdown()


def test_host_pipeline_staging_grows_between_calls(golden_images, monkeypatch):
    """Three calls on one component, frame sizes growing and then shrinking: each call's chunk needs more staging than the last
    (grow_staging, trs_api.cu:443-451, reallocates all three sets), and the third call runs on the grown buffers."""
    monkeypatch.setenv("TRS_HOST_CHUNK_MB", "1")
    cfg = cfg_for(image_cases(golden_images)["full_house"])
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    staged = 0
    for k, (h, w, n) in enumerate(((7, 9, 3000), (240, 320, 30), (120, 160, 50))):
        chunk, chunks = host_chunks(n, h, w, 1 << 20)
        assert chunk * h * w * 3 > staged, f"call {k}: {chunk} frames of {h}x{w} need no more staging than the call before"
        assert k == 0 or chunks >= HOST_STREAMS, f"call {k}: {chunks} chunks leave a staging set unused"
        staged = chunk * h * w * 3
        frames = synth.frame_pool(n, h, w, seed=50 + k)
        want_u8, want_f32, want_st = device_reference(cfg, frames)
        u8, f32 = comp.process_host(frames, out_f32=np.empty(frames.shape, np.float32))
        assert np.array_equal(u8, want_u8), f"call {k} {h}x{w}: {describe(u8, want_u8)}"
        assert np.array_equal(f32, want_f32), f"call {k} {h}x{w} f32"
        assert counters(comp.last_stats) == want_st, f"call {k}"
    comp.onShutdown()


@pytest.mark.timeout(900)
def test_host_pipeline_at_the_benchmark_shape():
    """bench.py's e2e leg: 16,384 frames of 120x160 through the default 48 MB chunks (19 chunks, each staging set reused six times),
    pinned input and output, the f32 tensor kept on the device.  Against the device path byte for byte; the first 8,192 frames are
    every distinct frame of the expansion (pool[i % 256] + offset((i // 256) % 32)), checked against the oracle, and the second half
    repeats them."""
    h, w, n, pool = 120, 160, 16_384, 256
    chunk, chunks = host_chunks(n, h, w, DEFAULT_CHUNK_BYTES)
    assert chunks >= 6 * HOST_STREAMS, f"{chunks} chunks of {chunk} frames: fewer than six per staging set"
    cfg = cfg_for(dict(preprocessing_color_filter_enabled=True, preprocessing_edge_detection_enabled=True))
    src = synth.expand_numpy(synth.frame_pool(pool, h, w), n)
    distinct = pool * 32
    ref = ImgPreprocessing(cfg, device=0, collect_stats=True)
    d_u8, d_f32 = ref.process_device(torch.from_numpy(src).to(DEV), want_f32=True)
    want_st = counters(ref.stats())
    want_u8 = d_u8.cpu().numpy()
    ref.onShutdown()
    assert np.array_equal(want_u8[:distinct], oracle.process_batch(src[:distinct], cfg))
    assert np.array_equal(want_u8[distinct:], want_u8[:distinct])
    frames = pinned_like(src.shape, torch.uint8)
    frames[...] = src
    del src
    out = pinned_like(frames.shape, torch.uint8)
    keep = torch.empty(frames.shape, dtype=torch.float32, device=DEV)
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, _ = comp.process_host(frames, out_u8=out, keep_f32_dev=keep)
    assert np.array_equal(u8, want_u8), describe(u8, want_u8)
    assert torch.equal(keep, d_f32)
    assert counters(comp.last_stats) == want_st
    comp.onShutdown()


# ---- crop / resize / normalise (trs_normalise) ----------------------------------------------------------------------------------
def resize_plan(sms, n, h_in, w_in, roi, out_hw, kernel_switch=None, in_aligned=True):
    """The kernel trs_normalise picks for 16-byte aligned outputs (trs_api.cu:583-607), its grid and the trips of its grid-stride loop.
    rows / words: one output row per trip, grid = min(rows, 16 SMs); scalar: one pixel per thread per trip, grid = min(px / 256, 16 SMs)."""
    y0, y1, x0, x1 = roi
    ho, wo = out_hw
    cap = 16 * sms
    if (wo * 3) % 4 == 0 and wo + ho <= 8192 and kernel_switch != "TRS_RESIZE_SCALAR":
        rows = n * ho
        col_lo, col_hi = (3 * x0) & ~15, (3 * x1 + 15) & ~15
        span = min(col_hi, w_in * 3) - col_lo
        tab = (16 * ((wo * 3) >> 2) + 4 * ho + 15) & ~15
        grid = min(rows, cap)
        kern = "rows" if ((w_in * 3) % 16 == 0 and in_aligned and span % 16 == 0 and tab + RESIZE_DEPTH * span <= 48 * 1024
                          and kernel_switch != "TRS_RESIZE_GATHER") else "words"
        return kern, grid, rows // grid
    px = n * ho * wo
    grid = min(-(-px // 256), cap)
    return "scalar", grid, px // (grid * 256)


# (source h, w, window (y0, y1, x0, x1), output (h, w), frames, kernel of the default dispatch)
RESIZE_CASES = {
    "camera_240x320_to_120x160": (240, 320, (0, 240, 0, 320), (120, 160), 512, "rows"),
    "output_taller_than_the_grid": (240, 320, (0, 240, 0, 320), (2500, 8), 128, "rows"),
    "window_3x0_not_16_aligned": (240, 320, (10, 230, 17, 301), (77, 132), 800, "rows"),
    "upscale": (240, 320, (0, 240, 0, 320), (300, 332), 200, "rows"),
    "source_rows_of_966_bytes": (100, 322, (5, 90, 3, 300), (64, 100), 1000, "words"),
}


@pytest.mark.parametrize("switch", [None, "TRS_RESIZE_GATHER", "TRS_RESIZE_SCALAR"], ids=["default", "gather", "scalar"])
@pytest.mark.parametrize("case", list(RESIZE_CASES))
def test_crop_resize_many_rows_per_cta(monkeypatch, sm_count, case, switch):
    """Each resize kernel with many output rows per CTA: k_crop_resize_rows cycles its ring of RESIZE_DEPTH cp.async groups and
    advances (frame, row) by the grid stride with a carry, which only runs when a CTA gathers more than one row.  u8 only, f32
    only and both, against oracle.crop_resize."""
    h, w, roi, out_hw, n, default = RESIZE_CASES[case]
    kern, grid, trips = resize_plan(sm_count, n, h, w, roi, out_hw, switch)
    want_kern = {None: default, "TRS_RESIZE_GATHER": "words", "TRS_RESIZE_SCALAR": "scalar"}[switch]
    assert kern == want_kern, f"{case}: the dispatch rules pick {kern}, the test is written for {want_kern}"
    if kern == "scalar":
        assert trips >= 3, f"{case}: k_crop_resize makes {trips} full trips per thread (grid {grid}), the test needs >= 3"
    else:
        assert trips >= 3 * RESIZE_DEPTH, f"{case}: {trips} rows per CTA (grid {grid}), the test needs >= {3 * RESIZE_DEPTH} (three turns of the ring)"
    if case == "camera_240x320_to_120x160" and kern == "rows":
        assert grid % out_hw[0] != 0, f"grid {grid} is a multiple of h_out: the row carry never runs"
    if case == "output_taller_than_the_grid":
        assert grid < out_hw[0], f"grid {grid} >= h_out {out_hw[0]}: the frame index never advances by zero"
    if switch:
        monkeypatch.setenv(switch, "1")
    frames = synth.frame_pool(n, h, w, seed=7 + n)
    u8_want, f32_want = oracle.crop_resize(frames, roi, out_hw)
    d = torch.from_numpy(frames).to(DEV)
    comp = FrameNormalise(device=0, roi=roi, out_hw=out_hw)
    y0, y1, x0, x1 = roi
    ho, wo = out_hw
    for want_u8, want_f32 in ((True, False), (False, True), (True, True)):
        u8 = torch.full((n, ho, wo, 3), 7, dtype=torch.uint8, device=DEV) if want_u8 else None
        f32 = torch.full((n, ho, wo, 3), -1.0, dtype=torch.float32, device=DEV) if want_f32 else None
        nat.check(comp.ctx.lib.trs_normalise(comp.ctx.handle, C.c_void_p(d.data_ptr()), n, h, w, y0, y1, x0, x1, ho, wo,
                                             C.c_void_p(f32.data_ptr()) if want_f32 else None,
                                             C.c_void_p(u8.data_ptr()) if want_u8 else None,
                                             C.c_void_p(torch.cuda.current_stream(0).cuda_stream)), "trs_normalise")
        tag = f"{case} {kern} u8={want_u8} f32={want_f32}"
        if want_u8:
            got = u8.cpu().numpy()
            assert np.array_equal(got, u8_want), f"{tag}: {describe(got, u8_want)}"
        if want_f32:
            got = f32.cpu().numpy()
            assert np.array_equal(got, f32_want), f"{tag} f32: {describe(got, f32_want)}"
    comp.onShutdown()


def normalise_trips(sms, n_bytes):
    """k_normalise_stream<8> (trs_api.cu:566-579, misc_kernels.cuh:47-60): full unrolled trips of every thread, and the bytes
    k_normalise_bytes finishes."""
    words = n_bytes // 4
    grid = min(-(-words // (256 * 8)), 32 * sms)
    return words // (grid * 256 * 8), n_bytes - 4 * words


@pytest.mark.parametrize("n,h,w,offset", [(2560, 120, 160, 0), (2001, 121, 163, 0), (2560, 120, 160, 4)],
                         ids=["stream", "stream_and_byte_tail", "view_4_bytes_in"])
def test_normalise_several_unrolled_trips(sm_count, n, h, w, offset):
    """The identity normalise: the word stream at >= 3 full unrolled trips, the byte kernel behind it when the size is not a multiple
    of 4, and an input 4 bytes into its allocation, which must leave the stream kernel for the gathering one.  Against oracle.normalise."""
    n_bytes = n * h * w * 3
    trips, tail = normalise_trips(sm_count, n_bytes)
    if offset:
        kern, grid, rows = resize_plan(sm_count, n, h, w, (0, h, 0, w), (h, w), in_aligned=False)
        assert kern == "words" and rows >= 3, f"a misaligned input takes {kern} with {rows} rows per CTA"
    else:
        assert trips >= 3, f"{n} frames of {h}x{w}: {trips} full unrolled trips of k_normalise_stream, the test needs >= 3"
        assert (tail > 0) == (n_bytes % 4 != 0)
    frames = synth.frame_pool(n, h, w, seed=n + h)
    raw = torch.empty(n_bytes + 64, dtype=torch.uint8, device=DEV)
    view = raw[offset:offset + n_bytes].view(n, h, w, 3)
    view.copy_(torch.from_numpy(frames))
    assert view.data_ptr() % 16 == offset
    comp = FrameNormalise(device=0)
    got = comp.normalise_device(view).cpu().numpy()
    want = oracle.normalise(frames)
    assert np.array_equal(got, want), describe(got, want)
    comp.onShutdown()
