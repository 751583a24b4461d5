"""Several preprocessing configurations in one batch (trs_set_preproc_configs / trs_preprocess_configs, MultiTrackImgPreprocessing):
every frame gets exactly what ImgPreprocessing with its own configuration gives it, through every kernel the single-configuration
dispatch can pick, with per-configuration statistics, out-of-range indices, stream order, graph capture and bad arguments."""
import numpy as np
import pytest
import torch

import oracle
from tests.helpers import cfg_for, image_cases
from triton_racer_sim_b200 import ImgPreprocessing, MultiTrackImgPreprocessing, synth
from triton_racer_sim_b200 import _native as nat

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN_CFGS = ["full_house", "colour_only", "edge_only", "adjust_only", "dyn_contrast", "exotic", "edge_tight"]
SETS = ["f120", "f120_shift", "f240", "odd_7x9", "odd_33x50", "odd_45x160", "odd_121x163", "odd_64x96"]


def _cfgs(golden_images, names):
    cases = image_cases(golden_images)
    return [cfg_for(cases[c]) for c in names]


def _single(cfg, frames, want_f32=False, stats=False):
    comp = ImgPreprocessing(cfg, device=0, normalised_key='n' if want_f32 else None, collect_stats=stats)
    u8, f32 = comp.process_device(frames)
    st = comp.stats() if stats else None
    torch.cuda.synchronize()
    comp.onShutdown()
    return u8, f32, st


def _grid(ctx):
    return ctx.sm_count * 2


@pytest.mark.parametrize("mode", ["u8", "f32", "both"])
def test_every_frame_gets_its_configurations_golden_answer(golden_images, mode):
    """Each golden frame set repeated, with random indices over the golden configurations it has answers for (all seven at 120x160)."""
    cfgs = _cfgs(golden_images, GOLDEN_CFGS)
    comp = MultiTrackImgPreprocessing(cfgs, device=0, normalised_key='cam/normalised_img')
    rng = np.random.default_rng(11)
    for sname in SETS:
        src = golden_images[f"in/{sname}"]
        have = [c for c, name in enumerate(GOLDEN_CFGS) if f"out/{sname}/{name}" in golden_images.files]
        assert len(have) >= 2 and (sname != "f120" or len(have) == 7)
        reps = max(1, 40 // len(src))
        frames = np.concatenate([src] * reps)
        idx = rng.choice(np.array(have), len(frames)).astype(np.int32)
        want = np.stack([golden_images[f"out/{sname}/{GOLDEN_CFGS[c]}"][i % len(src)] for i, c in enumerate(idx)])
        u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV), torch.from_numpy(idx).to(DEV), want_u8=mode != "f32",
                                      want_f32=mode != "u8")
        if mode != "f32":
            assert np.array_equal(u8.cpu().numpy(), want), sname
        else:
            assert u8 is None
        if mode != "u8":
            assert np.array_equal(f32.cpu().numpy(), oracle.normalise(want)), sname
        else:
            assert f32 is None
    comp.onShutdown()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("env", [None, "TRS_NO_STORE_WARP", "TRS_NO_BANDED", "TRS_FORCE_GENERIC"])
@pytest.mark.parametrize("h,w", [(120, 160), (240, 320), (96, 128), (122, 166)])
def test_every_kernel_variant_with_many_frames_per_cta(golden_images, monkeypatch, env, h, w):
    """Four to eleven frames per CTA for each configuration's kernel (store-warp, banded store-warp, resident, banded, generic, the
    no-filter stream with a static and a per-frame table), indices random and sorted: each configuration's frames equal ImgPreprocessing
    with that configuration on the gathered frames, and the oracle on a subset."""
    if env:
        monkeypatch.setenv(env, "1")
    names = ["full_house", "dyn_contrast", "exotic", "edge_only", "adjust_only", "colour_only"]
    cfgs = _cfgs(golden_images, names)
    dyn_adjust = dict(cfgs[4], preprocessing_dynamic_brightness_enabled=True)
    cfgs.append(dyn_adjust)
    comp = MultiTrackImgPreprocessing(cfgs, device=0)
    k = len(cfgs)
    n = _grid(comp.ctx) * (7 if h * w < 50_000 else 4)
    frames = torch.from_numpy(synth.expand_numpy(synth.frame_pool(64, h, w, seed=41 + h), n, start=3)).to(DEV)
    rng = np.random.default_rng(h + w)
    for idx in (rng.integers(0, k, n), np.sort(rng.integers(0, k, n))):
        idx = idx.astype(np.int32)
        u8, _ = comp.process_device(frames, torch.from_numpy(idx).to(DEV))
        got = u8.cpu().numpy()
        for c, cfg in enumerate(cfgs):
            sel = np.flatnonzero(idx == c)
            want, _, _ = _single(cfg, frames[torch.from_numpy(sel).to(DEV)])
            assert np.array_equal(got[sel], want.cpu().numpy()), (env, h, w, c)
            sub = sel[:6]
            assert np.array_equal(got[sub], oracle.process_batch(frames[torch.from_numpy(sub).to(DEV)].cpu().numpy(), cfg)), (env, h, w, c)
    comp.onShutdown()


def test_one_configuration_equals_trs_preprocess(golden_images):
    cfg = _cfgs(golden_images, ["full_house"])[0]
    frames = torch.from_numpy(synth.expand_numpy(synth.frame_pool(64, 120, 160, seed=5), 1000)).to(DEV)
    comp = MultiTrackImgPreprocessing([cfg], device=0, normalised_key='n', collect_stats=True)
    u8, f32 = comp.process_device(frames, torch.zeros(1000, dtype=torch.int32, device=DEV))
    st = comp.stats()
    want_u8, want_f32, want_st = _single(cfg, frames, want_f32=True, stats=True)
    assert torch.equal(u8, want_u8) and torch.equal(f32, want_f32)
    assert len(st) == 1
    for key in ("frames", "mask0", "mask1", "mask2", "mask3", "edge", "strong", "cand", "roi_sum"):
        assert st[0][key] == want_st[key], key
    comp.onShutdown()


def test_empty_configurations_and_batch_sizes(golden_images):
    cfgs = _cfgs(golden_images, GOLDEN_CFGS)
    comp = MultiTrackImgPreprocessing(cfgs, device=0, normalised_key='n')
    g = _grid(comp.ctx)
    pool = synth.frame_pool(64, 120, 160, seed=9)
    want_by_cfg = [oracle.process_batch(pool, c) for c in cfgs]
    rng = np.random.default_rng(3)
    for n in (1, 2, g - 1, g + 1, 3 * g + 5):
        frames = pool[np.arange(n) % 64]
        for idx in (np.full(n, 3), np.full(n, len(cfgs) - 1), np.where(rng.random(n) < 0.5, 0, 5), rng.integers(0, len(cfgs), n)):
            idx = idx.astype(np.int32)
            u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV), torch.from_numpy(idx).to(DEV))
            want = np.stack([want_by_cfg[c][i % 64] for i, c in enumerate(idx)])
            assert np.array_equal(u8.cpu().numpy(), want), n
            assert np.array_equal(f32.cpu().numpy(), oracle.normalise(want)), n
    e = torch.empty((0, 120, 160, 3), dtype=torch.uint8, device=DEV)
    u8, f32 = comp.process_device(e, torch.empty(0, dtype=torch.int32, device=DEV))
    assert u8.shape == e.shape and f32.shape == e.shape
    comp.onShutdown()


def test_out_of_range_indices(golden_images):
    cfgs = _cfgs(golden_images, ["full_house", "exotic"])
    comp = MultiTrackImgPreprocessing(cfgs, device=0, normalised_key='n')
    frames = synth.frame_pool(40, 120, 160, seed=4)
    idx = np.array([0, -1, 1, 2, 2**31 - 1, 0, 1, -2**31] * 5, np.int32)
    u8, f32 = comp.process_device(torch.from_numpy(frames).to(DEV), torch.from_numpy(idx).to(DEV))
    u8, f32 = u8.cpu().numpy(), f32.cpu().numpy()
    bad = (idx < 0) | (idx >= 2)
    assert (u8[bad] == 0).all() and np.isnan(f32[bad]).all()
    for c in range(2):
        assert np.array_equal(u8[idx == c], oracle.process_batch(frames[idx == c], cfgs[c]))
    with pytest.raises(ValueError):
        comp.step(frames, idx)
    with pytest.raises(ValueError):
        comp.step(frames[0], 2)
    with pytest.raises(ValueError):
        comp.step(frames[0], -1)
    comp.onShutdown()


def test_host_forms(golden_images):
    cfgs = _cfgs(golden_images, ["full_house", "edge_only", "adjust_only"])
    comp = MultiTrackImgPreprocessing(cfgs, device=0, normalised_key='cam/normalised_img')
    frames = synth.frame_pool(12, 120, 160, seed=8)
    idx = np.arange(12) % 3
    u8, f32 = comp.step(frames, idx)
    assert isinstance(u8, np.ndarray)
    for c in range(3):
        assert np.array_equal(u8[idx == c], oracle.process_batch(frames[idx == c], cfgs[c]))
    assert np.array_equal(f32, oracle.normalise(u8))
    one, one_f = comp.step(frames[4], 1)
    assert one.shape == (120, 160, 3) and np.array_equal(one, oracle.process_batch(frames[4:5], cfgs[1])[0])
    assert np.array_equal(one_f, oracle.normalise(one))
    assert comp.step(None, 0) == (None, None)
    comp.onShutdown()


def test_statistics_per_configuration(golden_images):
    names = ["full_house", "exotic", "dyn_contrast", "adjust_only"]
    cfgs = _cfgs(golden_images, names) + [dict(_cfgs(golden_images, ["edge_only"])[0])]
    comp = MultiTrackImgPreprocessing(cfgs, device=0, collect_stats=True)
    n = 2000
    frames = torch.from_numpy(synth.expand_numpy(synth.frame_pool(64, 120, 160, seed=21), n)).to(DEV)
    idx = np.random.default_rng(2).integers(0, len(cfgs) - 1, n).astype(np.int32)      # the last configuration gets no frames
    comp.process_device(frames, torch.from_numpy(idx).to(DEV))
    st = comp.stats()
    assert len(st) == len(cfgs)
    for c, cfg in enumerate(cfgs):
        sel = torch.from_numpy(np.flatnonzero(idx == c)).to(DEV)
        if len(sel) == 0:
            assert all(v == 0 for v in st[c].values()), c
            continue
        _, _, want = _single(cfg, frames[sel], stats=True)
        for key in ("frames", "mask0", "mask1", "mask2", "mask3", "edge", "strong", "cand", "roi_sum"):
            assert st[c][key] == want[key], (names[c] if c < len(names) else c, key)
    comp.onShutdown()


def test_stream_order_graph_capture_and_device(golden_images):
    cfgs = _cfgs(golden_images, ["full_house", "exotic", "dyn_contrast"])
    comp = MultiTrackImgPreprocessing(cfgs, device=0)
    n = 1500
    pool = synth.expand_numpy(synth.frame_pool(64, 120, 160, seed=31), n)
    frames = torch.from_numpy(pool).to(DEV)
    rng = np.random.default_rng(6)
    idx_a, idx_b = (rng.integers(0, 3, n).astype(np.int32) for _ in range(2))
    want_a = np.empty_like(pool)
    want_b = np.empty_like(pool)
    for c in range(3):
        want_a[idx_a == c] = oracle.process_batch(pool[idx_a == c], cfgs[c])
        want_b[idx_b == c] = oracle.process_batch(pool[idx_b == c], cfgs[c])
    ta, tb = torch.from_numpy(idx_a).to(DEV), torch.from_numpy(idx_b).to(DEV)
    # queued behind work on the caller's stream: the frames and the indices are written there first
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        f2 = torch.zeros_like(frames)
        f2.copy_(frames)
        t2 = torch.full_like(ta, 7)
        t2.copy_(ta)
        out, _ = comp.process_device(f2, t2)
    s.synchronize()
    assert np.array_equal(out.cpu().numpy(), want_a)
    # 30+ back-to-back calls with alternating indices
    outs = [comp.process_device(frames, ta if i % 2 == 0 else tb)[0] for i in range(32)]
    torch.cuda.synchronize()
    for i, o in enumerate(outs):
        assert np.array_equal(o.cpu().numpy(), want_a if i % 2 == 0 else want_b), i
    # CUDA graph: captured once, replayed with another index tensor in the same buffer
    idx_buf = ta.clone()
    out_buf = torch.empty_like(frames)
    gs = torch.cuda.Stream()
    gs.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(gs):
        comp.process_device(frames, idx_buf, out_u8=out_buf)           # first call of the size: scratch allocated outside the capture
    torch.cuda.current_stream().wait_stream(gs)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        comp.process_device(frames, idx_buf, out_u8=out_buf)
    for idx_t, want in ((tb, want_b), (ta, want_a), (tb, want_b)):
        idx_buf.copy_(idx_t)
        out_buf.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(out_buf.cpu().numpy(), want)
    # the caller's current device is left alone
    before = torch.cuda.current_device()
    comp.process_device(frames[:10], ta[:10])
    assert torch.cuda.current_device() == before
    comp.onShutdown()


def test_setting_configurations(golden_images):
    full, exotic, edge = _cfgs(golden_images, ["full_house", "exotic", "edge_only"])
    single = ImgPreprocessing(full, device=0)
    frames = synth.frame_pool(16, 120, 160, seed=2)
    p = (nat.PreprocParams * 2)(nat.preproc_params_from_cfg(exotic), nat.preproc_params_from_cfg(edge))
    nat.check(single.ctx.lib.trs_set_preproc_configs(single.ctx.handle, p, 2), "trs_set_preproc_configs")
    u8, _ = single.process_device(torch.from_numpy(frames).to(DEV))
    assert np.array_equal(u8.cpu().numpy(), oracle.process_batch(frames, full))      # trs_preprocess keeps the single configuration
    # bad arguments: ValueError, never a fault
    with pytest.raises(ValueError):
        nat.check(single.ctx.lib.trs_set_preproc_configs(single.ctx.handle, p, 0), "trs_set_preproc_configs")
    many = (nat.PreprocParams * 17)(*([nat.preproc_params_from_cfg(full)] * 17))
    with pytest.raises(ValueError):
        nat.check(single.ctx.lib.trs_set_preproc_configs(single.ctx.handle, many, 17), "trs_set_preproc_configs")
    with pytest.raises(ValueError):
        MultiTrackImgPreprocessing([full] * 17, device=0)
    with pytest.raises(ValueError):
        MultiTrackImgPreprocessing([], device=0)
    bad = dict(full, preprocessing_color_filter_enabled=True)
    bad['preprocessing_color_filter_destination_channels'] = [3] * len(full['preprocessing_color_filter_hsvs'])
    with pytest.raises(ValueError, match="configuration 1"):
        MultiTrackImgPreprocessing([full, bad], device=0)
    single.onShutdown()
    comp = MultiTrackImgPreprocessing([full, exotic], device=0)
    f = torch.from_numpy(frames).to(DEV)
    with pytest.raises(ValueError):
        comp.process_device(f, torch.zeros(16, dtype=torch.float32, device=DEV))
    with pytest.raises(ValueError):
        comp.process_device(f, torch.zeros(15, dtype=torch.int32, device=DEV))
    with pytest.raises(ValueError):
        comp.process_device(f, torch.zeros(16, dtype=torch.int32))                       # index tensor on the host
    with pytest.raises(ValueError):
        comp.process_device(f[..., :2].contiguous(), torch.zeros(16, dtype=torch.int32, device=DEV))
    with pytest.raises(ValueError):
        comp.step(frames, np.zeros(16, np.float32))
    # the context still works after the refusals
    u8, _ = comp.process_device(f, torch.ones(16, dtype=torch.int32, device=DEV))
    assert np.array_equal(u8.cpu().numpy(), oracle.process_batch(frames, exotic))
    comp.onShutdown()
