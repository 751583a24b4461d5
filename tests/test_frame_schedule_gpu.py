"""The store-warp kernels (k_preprocess_sw, k_preprocess_bsw) hand out frames on demand from a per-launch counter (preproc_fast.cuh
draw_frames): which CTA processes which frame depends on timing.  Results must not.

  * order invariance: a batch and a seeded permutation of it give the same outputs (permuted back) and the same counters, for every
    converted kernel and for frame counts around the grid size (n = 1, n < grid, n = grid + 1, and a ragged n with >= 5 frames per CTA);
  * counter reset: many calls of varying size back to back on one stream, each checked against the oracle: a counter left over from the
    call before would leave frames unprocessed;
  * concurrency: two components (two contexts) at once on two streams, and the host pipeline's three streams over many chunks.

The grid restates trs_api.cu: two CTAs per SM for both kernels (grid = min(n, 2 x SMs))."""
import numpy as np
import pytest
import torch

import oracle
from tests.helpers import cfg_for, image_cases
from triton_racer_sim_b200 import ImgPreprocessing, synth
from triton_racer_sim_b200 import _native as nat

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
DEV = "cuda:0"
CTAS_PER_SM = 2

# (h, w, configuration): the kernel launch_preprocess picks for it
KERNELS = {
    "sw_120x160_static": (120, 160, "full_house"),          # k_preprocess_sw<2, DEFAULT_F0, DEFAULT_F1, 120, 160>
    "sw_100x160_any_size": (100, 160, "full_house"),        # k_preprocess_sw<2, DEFAULT_F0, DEFAULT_F1, 0, 0>
    "sw_run_time_ranges_table": (120, 160, "exotic"),       # k_preprocess_sw<2, -1, -1, 0, 0>, dynamic brightness / contrast table
    "bsw_240x320": (240, 320, "full_house"),                # k_preprocess_bsw<..., LUT = false>
    "bsw_240x320_table": (240, 320, "dyn_contrast"),        # k_preprocess_bsw<..., LUT = true>
}


@pytest.fixture(scope="module")
def grid():
    ctx = nat.Context(0)
    g = CTAS_PER_SM * ctx.sm_count
    ctx.close()
    return g


def counters(st):
    """Every counter but the timers and the hysteresis sweeps: how many rounds the store warps need depends on how far the compute warps'
    per-band relaxation got, which is timing (test_batched_loops_gpu.py excludes it for the same reason)."""
    return {k: v for k, v in st.items() if not k.startswith("t_") and k != "hyst_sweeps"}


def describe(got, want):
    bad = np.argwhere(got != want)
    return f"{len(bad)} of {got.size} differ; first at {bad[:5].tolist()}"


def frames_for(h, w, n, seed):
    """Pool kinds repeat with period 4 (synth.frame_pool), as in bench.py's batches: a fixed stride would give a CTA one kind only."""
    return synth.expand_numpy(synth.frame_pool(64, h, w, seed=seed), n, start=5)


def run(comp, frames_dev, f32=True):
    u8, f = comp.process_device(frames_dev, want_f32=f32)
    return u8.cpu().numpy(), (f.cpu().numpy() if f is not None else None), counters(comp.stats())


@pytest.mark.parametrize("size", ["one", "below_grid", "grid_plus_one", "ragged_5_per_cta"])
@pytest.mark.parametrize("kernel", list(KERNELS))
def test_order_invariance(golden_images, grid, kernel, size):
    h, w, cname = KERNELS[kernel]
    n = {"one": 1, "below_grid": grid // 3 + 1, "grid_plus_one": grid + 1, "ragged_5_per_cta": 5 * grid + 37}[size]
    cfg = cfg_for(image_cases(golden_images)[cname])
    frames = frames_for(h, w, n, seed=n + h)
    perm = np.random.default_rng(n).permutation(n)
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    u8, f32, st = run(comp, torch.from_numpy(frames).to(DEV))
    pu8, pf32, pst = run(comp, torch.from_numpy(np.ascontiguousarray(frames[perm])).to(DEV))
    comp.onShutdown()
    want = oracle.process_batch(frames, cfg)
    assert np.array_equal(u8, want), f"{kernel} n={n}: {describe(u8, want)}"
    assert np.array_equal(pu8, u8[perm]), f"{kernel} n={n} permuted u8: {describe(pu8, u8[perm])}"
    assert np.array_equal(pf32, f32[perm]), f"{kernel} n={n} permuted f32"
    assert pst == st, f"{kernel} n={n}: counters {pst} != {st}"
    assert st["frames"] == n


def test_counter_reset_between_back_to_back_calls(golden_images, grid):
    """34 calls on one stream and one context, nothing synchronised in between: both kernels (they share the context's counter), sizes
    from 1 to 6 grids, every small call right after a large one.  Each call's output is checked against the oracle afterwards."""
    cfg = cfg_for(image_cases(golden_images)["full_house"])
    sizes = [6 * grid + 5, grid // 2, 1, 3 * grid - 7, grid + 1, 17, 2 * grid, grid - 1]
    big = {(120, 160): frames_for(120, 160, 6 * grid + 5, seed=1), (240, 320): frames_for(240, 320, 2 * grid, seed=2)}
    want = {hw: oracle.process_batch(f, cfg) for hw, f in big.items()}
    dev = {hw: torch.from_numpy(f).to(DEV) for hw, f in big.items()}
    comp = ImgPreprocessing(cfg, device=0)
    calls = []
    for k in range(34):
        hw = (240, 320) if k % 5 == 4 else (120, 160)
        n = min(sizes[k % len(sizes)], dev[hw].shape[0])
        s = (37 * k) % (dev[hw].shape[0] - n + 1)
        out = torch.full((n,) + dev[hw].shape[1:], 7, dtype=torch.uint8, device=DEV)
        comp.process_device(dev[hw][s:s + n], out_u8=out, want_f32=False)
        calls.append((hw, s, n, out))
    torch.cuda.synchronize()
    comp.onShutdown()
    for k, (hw, s, n, out) in enumerate(calls):
        got = out.cpu().numpy()
        assert np.array_equal(got, want[hw][s:s + n]), f"call {k} ({n} frames of {hw}): {describe(got, want[hw][s:s + n])}"


def test_two_contexts_at_once_on_two_streams(golden_images, grid):
    """The headline configuration on two components (each its own context and counter), launched on two streams so the launches overlap."""
    cfg = cfg_for(image_cases(golden_images)["full_house"])
    n = 8 * grid + 3
    frames = [frames_for(120, 160, n, seed=10 + i) for i in range(2)]
    comps = [ImgPreprocessing(cfg, device=0) for _ in range(2)]
    dev = [torch.from_numpy(f).to(DEV) for f in frames]
    streams = [torch.cuda.Stream(device=DEV) for _ in range(2)]
    outs = [torch.empty_like(d) for d in dev]
    f32 = [torch.empty(d.shape, dtype=torch.float32, device=DEV) for d in dev]
    torch.cuda.synchronize()
    for _ in range(3):
        for i in range(2):
            with torch.cuda.stream(streams[i]):
                comps[i].process_device(dev[i], out_u8=outs[i], out_f32=f32[i], want_f32=True)
    torch.cuda.synchronize()
    for i in range(2):
        want = oracle.process_batch(frames[i], cfg)
        got = outs[i].cpu().numpy()
        assert np.array_equal(got, want), f"component {i}: {describe(got, want)}"
        assert np.array_equal(f32[i].cpu().numpy(), oracle.normalise(want)), f"component {i} f32"
        comps[i].onShutdown()


@pytest.mark.parametrize("h,w", [(120, 160), (240, 320)])
def test_host_pipeline_pinned_many_chunks(golden_images, h, w):
    """trs_preprocess_host from pinned buffers (so the copies are asynchronous and the three streams' kernels really overlap), the default
    48 MB chunks with several frames per CTA in each, >= 7 chunks and a ragged last one: every staging set's counter is in use at once."""
    cfg = cfg_for(image_cases(golden_images)["full_house"])
    fb = h * w * 3
    chunk = ((48 << 20) // fb + 3) & ~3                             # trs_api.cu host chunking (TrsSwitches::host_chunk_bytes)
    n = 7 * chunk + chunk // 3
    src = frames_for(h, w, n, seed=h)
    frames = torch.empty(src.shape, dtype=torch.uint8, pin_memory=True).numpy()
    frames[...] = src
    out = torch.empty(src.shape, dtype=torch.uint8, pin_memory=True).numpy()
    comp = ImgPreprocessing(cfg, device=0, collect_stats=True)
    got, _ = comp.process_host(frames, out_u8=out)
    st = counters(comp.last_stats)
    comp.onShutdown()
    want = oracle.process_batch(src, cfg)
    assert np.array_equal(got, want), describe(got, want)
    assert st["frames"] == n
