#!/usr/bin/env python
"""Preprocessing of a batch whose frames come with K = 2, 4, 8 configurations (drawn from the golden ones, and K copies of full_house, which
isolates the overhead from the configurations' own costs), frames assigned to configurations at random and in sorted order, u8 and f32
outputs.  Times four ways of giving every frame its own configuration's answer:

  multi   MultiTrackImgPreprocessing: one stream-ordered call (trs_preprocess_configs)
  split   the group sizes to the host (one sync), each group gathered with index_select, one ImgPreprocessing call per group, outputs
          scattered back
  k_full  K ImgPreprocessing calls over the whole batch, torch.where picks each frame's configuration (K times the work, no sync)
  ideal   the sum of each group's time when it is run alone as a contiguous batch (what K separate fleets would cost)

Sizes: 65,536 frames at 120x160 and 16,384 at 240x320 (each 22.6 GB of traffic per call: far beyond the 126 MB of L2), and 4,096 frames at
120x160 (one step of a simulator fleet, where the K launches with few frames each show).  The outputs of multi, split and k_full are compared
bit for bit before anything is timed.  torch.profiler records once which kernels multi and each group's single-configuration call launch.
The card's name and power limit are read in the same run.
usage: tools/preprocess_configs_bench.py [--reps R] [--out FILE]  -> one JSON object (stdout, and FILE if given)"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from tests.helpers import cfg_for, image_cases
from triton_racer_sim_b200 import ImgPreprocessing, MultiTrackImgPreprocessing, synth

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("no CUDA device: this measures the GPU path and has no CPU path")
DEV = "cuda:0"
golden = np.load(os.path.join(ROOT, "tests", "golden", "images.npz"))
CASES = image_cases(golden)
ORDER = ["full_house", "exotic", "dyn_contrast", "edge_only", "colour_only", "edge_tight", "adjust_only"]


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type.name == "CUDA" and "Memset" not in e.name and "Memcpy" not in e.name]
    return [n for n in names if "k_" in n]


def config_sets(k):
    return {"golden": [cfg_for(CASES[ORDER[j % len(ORDER)]]) for j in range(k)], "full_house_copies": [cfg_for(CASES["full_house"])] * k}


_frames = {}


def run_case(n, h, w, k, set_name, cfgs, assign, launches=False):
    if (n, h, w) not in _frames:
        _frames.clear()
        _frames[(n, h, w)] = torch.from_numpy(synth.expand_numpy(synth.frame_pool(64, h, w, seed=7 + h), n)).to(DEV)
    frames = _frames[(n, h, w)]
    rng = np.random.default_rng(n + k)
    idx_np = rng.integers(0, k, n).astype(np.int32)
    if assign == "sorted":
        idx_np = np.sort(idx_np)
    idx = torch.from_numpy(idx_np).to(DEV)
    multi_c = MultiTrackImgPreprocessing(cfgs, device=0, normalised_key="n")
    singles = [ImgPreprocessing(c, device=0, normalised_key="n") for c in cfgs]
    out_u8, out_f32 = torch.empty_like(frames), torch.empty(frames.shape, dtype=torch.float32, device=DEV)
    tmp_u8, tmp_f32 = torch.empty_like(frames), torch.empty(frames.shape, dtype=torch.float32, device=DEV)

    def multi():
        return multi_c.process_device(frames, idx, out_u8=out_u8, out_f32=out_f32)

    def split():
        counts = torch.bincount(idx, minlength=k).cpu().tolist()                 # the host sync
        order = torch.argsort(idx, stable=True)
        a = 0
        for c in range(k):
            if counts[c]:
                rows = order[a:a + counts[c]]
                u8, f32 = singles[c].process_device(frames.index_select(0, rows))
                out_u8.index_copy_(0, rows, u8)
                out_f32.index_copy_(0, rows, f32)
            a += counts[c]
        return out_u8, out_f32

    def k_full():
        m = idx.view(n, 1, 1, 1)
        for c in range(k):
            singles[c].process_device(frames, out_u8=tmp_u8, out_f32=tmp_f32)
            torch.where(m == c, tmp_u8, out_u8, out=out_u8)
            torch.where(m == c, tmp_f32, out_f32, out=out_f32)
        return out_u8, out_f32

    results = {}
    for name, fn in (("multi", multi), ("split", split), ("k_full", k_full)):
        out_u8.zero_()
        out_f32.zero_()
        fn()
        torch.cuda.synchronize()
        results[name] = (out_u8.clone(), out_f32.view(torch.int32).clone())
    same = all(torch.equal(results["multi"][0], r[0]) and torch.equal(results["multi"][1], r[1]) for r in results.values())
    del results
    if not same:
        sys.exit(f"n={n} {h}x{w} K={k} {set_name} {assign}: the three ways disagree; nothing timed")
    run = {"n": n, "h": h, "w": w, "k": k, "configs": set_name, "assign": assign, "identical": True}
    for name, fn in (("multi", multi), ("split", split), ("k_full", k_full)):
        t_s = timed(fn, args.reps)
        run[name] = {"ms": round(t_s * 1e3, 4), "frames_per_s": n / t_s}
    # ideal: each group alone, contiguous, outputs in its own buffers
    ideal = 0.0
    groups = []
    for c in range(k):
        rows = torch.from_numpy(np.flatnonzero(idx_np == c)).to(DEV)
        if len(rows) == 0:
            continue
        g = frames.index_select(0, rows)
        gu8, gf32 = torch.empty_like(g), torch.empty(g.shape, dtype=torch.float32, device=DEV)
        ideal += timed(lambda: singles[c].process_device(g, out_u8=gu8, out_f32=gf32), args.reps)
        groups.append((c, g, gu8, gf32))
    run["ideal"] = {"ms": round(ideal * 1e3, 4), "frames_per_s": n / ideal}
    run["multi_over_ideal"] = run["multi"]["ms"] / run["ideal"]["ms"]
    run["split_over_multi"] = run["split"]["ms"] / run["multi"]["ms"]
    run["k_full_over_multi"] = run["k_full"]["ms"] / run["multi"]["ms"]
    if launches:
        run["launches_multi"] = kernels_of(multi)
        run["launches_single"] = {str(c): kernels_of(lambda: singles[c].process_device(g, out_u8=gu8, out_f32=gf32)) for c, g, gu8, gf32 in groups}
    del groups
    multi_c.onShutdown()
    for s in singles:
        s.onShutdown()
    del frames, out_u8, out_f32, tmp_u8, tmp_f32
    torch.cuda.empty_cache()
    return run


out = {"card": card(), "reps": args.reps, "bytes_per_frame_120x160": 120 * 160 * 3 * 6, "runs": []}
for n, h, w in ((65_536, 120, 160), (16_384, 240, 320), (4_096, 120, 160)):
    for k in (2, 4, 8):
        for set_name, cfgs in config_sets(k).items():
            for assign in ("random", "sorted"):
                r = run_case(n, h, w, k, set_name, cfgs, assign, launches=(k == 8 and set_name == "golden" and assign == "sorted" and n != 4_096))
                print(json.dumps({x: r[x] for x in ("n", "h", "w", "k", "configs", "assign", "multi_over_ideal", "split_over_multi", "k_full_over_multi")}),
                      file=sys.stderr, flush=True)
                out["runs"].append(r)
text = json.dumps(out)
print(text)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
