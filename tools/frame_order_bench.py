#!/usr/bin/env python
"""ImgPreprocessing.process_device on bench.py's own batches (full-house configuration), the same frames in three orders:

  bench     bench.py's order: frame f is pool frame f % P, so its kind (synth.frame_pool: noise / smooth / smooth / track) is f % 4
  shuffled  a seeded random permutation
  sorted    sorted by kind (all noise frames first)

for the headline (65,536 x 120x160, u8 + f32) and the two 240x320 configurations (mask u8, chain u8 + f32) at 16,384 and 65,536 frames.
A kernel whose frame schedule is fixed by frame index runs each order at a different speed when frames cost different amounts; one that
hands out frames on demand runs them alike.

Before anything is timed, every order's outputs, permuted back, are compared byte for byte with the bench order's (u8 directly; f32 as
exactly u8 / 255 of the same call, which with equal u8 outputs makes the f32 outputs equal too), and the statistics counters of a
collect_stats=True run of each order must be equal (all but hyst_sweeps, which depends on timing in every build and is reported).  Then the three orders alternate within each of --steps rounds (CUDA events per call)
after --warmup rounds.  The card's name, power limit and maximum SM clock are read in the same run.

usage: tools/frame_order_bench.py [--steps S] [--warmup W] [--only NAME ...] [--out FILE]  -> one JSON line (stdout, and FILE if given)"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from triton_racer_sim_b200 import ImgPreprocessing, synth
from triton_racer_sim_b200.config import full_house_config

CASES = [  # name, h, w, frames, pool size (bench.py's), f32 output
    ("full_chain_120x160", 120, 160, 65536, 1024, True),
    ("full_house_mask_240x320_16k", 240, 320, 16384, 256, False),
    ("full_chain_240x320_16k", 240, 320, 16384, 256, True),
    ("full_house_mask_240x320", 240, 320, 65536, 256, False),
    ("full_chain_240x320", 240, 320, 65536, 256, True),
]
ORDERS = ("bench", "shuffled", "sorted")

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--only", nargs="*", default=None)
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("no CUDA device: this measures the GPU path and has no CPU path")
DEV = torch.device("cuda", 0)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def permutations(n):
    """order[k] = bench-order frame placed at position k."""
    rng = np.random.default_rng(20261020 + n)
    kind = np.arange(n) % 4
    return {"bench": np.arange(n), "shuffled": rng.permutation(n), "sorted": np.argsort(kind, kind="stable")}


def check_f32(u8, f32, chunk=2048):
    for s in range(0, u8.shape[0], chunk):
        if not torch.equal(f32[s:s + chunk], u8[s:s + chunk].float() / 255.0):
            return False
    return True


out = {"card": card(), "steps": args.steps, "warmup": args.warmup, "cases": []}
cfg = full_house_config()
pools = {}
for name, h, w, n, psize, f32 in CASES:
    if args.only and name not in args.only:
        continue
    if (h, w) not in pools:
        pools = {(h, w): torch.from_numpy(synth.frame_pool(psize, h, w)).to(DEV)}
    base = synth.expand_torch(pools[(h, w)], n)
    perms = {o: torch.from_numpy(p).to(DEV) for o, p in permutations(n).items()}
    inputs = {o: (base if o == "bench" else base.index_select(0, perms[o])) for o in ORDERS}
    o_u8 = torch.empty_like(base)
    o_f32 = torch.empty(base.shape, dtype=torch.float32, device=DEV) if f32 else None
    comp = ImgPreprocessing(cfg, device=0)
    comp_s = ImgPreprocessing(cfg, device=0, collect_stats=True)

    # ---- results first: outputs permuted back and counters, every order against the bench order
    comp.process_device(inputs["bench"], out_u8=o_u8, out_f32=o_f32, want_f32=f32)
    ref = o_u8.clone()
    identical = check_f32(o_u8, o_f32) if f32 else True
    stats = {}
    for o in ORDERS:
        if o != "bench":
            comp.process_device(inputs[o], out_u8=o_u8, out_f32=o_f32, want_f32=f32)
            for s in range(0, n, 4096):
                identical &= torch.equal(o_u8[s:s + 4096], ref.index_select(0, perms[o][s:s + 4096]))
            if f32:
                identical &= check_f32(o_u8, o_f32)
        comp_s.process_device(inputs[o], out_u8=o_u8, out_f32=o_f32, want_f32=f32)
        stats[o] = comp_s.stats()
    result = {o: {k: v for k, v in stats[o].items() if k != "hyst_sweeps"} for o in ORDERS}
    same_stats = all(result[o] == result["bench"] for o in ORDERS)
    del ref
    if not (identical and same_stats):
        sys.exit(f"{name}: the orders disagree (outputs identical: {identical}, counters equal: {same_stats}); nothing timed")

    # ---- timing: the three orders alternate within each round
    ev = {o: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] for o in ORDERS}
    for r in range(args.warmup + args.steps):
        for o in ORDERS:
            if r >= args.warmup:
                ev[o][r - args.warmup][0].record()
            comp.process_device(inputs[o], out_u8=o_u8, out_f32=o_f32, want_f32=f32)
            if r >= args.warmup:
                ev[o][r - args.warmup][1].record()
    torch.cuda.synchronize()
    case = {"name": name, "frames": n, "h": h, "w": w, "f32": f32, "outputs_identical": True, "counters_equal": True,
            "counters": stats["bench"], "hyst_sweeps": {o: stats[o]["hyst_sweeps"] for o in ORDERS}}
    for o in ORDERS:
        ms = np.array([a.elapsed_time(b) for a, b in ev[o]])
        case[o] = {"ms_median": round(float(np.median(ms)), 4), "ms_min": round(float(ms.min()), 4), "ms_max": round(float(ms.max()), 4),
                   "frames_per_s": n / (float(np.median(ms)) * 1e-3)}
    case["shuffled_speedup_vs_bench"] = case["bench"]["ms_median"] / case["shuffled"]["ms_median"]
    case["sorted_speedup_vs_bench"] = case["bench"]["ms_median"] / case["sorted"]["ms_median"]
    out["cases"].append(case)
    comp.onShutdown()
    comp_s.onShutdown()
    del base, inputs, perms, o_u8, o_f32
    torch.cuda.empty_cache()

text = json.dumps(out)
print(text)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
