#!/usr/bin/env python
"""Nearest waypoint for 1,048,576 cars over K = 2, 4, 8 tracks (the shipped centre lines and copies shifted away from them), cars assigned to
tracks at random or in sorted order.  Times four ways of getting every car its own track's answer:

  multi   MultiTrackLocationTracker: one stream-ordered call (trs_locate_tracks)
  k_full  K LocationTrackers over the whole batch, then torch.where picks each car's track (K times the work, no sync)
  split   the batch split by track on the host's knowledge of the group sizes (one sync), one LocationTracker call per group, results
          scattered back
  single  for scale: one LocationTracker on 1,048,576 cars of one track (the single-track rate)

The outputs of multi, k_full and split are compared bit for bit before anything is timed.  The card's name and power limit are read in the same
run.  usage: tools/locate_tracks_bench.py [--n N] [--reps R] [--out FILE]  -> one JSON object (stdout, and FILE if given)"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from triton_racer_sim_b200 import LocationTracker, MultiTrackLocationTracker, synth

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=1 << 20)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("no CUDA device: this measures the GPU path and has no CPU path")
n = args.n
DEV = "cuda:0"
golden = np.load(os.path.join(ROOT, "tests", "golden", "tracks.npz"))
base = [golden["wp/generated_track"], golden["wp/mountain_track"]]


def track_set(k):
    """The two shipped lines, then copies shifted by 1 km steps along x and z (their own cells, no overlap)."""
    return [base[j % 2] + np.array([1000.0 * (j // 2), 0.0, 1000.0 * (j // 2)]) for j in range(k)]


def timed(fn, reps):
    for _ in range(3):
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


out = {"cars": n, "card": card(), "reps": args.reps, "runs": []}
for k in (2, 4, 8):
    lines = track_set(k)
    mt = MultiTrackLocationTracker(lines, device=0)
    singles = [LocationTracker(line, device=0) for line in lines]
    rng = np.random.default_rng(k)
    per_track = [torch.from_numpy(synth.car_states(line, n, seed=100 + t)[0]).to(DEV) for t, line in enumerate(lines)]
    for assign in ("random", "sorted"):
        trk_np = rng.integers(0, k, n).astype(np.int32)
        if assign == "sorted":
            trk_np = np.sort(trk_np)
        trk = torch.from_numpy(trk_np).to(DEV)
        pick = torch.arange(n, device=DEV)
        xyz = torch.zeros((n, 3), dtype=torch.float64, device=DEV)
        for t in range(k):
            m = trk == t
            xyz[m] = per_track[t][pick[m]]
        xyz = xyz.contiguous()

        def multi():
            return mt.locate_device(xyz, trk)

        def k_full():
            idx = torch.empty(n, dtype=torch.int32, device=DEV)
            seg = torch.empty(n, dtype=torch.float64, device=DEV)
            for t in range(k):
                i, s = singles[t].locate_device(xyz)
                m = trk == t
                idx = torch.where(m, i, idx)
                seg = torch.where(m, s, seg)
            return idx, seg

        def split():
            counts = torch.bincount(trk, minlength=k).cpu().tolist()              # the host sync
            order = torch.argsort(trk, stable=True)
            idx = torch.empty(n, dtype=torch.int32, device=DEV)
            seg = torch.empty(n, dtype=torch.float64, device=DEV)
            a = 0
            for t in range(k):
                if counts[t]:
                    rows = order[a:a + counts[t]]
                    i, s = singles[t].locate_device(xyz.index_select(0, rows))
                    idx[rows] = i
                    seg[rows] = s
                a += counts[t]
            return idx, seg

        results = {name: fn() for name, fn in (("multi", multi), ("k_full", k_full), ("split", split))}
        torch.cuda.synchronize()
        same = all(torch.equal(results["multi"][0], r[0]) and torch.equal(results["multi"][1].view(torch.int64), r[1].view(torch.int64))
                   for r in results.values())
        if not same:
            sys.exit(f"K={k} {assign}: the three ways disagree; nothing timed")
        run = {"k": k, "assign": assign, "identical": same}
        for name, fn in (("multi", multi), ("k_full", k_full), ("split", split)):
            t_s = timed(fn, args.reps)
            run[name] = {"ms": round(t_s * 1e3, 4), "cars_per_s": n / t_s}
        run["speedup_vs_k_full"] = run["k_full"]["ms"] / run["multi"]["ms"]
        run["speedup_vs_split"] = run["split"]["ms"] / run["multi"]["ms"]
        out["runs"].append(run)
    mt.onShutdown()
    for s in singles:
        s.onShutdown()
one = LocationTracker(base[0], device=0)
d = torch.from_numpy(synth.car_states(base[0], n, seed=4)[0]).to(DEV)
t_s = timed(lambda: one.locate_device(d), args.reps)
out["single_generated_track"] = {"ms": round(t_s * 1e3, 4), "cars_per_s": n / t_s}
one.onShutdown()
text = json.dumps(out)
print(text)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
