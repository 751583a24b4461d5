#!/usr/bin/env python
"""Tub recording on the GPU: the JPEG encoder behind trs_jpeg_encode, alone and in the recording pipeline, against Pillow on every host
core.  Prints one JSON line (and writes it to --out).

  encoder       N device frames -> packed files on the device (both passes, the host offset scan between them), at 65,536 x 120x160
                and 16,384 x 240x320, quality 75; the files copied to the host separately.  HBM bound: the frames are read once per
                pass and the files written once, over 7.7 TB/s (data-sheet HBM3e bandwidth of one B200).
  pipeline      pinned host frames -> H2D -> process_device (the chain) -> trs_jpeg_encode -> trs_jpeg_encode_copy -> host bytes, in
                chunks of 8,192 on one stream; against the existing leg in the same run: process_host with the processed u8 frames
                back on the host (the pixels a host-side Pillow recorder would have to encode).
  pillow        Image.fromarray(f).save(BytesIO, "JPEG") (the recorder's call) in one process per host core.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_BPS = 7.7e12


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def frames_for(n, h, w, seed):
    from triton_racer_sim_b200 import synth
    pool = synth.frame_pool(64, h, w, seed=seed)
    return np.ascontiguousarray(np.concatenate([pool] * ((n + 63) // 64))[:n])


def time_encoder(n, h, w, reps, quality=75):
    import ctypes as C
    from triton_racer_sim_b200 import _native as nat
    frames = torch.from_numpy(frames_for(n, h, w, seed=h + w)).cuda(0)
    ctx = nat.Context(0)
    offs = np.zeros(n + 1, np.uint64)
    st = torch.cuda.current_stream(0)
    sp = C.c_void_p(st.cuda_stream)

    def enc():
        nat.check(ctx.lib.trs_jpeg_encode(ctx.handle, C.c_void_p(frames.data_ptr()), n, h, w, quality, C.c_void_p(offs.ctypes.data), sp),
                  "trs_jpeg_encode")
    enc()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        enc()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    out_bytes = int(offs[n])
    blob = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    t0 = time.perf_counter()
    nat.check(ctx.lib.trs_jpeg_encode_copy(ctx.handle, C.c_void_p(blob.data_ptr()), C.c_ulonglong(out_bytes), sp), "trs_jpeg_encode_copy")
    t_copy = time.perf_counter() - t0
    ctx.close()
    in_bytes = n * h * w * 3
    t = float(np.median(times))
    hbm_s = (2 * in_bytes + out_bytes) / HBM_BPS
    return {"n": n, "h": h, "w": w, "quality": quality, "median_s": t, "min_s": min(times), "max_s": max(times),
            "records_per_s": n / t, "in_bytes": in_bytes, "out_bytes": out_bytes, "bytes_per_record": out_bytes / n,
            "hbm_bound_s": hbm_s, "share_of_hbm_bound": hbm_s / t, "copy_s": t_copy, "copy_gbps": out_bytes / t_copy / 1e9}


def time_pipeline(n, chunk, reps):
    import ctypes as C
    from triton_racer_sim_b200 import ImgPreprocessing
    from triton_racer_sim_b200 import _native as nat
    from triton_racer_sim_b200.config import full_house_config
    h, w = 120, 160
    host = frames_for(n, h, w, seed=5)
    pinned = torch.from_numpy(host).pin_memory()
    comp = ImgPreprocessing(full_house_config(), device=0)
    ctx = nat.Context(0)
    st = torch.cuda.current_stream(0)
    sp = C.c_void_p(st.cuda_stream)
    out_blob = torch.empty(n * 20000, dtype=torch.uint8).pin_memory()          # room for the files of every record
    offs = np.zeros(chunk + 1, np.uint64)

    def record():
        pos = 0
        for c0 in range(0, n, chunk):
            cn = min(chunk, n - c0)
            dev = pinned[c0:c0 + cn].cuda(0, non_blocking=True)
            u8, _ = comp.process_device(dev, want_f32=False)
            nat.check(ctx.lib.trs_jpeg_encode(ctx.handle, C.c_void_p(u8.data_ptr()), cn, h, w, 75, C.c_void_p(offs.ctypes.data), sp),
                      "trs_jpeg_encode")
            nb = int(offs[cn])
            if pos + nb > out_blob.numel():
                raise RuntimeError("host buffer too small for the recorded files")
            nat.check(ctx.lib.trs_jpeg_encode_copy(ctx.handle, C.c_void_p(out_blob.data_ptr() + pos), C.c_ulonglong(nb), sp),
                      "trs_jpeg_encode_copy")
            pos += nb
        return pos

    u8_host = np.empty_like(host)
    u8_pinned = torch.empty(host.shape, dtype=torch.uint8).pin_memory().numpy()

    def leg(out):
        comp.process_host(pinned.numpy(), out_u8=out)

    record(); leg(u8_host); leg(u8_pinned)
    res = {"n": n, "h": h, "w": w, "chunk": chunk}
    for name, fn in (("record_gpu_encode", record), ("u8_d2h_pageable", lambda: leg(u8_host)), ("u8_d2h_pinned", lambda: leg(u8_pinned))):
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
            if name == "record_gpu_encode":
                res["record_out_bytes"] = r
        t = float(np.median(ts))
        res[name] = {"median_s": t, "records_per_s": n / t}
    # the recorder's files from the pipeline equal Pillow's of the same processed frames (first chunk)
    import oracle
    from PIL import Image
    want = oracle.process_batch(host[:16], full_house_config())
    files = []
    for f in want:
        b = io.BytesIO(); Image.fromarray(f).save(b, "JPEG"); files.append(b.getvalue())
    res["pipeline_files_equal_pillow"] = out_blob[:sum(len(f) for f in files)].numpy().tobytes() == b"".join(files)
    comp.onShutdown(); ctx.close()
    return res


def _pil_worker(args):
    from PIL import Image
    h, w, n, seed = args
    from triton_racer_sim_b200 import synth
    pool = synth.frame_pool(16, h, w, seed=seed)
    t0 = time.perf_counter()
    for k in range(n):
        b = io.BytesIO()
        Image.fromarray(pool[k % 16]).save(b, "JPEG")
    return time.perf_counter() - t0


def time_pillow(per_proc):
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    with mp.get_context("spawn").Pool(cores) as p:
        p.map(_pil_worker, [(120, 160, 50, k) for k in range(cores)])                 # warm-up: imports in every worker
        t0 = time.perf_counter()
        p.map(_pil_worker, [(120, 160, per_proc, k) for k in range(cores)])
        wall = time.perf_counter() - t0
    one = _pil_worker((120, 160, per_proc, 0))
    return {"cores": cores, "records": cores * per_proc, "wall_s": wall, "records_per_s": cores * per_proc / wall,
            "one_thread_records_per_s": per_proc / one}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a rehearsal of the script, not a measurement)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU encoder: there is no CPU path"
    res = {"tool": "jpeg_encode_bench", "card": card(), "torch": torch.__version__}
    sizes = [(256, 120, 160), (64, 240, 320)] if a.small else [(65536, 120, 160), (16384, 240, 320)]
    res["encoder"] = [time_encoder(n, h, w, a.reps) for n, h, w in sizes]
    res["pipeline"] = time_pipeline(512 if a.small else 65536, 128 if a.small else 8192, a.reps)
    res["pillow"] = time_pillow(50 if a.small else 2000)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
