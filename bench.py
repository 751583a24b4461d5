#!/usr/bin/env python
"""bench.py — the hot path's headline number on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                       (the reference CPU path on the host cores)
    python bench.py ... --dump-outputs DIR                     (also write a fixed sample of the last timed step's outputs as DIR/*.npy)

A "step" is one pass of the fused observation chain (brightness/contrast -> HSV colour masks || 3-channel Canny ->
merge -> /255 float tensor) over one batch of synthetic 120x160 frames, sharded by env index with no data-path
collective.  Default workload = BASELINE.json's north-star configuration: 65,536 frames per GPU, u8 in, u8
`cam/processed_img` + f32 normalised tensor out (345,600 algorithmic bytes per frame, SURVEY.md §8(d)).
Rank 0 prints ONE JSON line.  Besides the headline keys it carries, measured by every rank on its own shard (max over ranks):
  stats_on                         the headline step with the per-step counters and their all-reduce inside the timed region
  e2e (+ pcie_probe, tub_mode)     host buffers through the Component API; the copy-only ceiling of the box at this rank count
  blocks.full_house_mask_240x320   BASELINE.json configs[2] at 65,536 frames per GPU
  blocks.full_chain_240x320        the full chain (u8 + f32 out) at 240x320, 65,536 frames per GPU
  blocks.full_pipeline_1M          configs[4]: 1,048,576 frames + car states per step over the N ranks (strong scaling)
  other_workloads                  the remaining configurations, rank 0 only
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (h, w, frames per GPU, want_u8, want_f32, algorithmic bytes per frame)
    "full_chain_120x160": (120, 160, 65536, True, True, 57600 + 57600 + 230400),
    "full_house_mask_240x320": (240, 320, 65536, True, False, 230400 + 230400),
    "full_chain_240x320": (240, 320, 65536, True, True, 230400 * 6),
    # BASELINE.json configs[4]: 1M frames + 1M car states per step over 8 GPUs = 131,072 of each per GPU; a step also runs the
    # nearest-waypoint lookup, the speed controller and the control multiplexer for the shard's cars (three more launches)
    "full_pipeline_1M_over_8": (120, 160, 131072, True, True, 57600 + 57600 + 230400),
}
METRIC = "preprocessed frames/sec (120x160), full observation chain"
METRICS = {"full_chain_120x160": METRIC, "full_house_mask_240x320": "preprocessed frames/sec (240x320), full-house colour + edge mask",
           "full_chain_240x320": "preprocessed frames/sec (240x320), full observation chain",
           "full_pipeline_1M_over_8": "preprocessed frames/sec (120x160), full observation pipeline incl. per-car lookup and control"}
KERNELS = {"full_chain_120x160": "trs::k_preprocess_sw<2,24,23,120,160>", "full_house_mask_240x320": "trs::k_preprocess_bsw<2,24,23,240,320,24,2>",
           "full_chain_240x320": "trs::k_preprocess_bsw<2,24,23,240,320,24,2>", "full_pipeline_1M_over_8": "trs::k_preprocess_sw<2,24,23,120,160>"}
NOTES = {
    "full_chain_120x160": "bound by the ALU pipe / issue slots and phase barriers, not by HBM: ten compute warps per CTA run strip walk, NMS and "
                          "hysteresis while two store warps stream the previous frame out (the SM -> L2 write port tops out at 29 B/clk); "
                          "see DESIGN.md 4.1 and profiles/",
    "full_house_mask_240x320": "6 algorithmic bytes per pixel: instruction bound by construction (SURVEY.md 8d); banded store-warp kernel, DESIGN.md 4.3",
    "full_chain_240x320": "18 algorithmic bytes per pixel like the 120x160 headline; banded store-warp kernel (frames do not fit shared memory whole), DESIGN.md 4.3",
    "full_pipeline_1M_over_8": "frames as full_chain_120x160; the per-car kernels (FP64 argmin over 1,185 waypoints, speed control, multiplexer) "
                               "add three launches per step and are counted in the step time but not in the algorithmic bytes",
}


_REAL_STDOUT = None
# --dump-outputs sample sizes: 32 frames of 240x320 with u8 and f32 outputs, both written as float32, are 59 MB (under 64 MB)
DUMP_FRAMES, DUMP_CARS = 32, 65536


def load_track(name: str):
    """One of the reference's two recorded centre lines (car_templates/track_data/*.json: 'generated_track' 1,185 points,
    'mountain_track' 2,664 points), as committed with the golden vectors (tests/golden/tracks.npz, key wp/<name>)."""
    import numpy as np
    with np.load(os.path.join(ROOT, "tests", "golden", "tracks.npz")) as z:
        return np.ascontiguousarray(z[f"wp/{name}"], np.float64)


def emit(line: dict):
    """The one JSON line, on the real stdout."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, start, groups):
    """Writes a fixed, seeded sample of rows of each output as out_dir/<name>.npy: int32 and float64 outputs as float64, the others as
    float32 (exact for u8 and f32).  groups: (index name, sample size, {name: device tensor with one row per frame or car}); the global
    index of each sampled row goes to out_dir/<index name>.npy, so that two builds can be compared output for output."""
    import numpy as np
    import torch
    arrays = {}
    for seed, (index_name, k, outputs) in enumerate(groups):
        outputs = {name: t for name, t in outputs.items() if t is not None}
        if not outputs:
            continue
        n = next(iter(outputs.values())).shape[0]
        rows = np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))
        arrays[index_name] = (rows + start).astype(np.float64)
        for name, t in outputs.items():
            a = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy()
            arrays[name] = a.astype(np.float64 if a.dtype in (np.float64, np.int32) else np.float32)
    assert sum(a.nbytes for a in arrays.values()) <= 64 * 10**6
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def read_tensor_peak():
    """Dense bf16/fp16 tensor-core peak (TFLOP/s) for the pilots' forward pass: the sustained cuBLAS figure of MEASURED_PEAKS.json."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        return float(j.get("bf16_tflops_sustained") or j["bf16_tflops"]), "measured (MEASURED_PEAKS.json, sustained bf16)"
    except Exception:
        return 2250.0, "fallback (nominal dense bf16, B200_PROFILING.md)"


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled every ~5 ms through NVML (nvidia_ml_py) on a background thread while the timed region runs;
    falls back to `nvidia-smi -lms` when NVML cannot be loaded."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.thread = None
        self.stop_flag = False
        self.samples = []          # (sm_mhz, reasons bitmask)
        self.max_mhz = None

    def _nvml_loop(self, nv, handle):
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(handle)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                self.samples.append((float(mhz), int(reasons)))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading

            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].strip().isdigit() else self.gpu
            handle = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            for _ in range(3):                     # the first queries of a process take tens of milliseconds: pay for them before the timed region
                nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
            self.nv = nv
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            nv = self.nv
            names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = sorted(m for m, _ in self.samples)
            mask = 0
            for _, r in self.samples:
                mask |= r
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["samples"] = len(sm)
            out["sm_max_mhz"] = self.max_mhz
            out["reasons"] = sorted(k for k, bit in names.items() if mask & bit)
            out["source"] = "nvml, 5 ms period"
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons = [], set()
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    out["sm_max_mhz"] = float(parts[2])
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        out["source"] = "nvidia-smi -lms 200"
        return out


def cpu_reference_leg(cfg, h, w, per_worker):
    from oracle import cpu_bench, cv2_chain
    res = cpu_bench.run("frames", per_worker, h, w, cfg)
    kind = "port"      # oracle/cv2_chain.py: the reference's call sequence over the same OpenCV/numpy (the Python reference cannot travel)
    return {
        "value": res["value"], "unit": "frames/s", "cores": res["cores"], "kind": kind,
        "sample": f"{res['units']} frames of {h}x{w} ({per_worker} per worker process, cv2.setNumThreads(1), "
                  f"{'OpenCV ' + cv2_chain.cv2.__version__ if cv2_chain.cv2 is not None else 'C oracle'}), wall {res['wall_s']:.1f} s, "
                  f"CPU: {cpu_bench.cpu_model()}",
        "single_core_value": res["single_core_value"],
    }


def other_workloads(torch, dev, local, pool120, h, w, cpu_legs=True):
    """Short runs of the remaining BASELINE.json configurations (device-resident inputs, CUDA events)."""
    import numpy as np

    from triton_racer_sim_b200 import FrameNormalise, ImgPreprocessing, LocationTracker, SpeedControl, synth
    from triton_racer_sim_b200 import _native as nat2
    from triton_racer_sim_b200.config import full_house_config
    peak, _ = read_peaks()
    out = {}
    sampler = ClockSampler(local)                  # one clock record over all of these short runs
    sampler.start()

    def timed(fn, reps=5, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3

    # configs[0]: the 7,000-record tub (120x160) through the full chain and through the trainer's /255 (keras_train.py:41-42)
    tub = synth.expand_torch(pool120, 7000)
    fh0 = ImgPreprocessing(full_house_config(), device=local)
    tu8, tf32 = torch.empty_like(tub), torch.empty(tub.shape, dtype=torch.float32, device=dev)
    t = timed(lambda: fh0.process_device(tub, out_u8=tu8, out_f32=tf32, want_f32=True), reps=20)
    out["tub_7000x120x160_full_chain"] = {"frames_per_s": 7000 / t, "ms": t * 1e3, "hbm_frac": 7000 * 345600 / t / 1e9 / peak,
                                          "note": "one launch, 24 frames per CTA: pipeline fill / drain visible; outputs (2 GB) near L2 size"}
    fh0.onShutdown()
    del tub, tu8, tf32
    # configs[1]: crop + resize + normalise for 4,096 cars x 120x160 (u8 in, f32 out): 288,000 algorithmic bytes per frame
    cars = synth.expand_torch(pool120, 4096)
    norm = FrameNormalise(device=local)
    t = timed(lambda: norm.normalise_device(cars), reps=50)
    out["normalise_4096x120x160"] = {"frames_per_s": 4096 / t, "GBps": 4096 * 288000 / t / 1e9, "hbm_frac": 4096 * 288000 / t / 1e9 / peak,
                                      "note": "1.18 GB per step: also fits L2 partially; launch latency visible"}
    big = synth.expand_torch(pool120, 32768)
    t = timed(lambda: norm.normalise_device(big), reps=10)
    out["normalise_32768x120x160"] = {"frames_per_s": 32768 / t, "GBps": 32768 * 288000 / t / 1e9, "hbm_frac": 32768 * 288000 / t / 1e9 / peak}
    norm.onShutdown()
    del big
    pool240 = torch.from_numpy(synth.frame_pool(256, 240, 320)).to(dev)
    src240 = synth.expand_torch(pool240, 4096)
    cam = FrameNormalise(device=local, out_hw=(120, 160))                 # camera.py:36: 320x240 -> 160x120 nearest
    t = timed(lambda: cam.normalise_device(src240), reps=10)
    out["resize2x_normalise_4096"] = {"frames_per_s": 4096 / t, "GBps_algorithmic": 4096 * 288000 / t / 1e9}
    cam.onShutdown()
    del src240, pool240
    # configs[3]: nearest waypoint + speed control for 1M car states on BOTH shipped centre lines (FP64-ALU bound, 76 B of HBM traffic per
    # state): 9 algorithmic flops per (state, waypoint) = 3 subtractions, 3 absolute values, 2 additions, 1 comparison, of which the fp64
    # pipe issues 6 instructions (|x| is an operand modifier)
    n = 1 << 20
    try:
        dfma_tflops, dadd_tinst = nat2.probe_fp64(local)
    except Exception:
        dfma_tflops, dadd_tinst = None, None
    spd = SpeedControl(dict(spd_ctl_break=True), device=local)
    out["waypoint_speed_1M_states"] = {}
    for tname in ("generated_track", "mountain_track"):
        wp = load_track(tname)
        xyz, cur, ms, st = synth.car_states(wp, n, seed=4)
        trk = LocationTracker(wp, device=local)
        d_xyz, d_cur = torch.from_numpy(xyz).to(dev), torch.from_numpy(cur).to(dev)
        d_ms, d_st = torch.from_numpy(ms).to(dev), torch.from_numpy(st).to(dev)

        def cars_step():
            trk.locate_device(d_xyz)
            spd.control_device(d_cur, d_st, d_ms)
        t = timed(cars_step, reps=10)
        t_loc = timed(lambda: trk.locate_device(d_xyz), reps=10)
        # the scanning kernel (every distinct point for every state: what small tables and non-finite centre lines still get) beside it
        os.environ["TRS_LOCATE"] = "thread"
        try:
            trk_scan = LocationTracker(wp, device=local)
        finally:
            del os.environ["TRS_LOCATE"]
        t_scan = timed(lambda: trk_scan.locate_device(d_xyz), reps=10)
        trk_scan.onShutdown()
        nw = wp.shape[0]
        nd = int(np.unique(wp, axis=0).shape[0])          # the kernels evaluate each distinct point at most once (a repeat cannot win the strict `<`)
        ent = {"states_per_s": n / t, "waypoints": int(nw), "distinct_waypoints": nd, "ms": t * 1e3, "locate_only_ms": t_loc * 1e3,
               "locate_only_states_per_s": n / t_loc, "locate_kernels": "trs::k_locate_grid (+ trs::k_locate_warp for the cars it puts off)",
               "hbm_GBps": n * 76 / t / 1e9, "hbm_frac": n * 76 / t / 1e9 / peak,
               "reference_loop_equivalent_tflops": n * nw * 9 / t_loc / 1e12,
               "note": "the grid walk evaluates the reference's distance only for the points in the cells around a car (about 20-30 of them) and "
                       "proves every other point farther away: the reference's argmin, bit for bit, so flops per state are no longer a measure of "
                       "the work; 76 B of HBM traffic per state (locate + speed control) is the remaining roofline, and the step is far from it "
                       "(divergent per-car walks through a shared-memory table)",
               "scan": {"locate_only_ms": t_scan * 1e3, "states_per_s": n / t_scan, "speedup_of_the_grid_walk": t_scan / t_loc}}
        if dfma_tflops:
            ach = n * nd * 9 / t_scan / 1e12
            ent["scan"]["roofline"] = {"bound": "fp64", "achieved": ach, "peak": dfma_tflops, "unit": "TFLOP/s", "frac": ach / dfma_tflops,
                               "fp64_pipe_frac": n * nd * 6 / t_scan / 1e12 / dadd_tinst, "peak_source": "trs_probe_fp64 on this GPU: dense DFMA chains "
                               f"(2 flops per instruction); DADD rate {dadd_tinst:.2f} T lane-instr/s", "kernel": "trs::k_locate",
                               "note": "achieved = 9 flops per (state, DISTINCT waypoint) evaluated / scan time; fp64_pipe_frac = the 6 "
                                       "fp64-pipe instructions per evaluation against the measured DADD issue rate (an add counts one flop, an FMA two); "
                                       "reference_loop_equivalent_tflops counts the reference's loop over all recorded points against the default path's time"}
        out["waypoint_speed_1M_states"][tname] = ent
        trk.onShutdown()
    spd.onShutdown()
    if cpu_legs:                      # the reference's pure-Python loop + math.atan laws on the host cores (bounded sample)
        try:
            from oracle import cpu_bench
            res = cpu_bench.run("cars", 1500, h, w, dict(spd_ctl_break=True))
            out["waypoint_speed_1M_states"].update({"cpu_states_per_s": res["value"], "cpu_cores": res["cores"],
                                                    "cpu_sample": f"{res['units']} states ({1500} per worker process), LocationTracker loop + pilot tail"})
        except Exception as e:
            out["waypoint_speed_1M_states"]["cpu_skipped"] = repr(e)
    d_cur = torch.from_numpy(cur).to(dev)
    # the step after the speed controller: drive-mode select + launch locks + driver assistance (SURVEY.md 8(f) rank 3), 1M cars
    from triton_racer_sim_b200 import ControlMultiplexer
    mux = ControlMultiplexer(dict(ai_launch_boost_throttle_enabled=True, ai_launch_lock_steering_enabled=True), device=local)
    rng = np.random.default_rng(6)
    d_mode = torch.from_numpy(rng.integers(0, 3, n).astype(np.int32)).to(dev)
    d_usr = torch.from_numpy(rng.uniform(-1, 1, (3, n))).to(dev)
    d_ai = torch.from_numpy(rng.uniform(-1, 1, (3, n))).to(dev)
    prm = nat2.ctl_params_from_cfg(mux.cfg, locks=True, assist=True)
    clock = [0.0]

    def mux_step():
        clock[0] += 0.05
        mux.mux_device(d_mode, d_usr, d_ai, clock[0], speed=d_cur, params=prm)
    t = timed(mux_step, reps=20)
    out["control_mux_1M_states"] = {"states_per_s": n / t, "hbm_GBps": n * (4 + 48 + 8 + 24 + 8 + 64) / t / 1e9,
                                     "note": "156 B of traffic per car (mode, 6 inputs, speed, 3 outputs, state read + written)"}
    mux.onShutdown()
    # the pilots' networks (SURVEY.md 8(f) rank 4): full-house forward pass on the tensor cores, alone and behind the fused chain
    try:
        from oracle import pilot_ref
        from triton_racer_sim_b200.pilot import KerasPilot, ModelType
        npil = 16384
        wts = pilot_ref.random_weights(pilot_ref.CNN_2D_FULL_HOUSE, h, w, seed=1)
        pilot = KerasPilot(dict(spd_ctl_break=True), wts, ModelType.CNN_2D_FULL_HOUSE, device=local, max_batch=16384)
        pf = synth.expand_torch(pool120, npil)
        p_spd = torch.rand(npil, device=dev, dtype=torch.float64) * 20
        p_seg = torch.rand(npil, device=dev) * 10
        t = timed(lambda: pilot.pilot_device(pf, p_spd, p_seg), reps=5)
        macs, hh, ww, cc = 0, h, w, 3
        for k, s_, f_ in pilot_ref.CONVS:
            hh, ww = (hh - k) // s_ + 1, (ww - k) // s_ + 1
            macs += hh * ww * f_ * k * k * cc
            cc = f_
        macs += hh * ww * cc * 200 + 2 * (100 * 50 + 50 * 25 + 25 + 16 + 16 * 32 + 32 * 64 + 64 * 100) + 64 * 100
        tpeak, tsrc = read_tensor_peak()
        entry = {"frames_per_s": npil / t, "ms": t * 1e3, "mflop_per_frame": 2 * macs / 1e6,
                 "roofline": {"bound": "tensor", "achieved": 2 * macs * npil / t / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                              "frac": 2 * macs * npil / t / 1e12 / tpeak, "peak_source": tsrc,
                              "note": "algorithmic flops of the reference's layers (no padding counted); fp16 operands, fp32 accumulate; "
                                      "stride-2 layers as GEMMs per input row (N = 3F / 2F), single-lane roles through elect.sync; paced by MMA completion on small-N tiles, not by the tensor pipe: DESIGN.md 4.8, profiles/r02_pilot.md"},
                 "launches_per_16384_frames": 10,
                 "note": "u8 frames + gym/speed + loc/segment -> model -> speed control (ai/steering, ai/throttle, ai/breaking)"}
        fh1 = ImgPreprocessing(full_house_config(), device=local)
        pu8 = torch.empty_like(pf)

        def obs_to_control():
            fh1.process_device(pf, out_u8=pu8, want_f32=False)
            pilot.pilot_device(pu8, p_spd, p_seg)
        t2 = timed(obs_to_control, reps=5)
        entry["with_preprocessing_frames_per_s"] = npil / t2
        fh1.onShutdown()
        if cpu_legs:
            import time as _t
            ncpu = 256
            fr = pool120[:ncpu].cpu().numpy()
            pilot_ref.forward(wts, pilot_ref.CNN_2D_FULL_HOUSE, fr[:32], np.zeros(32, np.float32), np.zeros(32, np.float32))
            t0 = _t.perf_counter()
            pilot_ref.forward(wts, pilot_ref.CNN_2D_FULL_HOUSE, fr, np.zeros(ncpu, np.float32), np.zeros(ncpu, np.float32))
            entry["cpu_frames_per_s"] = ncpu / (_t.perf_counter() - t0)
            entry["cpu_sample"] = f"{ncpu} frames, torch fp32 on {torch.get_num_threads()} host threads (oracle/pilot_ref.py)"
        out["pilot_full_house_16384x120x160"] = entry
        # the reference's own call, one car: numpy frame + python floats in, python floats out (H2D, kernels, D2H, synchronise)
        import time as _t2
        one = pool120[0].cpu().numpy()
        fh2 = ImgPreprocessing(full_house_config(), device=local)
        lat = {}
        for name, fn in (("img_preprocessing_step", lambda: fh2.step(one)),
                         ("keras_pilot_step", lambda: pilot.step(one, 7.5, 3.2, 0.0, 'ai'))):
            for _ in range(20):
                fn()
            t0 = _t2.perf_counter()
            for _ in range(200):
                fn()
            lat[name] = (_t2.perf_counter() - t0) / 200 * 1e6
        fh2.onShutdown()
        out["single_car_latency_us"] = dict(lat, note="N = 1 through Component.step with the reference's argument types, wall clock per call")
        pilot.onShutdown()
        del pf, pu8
    except Exception as e:
        out["pilot_full_house_16384x120x160"] = {"skipped": repr(e)}
    # tub ingestion (SURVEY.md 8(f) rank 1): JPEG files (packed, pinned host memory) -> GPU decode -> (N,H,W,3) u8 on the device;
    # host parsing and the H2D copy of the files are inside the timed region (wall clock: the call synchronises)
    try:
        import io

        from PIL import Image

        from triton_racer_sim_b200 import tub
        pool_np = pool120[:256].cpu().numpy()
        files = []
        for f in pool_np:
            b = io.BytesIO()
            Image.fromarray(f).save(b, format='JPEG')                    # datastorage.py:78
            files.append(b.getvalue())
        nrec = 32768
        blob, offsets = tub.pack_files([files[i % 256] for i in range(nrec)])
        pinned = torch.empty(len(blob), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = blob
        dec = torch.empty((nrec, h, w, 3), dtype=torch.uint8, device=dev)
        ctx = nat2.Context(local)
        for _ in range(2):
            tub.decode_jpeg_batch((pinned.numpy(), offsets), hw=(h, w), ctx=ctx, out=dec)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            tub.decode_jpeg_batch((pinned.numpy(), offsets), hw=(h, w), ctx=ctx, out=dec)
        torch.cuda.synchronize()
        t = (time.perf_counter() - t0) / 3
        t0 = time.perf_counter()
        for b in files[:256]:
            np.asarray(Image.open(io.BytesIO(b)))
        t_pil = (time.perf_counter() - t0) / 256
        out["tub_jpeg_ingest_32768x120x160"] = {"records_per_s": nrec / t, "h2d_bytes_per_record": len(blob) / nrec,
                                                 "pillow_1_thread_records_per_s": 1.0 / t_pil,
                                                 "note": "baseline 4:2:0 JPEG as the recorder writes it; bit-exact with Pillow; parse + H2D + 3 kernels"}
        ctx.close()
    except Exception as e:                                               # Pillow missing on the box: report, do not fail the bench
        out["tub_jpeg_ingest_32768x120x160"] = {"skipped": repr(e)}
    out["clocks"] = sampler.stop()
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the same chain on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from triton_racer_sim_b200.config import full_house_config
    h, w, _, _, _, _ = WORKLOADS[args.workload]
    cfg = full_house_config()
    from oracle import cpu_bench
    per_worker = 256                                            # one step = cores x 256 frames (bounded sample of the workload)
    vals, ms = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = cpu_bench.run("frames", per_worker, h, w, cfg)
        if i >= args.warmup:
            vals.append(res["value"])
            ms.append(res["slowest_worker_s"] * 1e3)
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRICS[args.workload], "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sum(ms) / len(ms), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "frames_per_step": res["units"], "threads": res["cores"]},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": res["cores"], "kind": "port",
                         "sample": f"{res['units']} frames of {h}x{w} per step, one process per core, cv2.setNumThreads(1); CPU: {cpu_bench.cpu_model()}"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------------------------------------
# helpers shared by the timed blocks
# ---------------------------------------------------------------------------------------------------------------------------
class Rig:
    """What every timed block needs: the rank layout, the device, barriers and max-over-ranks timing."""

    def __init__(self, torch, dist, sharding, rank, world, local, dev):
        self.torch, self.dist, self.sharding = torch, dist, sharding
        self.rank, self.world, self.local, self.dev = rank, world, local, dev

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, step, steps, warmup, clocks=True):
        """W warm-up steps, then K steps between CUDA events on the launching stream, barrier + synchronize on both sides, max over
        ranks.  Returns (ms per step, clock record of rank 0 or None)."""
        torch = self.torch
        for _ in range(max(3, warmup)):
            step()
        self.barrier()
        sampler = ClockSampler(self.local) if (clocks and self.rank == 0) else None
        if sampler:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record()
        for _ in range(steps):
            step()
        ev1.record()
        self.barrier()
        ms = self.sharding.max_over_ranks(ev0.elapsed_time(ev1), device=self.dev) / steps
        return ms, (sampler.stop() if sampler else None)


def roofline_block(bytes_per_frame, frames_per_gpu, ms, kernel, note, traffic=None, traffic_source=None):
    peak, peak_src = read_peaks()
    achieved = bytes_per_frame * frames_per_gpu / (ms * 1e-3) / 1e9                   # per-GPU GB/s of algorithmic traffic
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
         "peak_source": peak_src, "bytes_per_frame": bytes_per_frame, "kernel": kernel, "note": note}
    if traffic_source:
        r["traffic_source"] = traffic_source
    return r


def read_traffic(workload, frames):
    """DRAM bytes per launch of the dominant kernel from a committed `ncu --set full` capture (profiles/r02_traffic.json): used only when
    the capture was taken at this run's frame count, otherwise scaled per frame and labelled."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tj = json.load(f)
        ent = tj.get(workload)
        if not ent:
            return None, None
        per = ent["dram_bytes_per_frame"]
        src = f"ncu --set full capture at {ent['frames']} frames/launch ({ent['file']}): dram__bytes_read.sum + dram__bytes_write.sum"
        if ent["frames"] != frames:
            src += f", scaled per frame to this run's {frames}"
        return per * frames, src
    except Exception:
        return None, None


def pcie_probe(rig, host_in, host_out, chunk_frames, reps=3):
    """Copy-only twin of the host pipeline: the same pinned buffers, the same chunking over three streams (one H2D + one D2H per chunk),
    no kernel.  Every rank runs it at the same time, so contention for the host's memory and PCIe root complexes is in the number."""
    torch = rig.torch
    n = host_in.shape[0]
    streams = [torch.cuda.Stream(device=rig.dev) for _ in range(3)]
    st_in = [torch.empty((chunk_frames,) + tuple(host_in.shape[1:]), dtype=torch.uint8, device=rig.dev) for _ in range(3)]
    st_out = [torch.empty_like(b) for b in st_in]

    def once():
        for ci, f0 in enumerate(range(0, n, chunk_frames)):
            s = ci % 3
            cn = min(chunk_frames, n - f0)
            with torch.cuda.stream(streams[s]):
                st_in[s][:cn].copy_(host_in[f0:f0 + cn], non_blocking=True)
                host_out[f0:f0 + cn].copy_(st_out[s][:cn], non_blocking=True)
        for s in streams:
            s.synchronize()
    once()
    rig.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    rig.barrier()
    dt = rig.sharding.max_over_ranks(time.perf_counter() - t0, device=rig.dev) / reps
    nbytes = n * host_in[0].numel()
    return {"frames_per_s_per_rank": n / dt, "GBps_each_way_per_rank": nbytes / dt / 1e9,
            "GBps_aggregate_both_ways": 2 * nbytes * rig.world / dt / 1e9,
            "note": "copy-only: same pinned buffers and 48 MB chunks on three streams as trs_preprocess_host, no kernel, all ranks at once"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="full_chain_120x160", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU per step (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true")
    ap.add_argument("--no-blocks", action="store_true", help="skip the 240x320 / 1M-frame pipeline / statistics blocks")
    ap.add_argument("--quick", action="store_true", help="the headline step only (kernel iteration, ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of what the last step computed "
                                                          "(rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    if args.quick:
        args.no_cpu_baseline = args.no_e2e = args.no_others = args.no_blocks = True
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # stdout carries exactly ONE line, the JSON: everything any library prints meanwhile (NCCL's version banner, torchrun warnings)
    # is sent to stderr at the file-descriptor level; the descriptor is restored for the final print
    sys.stdout.flush()
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")       # NCCL's version / debug lines must not share stdout with the JSON line
    import numpy as np
    import torch
    import torch.distributed as dist

    from triton_racer_sim_b200 import ControlMultiplexer, ImgPreprocessing, LocationTracker, SpeedControl, sharding, synth
    from triton_racer_sim_b200 import _native as nat
    from triton_racer_sim_b200.config import full_house_config

    rank, world, local = sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    rig = Rig(torch, dist, sharding, rank, world, local, dev)
    h, w, frames, want_u8, want_f32, bytes_per_frame = WORKLOADS[args.workload]
    if args.frames:
        frames = args.frames
    cfg = full_house_config()

    # CPU baseline first (rank 0, N = 1 only), before the GPU is busy
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference_leg(cfg, h, w, per_worker=2048)

    # ---- workload: every rank builds its own contiguous block of env indices on its own GPU --------------
    pool_np = synth.frame_pool(1024, h, w)
    pool = torch.from_numpy(pool_np).to(dev)
    start, end = sharding.shard_range(frames * world, rank, world)
    batch = synth.expand_torch(pool, end - start, start=start)
    comp = ImgPreprocessing(cfg, device=local, collect_stats=False)
    out_u8 = torch.empty_like(batch) if want_u8 else None
    out_f32 = torch.empty(batch.shape, dtype=torch.float32, device=dev) if want_f32 else None

    def make_cars(ncar, seed):
        """The per-car stages of BASELINE.json configs[4]: nearest waypoint on the shipped centre line (tests/golden/tracks.npz holds both
        recorded tracks), speed control, control multiplexer: three more launches per step."""
        wp = load_track("generated_track")
        xyz, cur, ms_, st_ = synth.car_states(wp, ncar, seed=seed)
        rng = np.random.default_rng(40 + seed)
        c = {"trk": LocationTracker(wp, device=local), "spd": SpeedControl(dict(spd_ctl_break=True), device=local),
             "mux": ControlMultiplexer(dict(ai_launch_boost_throttle_enabled=True, ai_launch_lock_steering_enabled=True), device=local),
             "xyz": torch.from_numpy(xyz).to(dev), "cur": torch.from_numpy(cur).to(dev), "ms": torch.from_numpy(ms_).to(dev),
             "st": torch.from_numpy(st_).to(dev), "mode": torch.from_numpy(rng.integers(0, 3, ncar).astype(np.int32)).to(dev),
             "usr": torch.from_numpy(rng.uniform(-1, 1, (3, ncar))).to(dev), "clock": 0.0}
        c["prm"] = nat.ctl_params_from_cfg(c["mux"].cfg, locks=True, assist=True)
        return c

    def cars_step(c):
        idx, seg = c["trk"].locate_device(c["xyz"])
        s_, t_, b_, _ = c["spd"].control_device(c["cur"], c["st"], c["ms"])
        c["clock"] += 0.05
        mux = c["mux"].mux_device(c["mode"], c["usr"], torch.stack([s_, t_, b_]), c["clock"], speed=c["cur"], params=c["prm"])
        return {"loc_index": idx, "loc_segment": seg, "ai_steering": s_, "ai_throttle": t_, "ai_breaking": b_,
                "mux_steering": mux[0], "mux_throttle": mux[1], "mux_breaking": mux[2]}

    def close_cars(c):
        for k in ("trk", "spd", "mux"):
            c[k].onShutdown()

    cars = make_cars(end - start, 4 + rank) if args.workload == "full_pipeline_1M_over_8" else None
    last_cars = {}

    def step():
        comp.process_device(batch, out_u8=out_u8, out_f32=out_f32, want_u8=want_u8, want_f32=want_f32)
        if cars is not None:
            last_cars.update(cars_step(cars))

    # ---- headline: K steps of the workload ------------------------------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    rig.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = nat.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rig.barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    rig.barrier()
    elapsed_ms = sharding.max_over_ranks(ev0.elapsed_time(ev1), device=dev)
    launches = nat.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = elapsed_ms / args.steps
    total_frames = frames * world
    value = total_frames / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:              # before the blocks below write into out_u8 / out_f32 again (tub mode: JPEG-decoded frames)
        dump_outputs(args.dump_outputs, start, [("frame_index", DUMP_FRAMES, {"cam_processed_img": out_u8, "cam_normalised_img": out_f32}),
                                                ("car_index", DUMP_CARS, last_cars)])

    # ---- the same step with the per-step statistics ON: counters in the kernel + the system's only collective (a 192-byte all-reduce over
    # NCCL) every step, inside the timed region (north_star: "NCCL used only to gather per-step statistics") ------------------------------
    stats_on = None
    comp_stats = ImgPreprocessing(cfg, device=local, collect_stats=True)
    last_stats = [None]

    def step_stats():
        comp_stats.process_device(batch, out_u8=out_u8, out_f32=out_f32, want_u8=want_u8, want_f32=want_f32)
        last_stats[0] = sharding.reduce_stats(comp_stats._stats_dev)
    if not args.no_blocks:
        ms_s, clk_s = rig.timed(step_stats, max(10, args.steps // 2), args.warmup)
        stats_on = {"ms_per_step": ms_s, "delta_ms_vs_stats_off": ms_s - ms_per_step, "value": total_frames / (ms_s * 1e-3), "unit": "frames/s",
                    "steps": max(10, args.steps // 2), "collective": f"all_reduce(SUM) of {nat.STAT_COUNT} x int64 per step over {world} rank(s)"
                    + (" (NCCL)" if world > 1 else " (single rank: no collective issued)"), "clocks": clk_s,
                    "note": "counters (frames, mask / edge / strong / candidate pixels, hysteresis rounds) accumulated by the store warps, "
                            "zeroed and all-reduced every step inside the timed region"}
    else:
        comp_stats.process_device(batch[: min(1024, batch.shape[0])], want_f32=False)
        last_stats[0] = sharding.reduce_stats(comp_stats._stats_dev)
    st = last_stats[0].cpu()
    comp_stats.onShutdown()

    # ---- end to end through the Component API with HOST buffers (pinned), copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        n_e2e = min(frames, 16384)
        host_in = torch.empty((n_e2e, h, w, 3), dtype=torch.uint8, pin_memory=True)
        host_in.copy_(batch[:n_e2e])
        host_out = torch.empty((n_e2e, h, w, 3), dtype=torch.uint8, pin_memory=True)
        keep_f32 = out_f32[:n_e2e] if want_f32 else None            # the float tensor stays on the GPU for the pilot's model
        in_np, out_np = host_in.numpy(), host_out.numpy()
        e2e_steps = max(3, args.steps // 4)
        for _ in range(2):
            comp.process_host(in_np, out_u8=out_np, keep_f32_dev=keep_f32)
        rig.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            comp.process_host(in_np, out_u8=out_np, keep_f32_dev=keep_f32)     # synchronises before returning
        rig.barrier()
        e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, device=dev) / e2e_steps
        fb = h * w * 3
        e2e = {"value": n_e2e * world / e2e_s, "unit": "frames/s", "frames_per_step": n_e2e * world,
               "h2d_bytes_per_step": n_e2e * fb * world, "d2h_bytes_per_step": n_e2e * fb * world,
               "frames_per_step_per_rank": n_e2e, "h2d_bytes_per_step_per_rank": n_e2e * fb, "d2h_bytes_per_step_per_rank": n_e2e * fb,
               "value_per_rank": n_e2e / e2e_s,
               "note": "host u8 frames -> Component.step -> host u8 cam/processed_img; f32 tensor produced and left on the GPU; "
                       "frames / bytes per step are whole-job figures (all ranks), *_per_rank beside them"}
        # the copy-only ceiling of this box at this rank count
        chunk_frames = max(1, ((48 << 20) // fb + 3) & ~3)
        probe = pcie_probe(rig, host_in, host_out, chunk_frames)
        e2e["pcie_ceiling_per_rank"] = probe["frames_per_s_per_rank"]
        e2e["pcie_probe"] = probe
        e2e["frac_of_pcie_ceiling"] = e2e["value_per_rank"] / probe["frames_per_s_per_rank"]
        # tub mode (keras_train.py:33-57 + manage.py:103-104: "N tub records"): the recorder's JPEG files on the host -> GPU decode -> chain ->
        # host u8; 6-7 KB per frame go in instead of 57.6 KB
        try:
            import io

            from PIL import Image

            from triton_racer_sim_b200 import tub
            files = []
            for f in pool_np[:256]:
                b = io.BytesIO()
                Image.fromarray(f).save(b, format='JPEG')                    # datastorage.py:78
                files.append(b.getvalue())
            # a stream of batches (the trainer's generator walks the tub batch by batch, keras_train.py:33-57): batch k's D2H copy runs on a
            # second stream under batch k + 1's upload + decode + chain (two sets of device / host buffers); every copy is inside the timed region
            blob, offsets = tub.pack_files([files[(start + i) % 256] for i in range(n_e2e)])
            pinned = torch.empty(len(blob), dtype=torch.uint8, pin_memory=True)
            pinned.numpy()[:] = blob
            total_blob = len(blob)
            dec = torch.empty((n_e2e, h, w, 3), dtype=torch.uint8, device=dev)
            tub_u8 = [torch.empty_like(dec) for _ in range(2)]
            tub_host = [host_out, torch.empty((n_e2e, h, w, 3), dtype=torch.uint8, pin_memory=True)]
            copy_stream = torch.cuda.Stream(device=dev)
            copied = [None, None]

            def tub_steps(k_steps):
                main = torch.cuda.current_stream()
                for k in range(k_steps):
                    s_ = k & 1
                    if copied[s_] is not None:
                        copied[s_].synchronize()                             # buffer set s_ is free again (its D2H copy of batch k - 2 is done)
                    tub.decode_jpeg_batch((pinned.numpy(), offsets), hw=(h, w), ctx=comp.ctx, out=dec)       # H2D of the files + decode (synchronises)
                    comp.process_device(dec, out_u8=tub_u8[s_], out_f32=keep_f32, want_f32=want_f32)
                    done = torch.cuda.Event()
                    done.record(main)
                    copy_stream.wait_event(done)
                    with torch.cuda.stream(copy_stream):
                        tub_host[s_].copy_(tub_u8[s_], non_blocking=True)
                        copied[s_] = torch.cuda.Event()
                        copied[s_].record(copy_stream)
                copy_stream.synchronize()
                main.synchronize()
            tub_steps(2)
            rig.barrier()
            tsteps = max(6, e2e_steps)
            t0 = time.perf_counter()
            tub_steps(tsteps)
            rig.barrier()
            tub_s = sharding.max_over_ranks(time.perf_counter() - t0, device=dev) / tsteps
            e2e["tub_mode"] = {"value": n_e2e * world / tub_s, "unit": "frames/s", "frames_per_step": n_e2e * world, "steps": tsteps,
                               "h2d_bytes_per_step": int(total_blob) * world, "d2h_bytes_per_step": n_e2e * fb * world,
                               "h2d_bytes_per_frame": total_blob / n_e2e, "value_per_rank": n_e2e / tub_s,
                               "note": "host JPEG files (Pillow-encoded, as the recorder writes them) -> trs_jpeg_decode_host -> fused chain -> host u8 "
                                       "cam/processed_img for a stream of batches: batch k's D2H copy overlaps batch k + 1's upload, decode and chain "
                                       "(pipeline fill and drain inside the timed region)"}
            del dec, tub_u8, tub_host, pinned
        except Exception as e:                                               # Pillow missing on the box: report, do not fail the bench
            e2e["tub_mode"] = {"skipped": repr(e)}
        del host_in, host_out

    # ---- more configurations of BASELINE.json, every rank on its own shard, each with its own roofline block and clock record -----------
    blocks = None
    if not args.no_blocks:
        blocks = {}
        reps = max(10, args.steps // 2)
        comp.onShutdown()
        del batch, out_u8, out_f32
        torch.cuda.empty_cache()
        # configs[2]: full-house colour + edge mask, 65,536 x 240x320 per GPU (u8 -> u8), then the full chain (u8 + f32) at the same size
        h2, w2, n2 = 240, 320, 65536
        pool240 = torch.from_numpy(synth.frame_pool(256, h2, w2)).to(dev)
        s2, e2_ = sharding.shard_range(n2 * world, rank, world)
        b240 = synth.expand_torch(pool240, e2_ - s2, start=s2)
        o240 = torch.empty_like(b240)
        fh = ImgPreprocessing(cfg, device=local)
        ms2, clk2 = rig.timed(lambda: fh.process_device(b240, out_u8=o240, want_f32=False), reps, args.warmup)
        tr, trs = read_traffic("full_house_mask_240x320", n2)
        blocks["full_house_mask_240x320"] = {
            "metric": METRICS["full_house_mask_240x320"], "value": n2 * world / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2, "steps": reps,
            "frames_per_gpu": n2, "scaling": "weak", "config": f"{n2} frames/GPU/step of {h2}x{w2}x3 u8 -> u8 processed_img (15.1 GB in + 15.1 GB out per GPU)",
            "roofline": roofline_block(230400 + 230400, n2, ms2, KERNELS["full_house_mask_240x320"], NOTES["full_house_mask_240x320"], tr, trs), "clocks": clk2}
        f240 = torch.empty(b240.shape, dtype=torch.float32, device=dev)
        ms3, clk3 = rig.timed(lambda: fh.process_device(b240, out_u8=o240, out_f32=f240, want_f32=True), reps, args.warmup)
        tr, trs = read_traffic("full_chain_240x320", n2)
        blocks["full_chain_240x320"] = {
            "metric": METRICS["full_chain_240x320"], "value": n2 * world / (ms3 * 1e-3), "unit": "frames/s", "ms_per_step": ms3,
            "steps": reps, "frames_per_gpu": n2, "scaling": "weak",
            "config": f"{n2} frames/GPU/step of {h2}x{w2}x3 u8 -> u8 processed_img + f32 /255 tensor (15.1 GB in, 15.1 + 60.4 GB out per GPU)",
            "roofline": roofline_block(230400 * 6, n2, ms3, KERNELS["full_chain_240x320"], NOTES["full_chain_240x320"], tr, trs),
            "clocks": clk3}
        fh.onShutdown()
        del b240, o240, f240, pool240
        torch.cuda.empty_cache()
        # configs[4]: the full observation pipeline over 1,048,576 frames + 1,048,576 car states per step, sharded by env index over the ranks
        # (strong scaling: the total is fixed, a rank owns 1M / N of each).  A rank walks its shard in chunks of <= 131,072 frames (the
        # per-GPU load of the 8-GPU configuration) that reuse one set of output buffers: 60 GB of inputs stay resident at N = 1.
        total, chunk = 1 << 20, 131072
        s5, e5 = sharding.shard_range(total, rank, world)
        n5 = e5 - s5
        in5 = synth.expand_torch(pool, n5, start=s5)
        cn = min(chunk, n5)
        o5 = torch.empty((cn, h, w, 3), dtype=torch.uint8, device=dev)
        f5 = torch.empty((cn, h, w, 3), dtype=torch.float32, device=dev)
        comp5 = ImgPreprocessing(cfg, device=local)
        cars5 = make_cars(n5, 4 + rank)

        def step5():
            for c0 in range(0, n5, chunk):
                c1 = min(n5, c0 + chunk)
                comp5.process_device(in5[c0:c1], out_u8=o5[: c1 - c0], out_f32=f5[: c1 - c0], want_f32=True)
            cars_step(cars5)
        l0 = nat.kernel_launches()
        ms5, clk5 = rig.timed(step5, reps, args.warmup)
        per_step_launches = (nat.kernel_launches() - l0) // (reps + max(3, args.warmup))
        blocks["full_pipeline_1M"] = {
            "metric": METRICS["full_pipeline_1M_over_8"], "value": total / (ms5 * 1e-3), "unit": "frames/s", "ms_per_step": ms5, "steps": reps,
            "frames_per_step": total, "car_states_per_step": total, "frames_per_gpu": n5, "scaling": "strong",
            "launches_per_step_per_rank": int(per_step_launches),
            "config": f"1,048,576 frames of {h}x{w}x3 + 1,048,576 car states per step over {world} rank(s): {n5} of each per GPU, frames in chunks of "
                      f"<= {chunk}; fused chain (u8 + f32 out), nearest waypoint on the shipped centre line (1,185 points), speed control, multiplexer",
            "roofline": roofline_block(bytes_per_frame, n5, ms5, KERNELS["full_pipeline_1M_over_8"], NOTES["full_pipeline_1M_over_8"]), "clocks": clk5}
        comp5.onShutdown()
        close_cars(cars5)
        del in5, o5, f5
        torch.cuda.empty_cache()
    elif cars is not None:
        close_cars(cars)

    # ---- the other BASELINE.json configurations, short runs on rank 0's GPU (reported, not the headline) -----------
    others = None
    if rank == 0 and not args.no_others:
        others = other_workloads(torch, dev, local, pool, h, w, cpu_legs=not args.no_cpu_baseline)

    if rank == 0:
        traffic, traffic_src = read_traffic(args.workload, frames)
        line = {
            "metric": METRICS[args.workload], "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {frames} frames/GPU/step of {h}x{w}x3 u8 -> "
                                   f"{'u8 processed_img' if want_u8 else ''}{' + ' if want_u8 and want_f32 else ''}{'f32 /255 tensor' if want_f32 else ''}, "
                                   "colour filter (2 HSV ranges) + 3-channel Canny, reference defaults",
                       "frames_per_gpu": frames, "h": h, "w": w, "sharding": f"env index, contiguous, {world} rank(s), no data-path collective",
                       "l2": f"inputs {frames * h * w * 3 / 1e9:.2f} GB + outputs per step, far larger than the 126 MB L2 (no flush needed)"},
            "roofline": roofline_block(bytes_per_frame, frames, ms_per_step, KERNELS[args.workload], NOTES[args.workload], traffic, traffic_src),
            "clocks": clocks, "gpu_launches": int(launches),
            "stats_sample": dict(zip(nat.STAT_NAMES[:10], st.tolist()[:10])),
        }
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        if e2e is not None:
            line["e2e"] = e2e
        if stats_on is not None:
            line["stats_on"] = stats_on
        if blocks is not None:
            line["blocks"] = blocks
        if others is not None:
            line["other_workloads"] = others
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
