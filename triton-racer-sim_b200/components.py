"""Batched drop-ins for the reference's hot-path components (same class names, keys, config names, hooks).

Every positional ``step`` argument gains a leading N (cars / tub records); N = 1 inputs in the reference's own
types (numpy HWC frame, python floats) still work and give the reference's result types back, so the classes
can be added to the reference's ``Car`` as they are.  All arithmetic runs in the sm_100a kernels behind
``libtrs_b200.so``; there is no CPU path here.

  ImgPreprocessing   components/img_preprocessing.py:9-108       cam/img -> cam/processed_img
  MultiTrackImgPreprocessing  the same with a configuration per track  cam/img, loc/track -> cam/processed_img
  LocationTracker    components/track_data_process.py:68-107     gym/x, gym/y, gym/z -> loc/segment
  MultiTrackLocationTracker  the same for cars on several tracks    gym/x, gym/y, gym/z, loc/track -> loc/segment
  SpeedControl       components/keras_pilot.py:80-95,99-118,142-153 + utils/mapping.py:23-35
  FrameNormalise     components/camera.py:36 + keras_pilot.py:49-50 / keras_train.py:41-42
  ControlMultiplexer components/controlmultiplexer.py:6-70        usr/*, ai/* -> mux/steering, mux/throttle, mux/breaking
  DriverAssistance   components/driver_assistance.py:4-34         mux/*, gym/speed -> mux/*
  three_segment_map  utils/mapping.py:9-16                        [-1, 1] command -> PWM value
"""
from __future__ import annotations

import ctypes as C
import json
import time

import numpy as np
import torch

from . import _native as nat
from .component import Component
from .config import default_config


def _device_index(device):
    if device is None:
        return torch.cuda.current_device()
    if isinstance(device, torch.device):
        return device.index if device.index is not None else torch.cuda.current_device()
    return int(device)


def _stream_ptr(dev: int):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _check_device_tensor(t, dev: int, dtype, name: str):
    """Every pointer handed to the library must be a contiguous tensor of the stated dtype on the context's GPU: a CPU or other-GPU
    tensor would otherwise become an illegal-address fault that poisons the CUDA context."""
    if t is None:
        return
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch tensor, got {type(t).__name__}")
    if not t.is_cuda or t.device.index != dev:
        raise ValueError(f"{name} must live on cuda:{dev}, got {t.device}")
    if dtype is not None and t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def _np_ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


class ImgPreprocessing(Component):
    """Batched ``ImgPreprocessing``: brightness/contrast, HSV colour masks, 3-channel Canny, merge [+ /255].

    ``step(frames)`` accepts
      * ``None``                                  -> ``(None,)``                       (img_preprocessing.py:20-21)
      * numpy uint8 (H,W,3)                       -> numpy uint8 (H,W,3)               (N = 1 drop-in)
      * numpy uint8 (N,H,W,3) (pageable/pinned)   -> numpy uint8 (N,H,W,3)             (host pipeline, chunked copies)
      * CUDA uint8 tensor (N,H,W,3) or (H,W,3)    -> CUDA tensor, same shape           (stream-ordered, no sync)
    The result is the one for *this* call.  The reference hands back the previous frame's result because its
    worker thread lags (img_preprocessing.py:18-35); ``emulate_latency=True`` reproduces that.
    ``normalised_key`` adds a second output: the float32 ``/255`` tensor the pilots consume (keras_pilot.py:49-50).
    Calls of one component go to one CUDA stream at a time (its context hands out frames to the kernel's CTAs from one counter);
    for concurrent streams use a component per stream.
    """

    def __init__(self, cfg={}, device=None, emulate_latency=False, normalised_key=None, collect_stats=False):
        outputs = ['cam/processed_img'] + ([normalised_key] if normalised_key else [])
        Component.__init__(self, inputs=['cam/img'], outputs=outputs, threaded=False)
        self.running = True
        self.cfg = default_config()
        self.cfg.update(cfg)
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.emulate_latency = bool(emulate_latency)
        self.want_f32 = normalised_key is not None
        self.collect_stats = bool(collect_stats)
        self.processed_img = None          # same attribute name as the reference (img_preprocessing.py:14)
        self.normalised_img = None
        self.last_stats = None
        self._stats_dev = None
        self._apply_cfg()

    def _apply_cfg(self):
        p = nat.preproc_params_from_cfg(self.cfg)
        nat.check(self.ctx.lib.trs_set_preproc_params(self.ctx.handle, C.byref(p)), "trs_set_preproc_params")

    # -- device path ------------------------------------------------------------------------------------
    def process_device(self, frames: torch.Tensor, out_u8=None, out_f32=None, want_u8=True, want_f32=None):
        """(N,H,W,3) uint8 CUDA tensor -> (u8 tensor or None, f32 tensor or None).  Enqueued on the current stream."""
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError(f"expected (N,H,W,3) uint8 frames, got {tuple(frames.shape)} {frames.dtype}")
        if not frames.is_cuda or frames.device.index != self.device:
            raise ValueError(f"frames must live on cuda:{self.device}")
        frames = frames.contiguous()
        n, h, w, _ = frames.shape
        want_f32 = self.want_f32 if want_f32 is None else want_f32
        if want_u8 and out_u8 is None:
            out_u8 = torch.empty_like(frames)
        if want_f32 and out_f32 is None:
            out_f32 = torch.empty(frames.shape, dtype=torch.float32, device=frames.device)
        for t, dt, name in ((out_u8, torch.uint8, "out_u8"), (out_f32, torch.float32, "out_f32")):
            _check_device_tensor(t, self.device, dt, name)
            if t is not None and tuple(t.shape) != tuple(frames.shape):
                raise ValueError(f"{name} must have the frames' shape {tuple(frames.shape)}, got {tuple(t.shape)}")
        stats = None
        if self.collect_stats:
            if self._stats_dev is None:
                self._stats_dev = torch.zeros(nat.STAT_COUNT, dtype=torch.int64, device=frames.device)
            self._stats_dev.zero_()
            stats = self._stats_dev
        nat.check(self.ctx.lib.trs_preprocess(self.ctx.handle, _ptr(frames), n, h, w, _ptr(out_u8), _ptr(out_f32), _ptr(stats),
                                              _stream_ptr(self.device)), "trs_preprocess")
        return out_u8, out_f32

    def stats(self) -> dict:
        """Counters of the last call (synchronises)."""
        if self._stats_dev is None:
            return {}
        v = self._stats_dev.cpu().tolist()
        return dict(zip(nat.STAT_NAMES, v))

    # -- host path --------------------------------------------------------------------------------------
    def process_host(self, frames: np.ndarray, out_u8=None, out_f32=None, keep_f32_dev=None, want_u8=True):
        """(N,H,W,3) uint8 numpy -> numpy.  H2D copy, kernels and D2H copy are pipelined in chunks inside the library."""
        if frames.dtype != np.uint8 or frames.ndim != 4 or frames.shape[-1] != 3:
            raise ValueError(f"expected (N,H,W,3) uint8 frames, got {frames.shape} {frames.dtype}")
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        if want_u8 and out_u8 is None:
            out_u8 = np.empty_like(frames)
        stats = (C.c_ulonglong * nat.STAT_COUNT)() if self.collect_stats else None
        if keep_f32_dev is not None:
            _check_device_tensor(keep_f32_dev, self.device, torch.float32, "keep_f32_dev")
        # the caller's stream is handed over so that work queued on it (a pilot still reading keep_f32_dev) is waited for first
        nat.check(self.ctx.lib.trs_preprocess_host(self.ctx.handle, _np_ptr(frames), n, h, w, _np_ptr(out_u8), _np_ptr(out_f32),
                                                   _ptr(keep_f32_dev), stats, _stream_ptr(self.device)), "trs_preprocess_host")
        if stats is not None:
            self.last_stats = dict(zip(nat.STAT_NAMES, list(stats)))
        return out_u8, out_f32

    # -- Component API ----------------------------------------------------------------------------------
    def step(self, *args):
        img = args[0]
        if img is None:
            result = (None, None)
        elif isinstance(img, torch.Tensor):
            single = img.dim() == 3
            u8, f32 = self.process_device(img[None] if single else img)
            result = (u8[0], f32[0] if f32 is not None else None) if single else (u8, f32)
        else:
            arr = np.asarray(img)
            single = arr.ndim == 3
            batch = arr[None] if single else arr
            f32 = np.empty(batch.shape, np.float32) if self.want_f32 else None
            u8, f32 = self.process_host(batch, out_f32=f32)
            result = (u8[0], f32[0] if f32 is not None else None) if single else (u8, f32)
        if self.emulate_latency:
            previous = (self.processed_img, self.normalised_img)
            self.processed_img, self.normalised_img = result
            result = previous
        else:
            self.processed_img, self.normalised_img = result
        return (result[0], result[1]) if self.want_f32 else (result[0],)

    def thread_step(self):
        """The reference polls a hand-off slot from a worker thread (img_preprocessing.py:23-35); here `step` does the
        work itself on the GPU stream, so there is nothing to run."""
        return

    def onShutdown(self):
        self.running = False
        self.ctx.close()

    def getName(self):
        return 'Image Preprocessing'


class MultiTrackImgPreprocessing(Component):
    """``ImgPreprocessing`` for a batch of cars on several tracks: frame i with ``cfgs[t_i]``.

    Each frame's outputs are exactly what ``ImgPreprocessing(cfgs[t_i])`` gives it, in one stream-ordered call for the whole batch.
    ``cfgs``: one reference config dict per track (its ``myconfig.json``, manage.py:91-94), at most ``nat.MAX_PREPROC_CONFIGS``.

    Inputs ``cam/img, loc/track``; outputs ``cam/processed_img`` [+ ``normalised_key``, the float32 ``/255`` tensor].  ``loc/track`` is the
    per-car index ``MultiTrackLocationTracker`` takes.  ``step(frames, track)`` accepts
      * a CUDA uint8 (N,H,W,3) batch with an int32 (N,) CUDA index tensor  -> CUDA tensors      (stream-ordered, no sync)
      * a numpy uint8 (N,H,W,3) batch with an integer (N,) array           -> numpy             (one upload, one download)
      * one numpy uint8 (H,W,3) frame with a Python int                    -> numpy (H,W,3)     (N = 1 drop-in)
      * ``None``                                                            -> ``None``
    An index outside ``[0, K)`` gives u8 0 and f32 NaN on the device path, and raises ``ValueError`` from the host forms.
    Calls of one component go to one CUDA stream at a time.
    """

    def __init__(self, cfgs, device=None, normalised_key=None, collect_stats=False):
        outputs = ['cam/processed_img'] + ([normalised_key] if normalised_key else [])
        Component.__init__(self, inputs=['cam/img', 'loc/track'], outputs=outputs, threaded=False)
        k = len(cfgs)
        if not 1 <= k <= nat.MAX_PREPROC_CONFIGS:
            raise ValueError(f"1 to {nat.MAX_PREPROC_CONFIGS} configurations, got {k}")
        self.cfgs = []
        for c in cfgs:
            full = default_config()
            full.update(c)
            self.cfgs.append(full)
        self.n_cfgs = k
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.want_f32 = normalised_key is not None
        self.collect_stats = bool(collect_stats)
        self._stats_dev = None
        params = (nat.PreprocParams * k)(*[nat.preproc_params_from_cfg(c) for c in self.cfgs])
        nat.check(self.ctx.lib.trs_set_preproc_configs(self.ctx.handle, params, k), "trs_set_preproc_configs")

    def process_device(self, frames: torch.Tensor, track: torch.Tensor, out_u8=None, out_f32=None, want_u8=True, want_f32=None):
        """(N,H,W,3) uint8 and (N,) int32 CUDA tensors -> (u8 tensor or None, f32 tensor or None).  Enqueued on the current stream."""
        if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError(f"expected (N,H,W,3) uint8 frames, got {getattr(frames, 'shape', None)} {getattr(frames, 'dtype', type(frames))}")
        _check_device_tensor(frames, self.device, torch.uint8, "frames")
        n, h, w, _ = frames.shape
        _check_device_tensor(track, self.device, torch.int32, "track")
        if tuple(track.shape) != (n,):
            raise ValueError(f"track must have shape ({n},), got {tuple(track.shape)}")
        want_f32 = self.want_f32 if want_f32 is None else want_f32
        if want_u8 and out_u8 is None:
            out_u8 = torch.empty_like(frames)
        if want_f32 and out_f32 is None:
            out_f32 = torch.empty(frames.shape, dtype=torch.float32, device=frames.device)
        for t, dt, name in ((out_u8, torch.uint8, "out_u8"), (out_f32, torch.float32, "out_f32")):
            _check_device_tensor(t, self.device, dt, name)
            if t is not None and tuple(t.shape) != tuple(frames.shape):
                raise ValueError(f"{name} must have the frames' shape {tuple(frames.shape)}, got {tuple(t.shape)}")
        stats = None
        if self.collect_stats:
            if self._stats_dev is None:
                self._stats_dev = torch.zeros((self.n_cfgs, nat.STAT_COUNT), dtype=torch.int64, device=frames.device)
            self._stats_dev.zero_()
            stats = self._stats_dev
        nat.check(self.ctx.lib.trs_preprocess_configs(self.ctx.handle, _ptr(frames), _ptr(track), n, h, w, _ptr(out_u8), _ptr(out_f32),
                                                      _ptr(stats), _stream_ptr(self.device)), "trs_preprocess_configs")
        return out_u8, out_f32

    def stats(self) -> list:
        """Counters of the last device call, one dict per configuration (synchronises)."""
        if self._stats_dev is None:
            return []
        return [dict(zip(nat.STAT_NAMES, row)) for row in self._stats_dev.cpu().tolist()]

    def _host_tracks(self, track, n: int):
        t = np.asarray(track)
        if not np.issubdtype(t.dtype, np.integer):
            raise ValueError(f"track indices must be integers, got {t.dtype}")
        if t.shape != (n,):
            raise ValueError(f"track must have shape ({n},), got {t.shape}")
        if t.size and (t.min() < 0 or t.max() >= self.n_cfgs):
            raise ValueError(f"track index outside [0, {self.n_cfgs})")
        return np.ascontiguousarray(t, np.int32)

    def step(self, *args):
        img, track = args[0], args[1]
        if img is None:
            return (None, None) if self.want_f32 else (None,)
        if isinstance(img, torch.Tensor):
            u8, f32 = self.process_device(img, track)
            return (u8, f32) if self.want_f32 else (u8,)
        arr = np.asarray(img)
        single = arr.ndim == 3
        if single:
            if isinstance(track, (bool, np.bool_)) or not isinstance(track, (int, np.integer)):
                raise ValueError(f"one frame takes one integer track index, got {type(track).__name__}")
            track = [track]
        batch = arr[None] if single else arr
        if batch.dtype != np.uint8 or batch.ndim != 4 or batch.shape[-1] != 3:
            raise ValueError(f"expected (N,H,W,3) uint8 frames, got {batch.shape} {batch.dtype}")
        dev = f"cuda:{self.device}"
        t = torch.from_numpy(self._host_tracks(track, batch.shape[0])).to(dev)
        u8, f32 = self.process_device(torch.from_numpy(np.ascontiguousarray(batch)).to(dev), t)
        u8 = u8.cpu().numpy()
        f32 = f32.cpu().numpy() if f32 is not None else None
        if single:
            u8, f32 = u8[0], (f32[0] if f32 is not None else None)
        return (u8, f32) if self.want_f32 else (u8,)

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Multi-Track Image Preprocessing'


class LocationTracker(Component):
    """Batched ``LocationTracker``: nearest waypoint (L1, float64, first index on ties, sentinel 100) -> segment."""

    def __init__(self, track_data_path, min_map=0, max_map=10, device=None):
        Component.__init__(self, inputs=['gym/x', 'gym/y', 'gym/z'], outputs=['loc/segment'])
        if isinstance(track_data_path, (str, bytes)) or hasattr(track_data_path, "__fspath__"):
            with open(track_data_path, 'r') as input_file:        # FileNotFoundError propagates (track_data_process.py:72)
                self.data = json.load(input_file)
        else:
            self.data = np.asarray(track_data_path, np.float64).tolist()
        self.max = max_map
        self.min = min_map
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        wp = np.ascontiguousarray(np.asarray(self.data, dtype=np.float64).reshape(-1, 3))
        # (max - min) is evaluated in python like the reference (ints stay exact), then handed over as doubles
        nat.check(self.ctx.lib.trs_set_track(self.ctx.handle, _np_ptr(wp), wp.shape[0], float(min_map), float(max_map)),
                  "trs_set_track")
        self.n_wp = wp.shape[0]

    def locate_device(self, xyz: torch.Tensor, want_idx=True, want_segment=True):
        """xyz (N,3) float64 CUDA tensor -> (idx int32 (N,), segment float64 (N,))."""
        if xyz.dtype != torch.float64 or xyz.dim() != 2 or xyz.shape[1] != 3:
            raise ValueError(f"expected (N,3) float64, got {tuple(xyz.shape)} {xyz.dtype}")
        xyz = xyz.contiguous()
        _check_device_tensor(xyz, self.device, torch.float64, "xyz")
        n = xyz.shape[0]
        idx = torch.empty(n, dtype=torch.int32, device=xyz.device) if want_idx else None
        seg = torch.empty(n, dtype=torch.float64, device=xyz.device) if want_segment else None
        nat.check(self.ctx.lib.trs_locate(self.ctx.handle, _ptr(xyz), n, _ptr(idx), _ptr(seg), _stream_ptr(self.device)), "trs_locate")
        return idx, seg

    def localize(self, point):
        seg = self.step(point[0], point[1], point[2])[0]
        return seg, 0.0

    def step(self, *args):
        x, y, z = args[0], args[1], args[2]
        if isinstance(x, torch.Tensor) and x.dim() >= 1:
            xyz = torch.stack([x.to(torch.float64), y.to(torch.float64), z.to(torch.float64)], dim=1)
            return self.locate_device(xyz, want_idx=False)[1],
        if isinstance(x, np.ndarray) and x.ndim >= 1:
            xyz = torch.from_numpy(np.stack([x, y, z], axis=1).astype(np.float64)).to(f"cuda:{self.device}")
            return self.locate_device(xyz, want_idx=False)[1].cpu().numpy(),
        xyz = torch.tensor([[float(x), float(y), float(z)]], dtype=torch.float64, device=f"cuda:{self.device}")  # TypeError on None, like the reference
        return float(self.locate_device(xyz, want_idx=False)[1].item()),

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Location Tracker'


def _per_track(v, k: int, name: str):
    vals = [v] * k if np.ndim(v) == 0 else list(v)
    if len(vals) != k:
        raise ValueError(f"{name}: one value per track ({k}), got {len(vals)}")
    return (C.c_double * k)(*[float(x) for x in vals])


class MultiTrackLocationTracker(Component):
    """``LocationTracker`` for a batch of cars on several tracks: car i on ``track_data_paths[t_i]``.

    Each car's segment is exactly what ``LocationTracker(track_data_paths[t_i], min_map[t_i], max_map[t_i])`` gives it, in one
    stream-ordered call for the whole batch.  ``track_data_paths``: centre line files or (N, 3) point arrays (at most
    ``nat.MAX_TRACKS``); ``min_map`` / ``max_map``: one value, or one per track.

    Inputs ``gym/x, gym/y, gym/z, loc/track``; output ``loc/segment``.  ``loc/track`` is a key of this project, not of the reference
    (where every car builds its own tracker, manage.py:97-99): the index of each car's track in ``track_data_paths``.
    A track index outside ``[0, K)`` gives index -1 and segment NaN on the device path, and raises ``ValueError`` from the host forms.
    """

    def __init__(self, track_data_paths, min_map=0, max_map=10, device=None):
        Component.__init__(self, inputs=['gym/x', 'gym/y', 'gym/z', 'loc/track'], outputs=['loc/segment'])
        lines = []
        for p in track_data_paths:
            if isinstance(p, (str, bytes)) or hasattr(p, "__fspath__"):
                with open(p, 'r') as input_file:
                    p = json.load(input_file)
            lines.append(np.ascontiguousarray(np.asarray(p, dtype=np.float64).reshape(-1, 3)))
        k = len(lines)
        if not 1 <= k <= nat.MAX_TRACKS:
            raise ValueError(f"1 to {nat.MAX_TRACKS} tracks, got {k}")
        self.min, self.max = min_map, max_map
        self.n_tracks = k
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        nat.check(self.ctx.lib.trs_set_tracks(self.ctx.handle, (C.c_void_p * k)(*[a.ctypes.data for a in lines]),
                                              (C.c_int * k)(*[a.shape[0] for a in lines]), _per_track(min_map, k, "min_map"),
                                              _per_track(max_map, k, "max_map"), k), "trs_set_tracks")
        self.n_wp = [a.shape[0] for a in lines]

    def locate_device(self, xyz: torch.Tensor, track: torch.Tensor, want_idx=True, want_segment=True):
        """xyz (N,3) float64 and track (N,) int32 CUDA tensors -> (idx int32 (N,), segment float64 (N,)).  Enqueued on the current stream."""
        if xyz.dtype != torch.float64 or xyz.dim() != 2 or xyz.shape[1] != 3:
            raise ValueError(f"expected (N,3) float64, got {tuple(xyz.shape)} {xyz.dtype}")
        xyz = xyz.contiguous()
        _check_device_tensor(xyz, self.device, torch.float64, "xyz")
        n = xyz.shape[0]
        _check_device_tensor(track, self.device, torch.int32, "track")
        if tuple(track.shape) != (n,):
            raise ValueError(f"track must have shape ({n},), got {tuple(track.shape)}")
        idx = torch.empty(n, dtype=torch.int32, device=xyz.device) if want_idx else None
        seg = torch.empty(n, dtype=torch.float64, device=xyz.device) if want_segment else None
        nat.check(self.ctx.lib.trs_locate_tracks(self.ctx.handle, _ptr(xyz), _ptr(track), n, _ptr(idx), _ptr(seg), _stream_ptr(self.device)),
                  "trs_locate_tracks")
        return idx, seg

    def _host_tracks(self, track):
        t = np.asarray(track)
        if not np.issubdtype(t.dtype, np.integer):
            raise ValueError(f"track indices must be integers, got {t.dtype}")
        if t.size and (t.min() < 0 or t.max() >= self.n_tracks):
            raise ValueError(f"track index outside [0, {self.n_tracks})")
        return t.astype(np.int32)

    def step(self, *args):
        x, y, z, track = args[0], args[1], args[2], args[3]
        if isinstance(x, torch.Tensor) and x.dim() >= 1:
            xyz = torch.stack([x.to(torch.float64), y.to(torch.float64), z.to(torch.float64)], dim=1)
            return self.locate_device(xyz, track, want_idx=False)[1],
        dev = f"cuda:{self.device}"
        if isinstance(x, np.ndarray) and x.ndim >= 1:
            t = torch.from_numpy(np.ascontiguousarray(self._host_tracks(track))).to(dev)
            xyz = torch.from_numpy(np.stack([x, y, z], axis=1).astype(np.float64)).to(dev)
            return self.locate_device(xyz, t, want_idx=False)[1].cpu().numpy(),
        t = torch.from_numpy(self._host_tracks([track])).to(dev)
        xyz = torch.tensor([[float(x), float(y), float(z)]], dtype=torch.float64, device=dev)
        return float(self.locate_device(xyz, t, want_idx=False)[1].item()),

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Multi-Track Location Tracker'


class SpeedControl(Component):
    """The pilots' post-model glue for ``cnn_2d_speed_control`` / ``cnn_2d_full_house``, batched.

    step(gym/speed (N,) f64, model steering (N,) f32, model speed (N,) f32) -> ai/steering, ai/throttle, ai/breaking (f64).
    ``features(gym/speed)`` gives the float32 ``speed / 20`` model input (keras_pilot.py:68,100).
    """

    def __init__(self, cfg={}, device=None):
        Component.__init__(self, inputs=['gym/speed', 'pilot/steering', 'pilot/speed'],
                           outputs=['ai/steering', 'ai/throttle', 'ai/breaking'])
        self.cfg = default_config()
        self.cfg.update(cfg)
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.params = nat.spd_params_from_cfg(self.cfg)
        self.last_feature = None

    def control_device(self, cur: torch.Tensor, steer: torch.Tensor, spd: torch.Tensor, want_feature=False):
        n = cur.shape[0]
        cur = cur.to(torch.float64).contiguous()
        steer = steer.to(torch.float32).contiguous()
        spd = spd.to(torch.float32).contiguous()
        for t, name in ((cur, "gym/speed"), (steer, "pilot/steering"), (spd, "pilot/speed")):
            _check_device_tensor(t, self.device, None, name)
            if t.dim() != 1 or t.shape[0] != n:
                raise ValueError(f"{name} must have shape ({n},), got {tuple(t.shape)}")
        out = torch.empty((3, n), dtype=torch.float64, device=cur.device)
        feat = torch.empty(n, dtype=torch.float32, device=cur.device) if want_feature else None
        nat.check(self.ctx.lib.trs_speed_control(self.ctx.handle, _ptr(cur), _ptr(spd), _ptr(steer), n, C.byref(self.params),
                                                 _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(feat), _stream_ptr(self.device)),
                  "trs_speed_control")
        return out[0], out[1], out[2], feat

    def step(self, *args):
        cur, steer, spd = args[0], args[1], args[2]
        if cur is None:
            return 0.0, 0.0, 0.0                                   # keras_pilot.py:46-47
        if isinstance(cur, torch.Tensor) and cur.dim() >= 1:
            s, t, b, _ = self.control_device(cur, steer, spd)
            return s, t, b
        dev = f"cuda:{self.device}"
        if isinstance(cur, np.ndarray) and cur.ndim >= 1:
            s, t, b, _ = self.control_device(torch.from_numpy(np.asarray(cur, np.float64)).to(dev),
                                             torch.from_numpy(np.asarray(steer, np.float32)).to(dev),
                                             torch.from_numpy(np.asarray(spd, np.float32)).to(dev))
            return s.cpu().numpy(), t.cpu().numpy(), b.cpu().numpy()
        s, t, b, _ = self.control_device(torch.tensor([float(cur)], dtype=torch.float64, device=dev),
                                         torch.tensor([float(steer)], dtype=torch.float32, device=dev),
                                         torch.tensor([float(spd)], dtype=torch.float32, device=dev))
        return float(s.item()), float(t.item()), float(b.item())

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Speed Control'


class FrameNormalise(Component):
    """Camera-side resize (nearest, camera.py:36), optional window crop, and the ``/255`` float32 normalisation
    (keras_pilot.py:49-50, keras_train.py:41-42) for N frames: cam/img -> cam/normalised_img."""

    def __init__(self, cfg={}, device=None, roi=None, out_hw=None):
        Component.__init__(self, inputs=['cam/img'], outputs=['cam/normalised_img'])
        self.cfg = default_config()
        self.cfg.update(cfg)
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.roi = roi                                  # (y0, y1, x0, x1) in source pixels, or None = whole frame
        self.out_hw = out_hw                            # (h, w) or None = window size (no resize)

    def normalise_device(self, frames: torch.Tensor, want_u8=False):
        if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError(f"expected (N,H,W,3) uint8 frames, got {tuple(frames.shape)} {frames.dtype}")
        frames = frames.contiguous()
        _check_device_tensor(frames, self.device, torch.uint8, "frames")
        n, h, w, _ = frames.shape
        y0, y1, x0, x1 = self.roi if self.roi is not None else (0, h, 0, w)
        ho, wo = self.out_hw if self.out_hw is not None else (y1 - y0, x1 - x0)
        out = torch.empty((n, ho, wo, 3), dtype=torch.float32, device=frames.device)
        u8 = torch.empty((n, ho, wo, 3), dtype=torch.uint8, device=frames.device) if want_u8 else None
        nat.check(self.ctx.lib.trs_normalise(self.ctx.handle, _ptr(frames), n, h, w, y0, y1, x0, x1, ho, wo, _ptr(out), _ptr(u8),
                                             _stream_ptr(self.device)), "trs_normalise")
        return (out, u8) if want_u8 else out

    def step(self, *args):
        img = args[0]
        if img is None:
            return None,
        if isinstance(img, torch.Tensor):
            single = img.dim() == 3
            out = self.normalise_device(img[None] if single else img)
            return (out[0] if single else out),
        arr = np.asarray(img)
        single = arr.ndim == 3
        t = torch.from_numpy(np.ascontiguousarray(arr[None] if single else arr)).to(f"cuda:{self.device}")
        out = self.normalise_device(t).cpu().numpy()
        return (out[0] if single else out),

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Frame Normalise'


def _mode_code(m):
    """DriveMode member (components/controller.py:7-10), its string value, or a TRS_MODE_* integer -> integer code."""
    v = getattr(m, 'value', m)
    if isinstance(v, str):
        return {'human': nat.MODE_HUMAN, 'ai_steering': nat.MODE_AI_STEERING, 'ai': nat.MODE_AI}[v]
    return int(v)


def _as_f64(x, dev, n=None):
    if isinstance(x, torch.Tensor):
        return x.to(device=dev, dtype=torch.float64).reshape(-1).contiguous()
    return torch.as_tensor(np.asarray(x, np.float64).reshape(-1), device=dev)


class ControlMultiplexer(Component):
    """Batched ``ControlMultiplexer`` (components/controlmultiplexer.py): user / pilot select by drive mode and the AI launch locks.

    ``step(mode, usr_steering, usr_throttle, usr_breaking, ai_steering, ai_throttle, ai_breaking, now=None)``: every argument a
    scalar (reference types: DriveMode member + python floats -> tuple of floats) or an (N,) array / CUDA tensor (-> CUDA f64
    tensors).  The reference ends its locks from sleeping threads; here the clock is ``now`` (seconds, default
    ``time.monotonic()``) and the per-car state (last mode, last launch times) lives in device tensors of this component.
    """

    def __init__(self, cfg={}, device=None):
        Component.__init__(self, inputs=['usr/mode', 'usr/steering', 'usr/throttle', 'usr/breaking', 'ai/steering', 'ai/throttle', 'ai/breaking'],
                           outputs=['mux/steering', 'mux/throttle', 'mux/breaking'])
        self.cfg = default_config()
        self.cfg.update(cfg)
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.params = nat.ctl_params_from_cfg(self.cfg, locks=True, assist=False)
        self.last_mode = None
        self.launch_times = None

    def _state(self, n, dev):
        if self.last_mode is None or self.last_mode.shape[0] != n:
            self.last_mode = torch.full((n,), nat.MODE_HUMAN, dtype=torch.int32, device=dev)          # controlmultiplexer.py:10
            self.launch_times = torch.full((nat.LAUNCH_SLOTS, n), nat.NEVER, dtype=torch.float64, device=dev)

    def mux_device(self, mode: torch.Tensor, usr: torch.Tensor, ai: torch.Tensor, now: float, speed: torch.Tensor = None, params=None):
        """mode (N,) int32, usr / ai (3, N) f64 on the device -> (3, N) f64 (steering, throttle, breaking)."""
        n = mode.shape[0]
        _check_device_tensor(mode, self.device, torch.int32, "mode")
        for t, name in ((usr, "usr"), (ai, "ai")):
            _check_device_tensor(t, self.device, torch.float64, name)
            if tuple(t.shape) != (3, n):
                raise ValueError(f"{name} must have shape (3, {n}), got {tuple(t.shape)}")
        _check_device_tensor(speed, self.device, torch.float64, "speed")
        self._state(n, mode.device)
        out = torch.empty((3, n), dtype=torch.float64, device=mode.device)
        nat.check(self.ctx.lib.trs_control_mux(self.ctx.handle, _ptr(mode), _ptr(usr), _ptr(ai), _ptr(speed), n,
                                               C.byref(params if params is not None else self.params), float(now), _ptr(self.last_mode),
                                               _ptr(self.launch_times), _ptr(out), _stream_ptr(self.device)), "trs_control_mux")
        return out

    def step(self, *args, now=None):
        mode = args[0]
        now = time.monotonic() if now is None else float(now)
        dev = f"cuda:{self.device}"
        batched = isinstance(mode, (torch.Tensor, np.ndarray, list, tuple))
        if batched:
            if isinstance(mode, torch.Tensor):
                m = mode.to(device=dev, dtype=torch.int32).contiguous()
            else:
                m = torch.as_tensor(np.asarray([_mode_code(x) for x in mode], np.int32), device=dev)
        else:
            m = torch.tensor([_mode_code(mode)], dtype=torch.int32, device=dev)
        vals = [_as_f64(a, dev) for a in args[1:7]]
        usr, ai = torch.stack(vals[0:3]), torch.stack(vals[3:6])
        out = self.mux_device(m, usr.contiguous(), ai.contiguous(), now)
        if batched:
            return out[0], out[1], out[2]
        o = out[:, 0].tolist()
        return o[0], o[1], o[2]

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Control Multiplexer'


class DriverAssistance(Component):
    """Batched ``DriverAssistance`` (components/driver_assistance.py): steering / speed limiter ``k / x``.  Keys as the reference
    (``mux/break`` included, driver_assistance.py:8-9); any ``None`` argument passes everything through (driver_assistance.py:15)."""

    def __init__(self, cfg={}, device=None):
        Component.__init__(self, inputs=['mux/steering', 'mux/throttle', 'mux/break', 'gym/speed'],
                           outputs=['mux/steering', 'mux/throttle', 'mux/break'], threaded=False)
        self.cfg = default_config()
        self.cfg.update(cfg)
        self.limit_mode = self.cfg['drive_assist_limit_mode']
        self.k = self.cfg['drive_assist_limit_k']
        self.device = _device_index(device)
        self.ctx = nat.Context(self.device)
        self.params = nat.ctl_params_from_cfg(self.cfg, locks=False, assist=True)

    def assist_device(self, steering, throttle, breaking, speed):
        n = steering.shape[0]
        dev = steering.device
        for t, name in ((steering, "mux/steering"), (throttle, "mux/throttle"), (breaking, "mux/break"), (speed, "gym/speed")):
            _check_device_tensor(t, self.device, torch.float64, name)
        usr = torch.stack([steering, throttle, breaking]).contiguous()
        mode = torch.full((n,), nat.MODE_HUMAN, dtype=torch.int32, device=dev)       # "human" selects the first triple unchanged
        last = torch.full((n,), nat.MODE_HUMAN, dtype=torch.int32, device=dev)
        launch = torch.full((nat.LAUNCH_SLOTS, n), nat.NEVER, dtype=torch.float64, device=dev)
        out = torch.empty((3, n), dtype=torch.float64, device=dev)
        nat.check(self.ctx.lib.trs_control_mux(self.ctx.handle, _ptr(mode), _ptr(usr), _ptr(usr), _ptr(speed), n, C.byref(self.params), 0.0,
                                               _ptr(last), _ptr(launch), _ptr(out), _stream_ptr(self.device)), "trs_control_mux")
        return out[0], out[1], out[2]

    def step(self, *args):
        steering, throttle, breaking, speed = args
        if any(a is None for a in args):
            return steering, throttle, breaking
        dev = f"cuda:{self.device}"
        batched = isinstance(steering, (torch.Tensor, np.ndarray))
        s, t, b, v = (_as_f64(a, dev) for a in args)
        so, to, bo = self.assist_device(s, t, b, v)
        if batched:
            return so, to, bo
        return float(so.item()), float(to.item()), float(bo.item())

    def onShutdown(self):
        self.ctx.close()

    def getName(self):
        return 'Driver Assistance'


def three_segment_map(val, min_map, mid_map, max_map, device=None):
    """``utils/mapping.py:9-16`` for N commands: CUDA tensor / array in -> CUDA f64 tensor out; python float in -> float out."""
    dev_i = _device_index(device)
    dev = f"cuda:{dev_i}"
    scalar = not isinstance(val, (torch.Tensor, np.ndarray, list, tuple))
    v = _as_f64(val, dev)
    out = torch.empty_like(v)
    ctx = nat.Context(dev_i)
    try:
        nat.check(ctx.lib.trs_pwm_map(ctx.handle, _ptr(v), v.shape[0], float(min_map), float(mid_map), float(max_map), _ptr(out), _stream_ptr(dev_i)),
                  "trs_pwm_map")
        torch.cuda.current_stream(dev_i).synchronize()
    finally:
        ctx.close()
    return float(out.item()) if scalar else out
