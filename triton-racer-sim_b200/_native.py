"""ctypes binding of libtrs_b200.so (the C ABI in include/trs_b200.h).

There is no fallback: if the library is missing, cannot be loaded, or no sm_100 GPU is present, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TRS_B200_LIB") or os.path.join(HERE, "libtrs_b200.so")     # (override: instrumented builds of the same library)
MAX_HSV = 4
STAT_COUNT = 24
STAT_NAMES = ["frames", "mask0", "mask1", "mask2", "mask3", "edge", "strong", "cand", "hyst_sweeps", "roi_sum",
              "t_wait_frame", "t_strip_walk", "t_phase_a", "t_phase_b", "t_phase_c", "t_total"]

# every symbol include/trs_b200.h declares (tests check the library exports exactly these)
SYMBOLS = [
    "trs_version", "trs_last_error", "trs_kernel_launches", "trs_ctx_create", "trs_ctx_destroy", "trs_ctx_device_info",
    "trs_set_preproc_params", "trs_preprocess", "trs_normalise", "trs_set_track", "trs_locate", "trs_speed_control",
    "trs_preprocess_host", "trs_host_alloc", "trs_host_free", "trs_debug_canny_stages", "trs_control_mux", "trs_pwm_map",
    "trs_jpeg_decode_host", "trs_telemetry_decode_host", "trs_jpeg_encode", "trs_jpeg_encode_copy",
    "trs_pilot_create", "trs_pilot_destroy", "trs_pilot_forward", "trs_pilot_debug_activation", "trs_pilot_layer_shape",
    "trs_pilot_cap", "trs_probe_fp64",
]
MODE_HUMAN, MODE_AI_STEERING, MODE_AI = 0, 1, 2          # TRS_MODE_*: DriveMode.HUMAN / AI_STEERING / AI (components/controller.py:7-10)
LAUNCH_SLOTS = 4                                          # TRS_LAUNCH_SLOTS
NEVER = -1.0e300                                          # TRS_NEVER


class PreprocParams(C.Structure):
    _fields_ = [
        ("contrast_ratio", C.c_double), ("contrast_offset", C.c_double), ("brightness_baseline", C.c_double),
        ("dynamic_brightness", C.c_int32), ("color_filter_enabled", C.c_int32), ("n_hsv", C.c_int32),
        ("edge_enabled", C.c_int32),
        ("hsv_lo", (C.c_double * 3) * MAX_HSV), ("hsv_hi", (C.c_double * 3) * MAX_HSV),
        ("color_dest", C.c_int32 * MAX_HSV), ("edge_dest", C.c_int32),
        ("canny_a", C.c_double), ("canny_b", C.c_double),
    ]


class SpdParams(C.Structure):
    _fields_ = [
        ("threshold", C.c_double), ("reverse_multiplier", C.c_double), ("break_multiplier", C.c_double),
        ("use_break", C.c_int32), ("smooth_steering", C.c_int32), ("smooth_threshold", C.c_double),
        ("numpy_legacy_promotion", C.c_int32), ("reserved", C.c_int32),
    ]


class CtlParams(C.Structure):
    _fields_ = [
        ("throttle_lock_enabled", C.c_int32), ("steering_lock_enabled", C.c_int32), ("assist_mode", C.c_int32), ("reserved", C.c_int32),
        ("throttle_lock_value", C.c_double), ("throttle_lock_duration", C.c_double), ("steering_lock_value", C.c_double),
        ("steering_lock_duration", C.c_double), ("assist_k", C.c_double),
    ]


class Tensor(C.Structure):
    """trs_tensor: one named host weight array in Keras layout."""
    _fields_ = [("name", C.c_char_p), ("data", C.POINTER(C.c_float)), ("ndim", C.c_int32), ("shape", C.c_int32 * 4)]


class NativeError(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library; raises with a build hint when it is absent (never falls back to a CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(f"{LIB_PATH} is missing: build it with `python -m triton_racer_sim_b200.build` "
                          "(nvcc, sm_100a). There is no CPU implementation of this path.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, u64p = C.c_void_p, C.c_int, C.POINTER(C.c_ulonglong)
    lib.trs_version.restype = C.c_int
    lib.trs_last_error.restype = C.c_char_p
    lib.trs_kernel_launches.restype = C.c_ulonglong
    lib.trs_ctx_create.argtypes = [i32, C.POINTER(vp)]
    lib.trs_ctx_destroy.argtypes = [vp]
    lib.trs_ctx_device_info.argtypes = [vp] + [C.POINTER(C.c_int)] * 4
    lib.trs_set_preproc_params.argtypes = [vp, C.POINTER(PreprocParams)]
    lib.trs_preprocess.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp]
    lib.trs_normalise.argtypes = [vp, vp] + [i32] * 9 + [vp, vp, vp]
    lib.trs_set_track.argtypes = [vp, vp, i32, C.c_double, C.c_double]
    lib.trs_locate.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.trs_speed_control.argtypes = [vp, vp, vp, vp, i32, C.POINTER(SpdParams), vp, vp, vp, vp, vp]
    lib.trs_preprocess_host.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.trs_host_alloc.argtypes = [C.POINTER(vp), C.c_ulonglong]
    lib.trs_host_free.argtypes = [vp]
    lib.trs_debug_canny_stages.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.trs_control_mux.argtypes = [vp, vp, vp, vp, vp, i32, C.POINTER(CtlParams), C.c_double, vp, vp, vp, vp]
    lib.trs_pwm_map.argtypes = [vp, vp, i32, C.c_double, C.c_double, C.c_double, vp, vp]
    lib.trs_jpeg_decode_host.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.trs_telemetry_decode_host.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.trs_jpeg_encode.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp]
    lib.trs_jpeg_encode_copy.argtypes = [vp, vp, C.c_ulonglong, vp]
    lib.trs_pilot_create.argtypes = [vp, i32, i32, i32, C.POINTER(Tensor), i32, i32, C.POINTER(vp)]
    lib.trs_pilot_destroy.argtypes = [vp]
    lib.trs_pilot_forward.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    lib.trs_pilot_debug_activation.argtypes = [vp, i32, vp, C.c_ulonglong, vp]
    lib.trs_pilot_layer_shape.argtypes = [vp, i32] + [C.POINTER(C.c_int)] * 3
    lib.trs_pilot_cap.argtypes = [vp, vp, i32, i32, C.c_double, vp, vp, vp, vp]
    lib.trs_probe_fp64.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    for name in SYMBOLS:
        getattr(lib, name)
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc == 0:
        return
    msg = load().trs_last_error().decode(errors="replace")
    if rc < 0:
        if rc == -4:
            raise NativeError(f"{what}: {msg}")
        raise ValueError(f"{what}: {msg}")
    raise NativeError(f"{what}: CUDA error {rc}: {msg}")


class Context:
    """One per GPU (trs_ctx).  Owns the uploaded parameters and the centre line."""

    _by_device: dict = {}

    def __init__(self, device: int = 0):
        lib = load()
        h = C.c_void_p()
        check(lib.trs_ctx_create(int(device), C.byref(h)), "trs_ctx_create")
        self.lib, self.handle, self.device = lib, h, int(device)
        sm, smem, maj, mnr = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        check(lib.trs_ctx_device_info(h, C.byref(sm), C.byref(smem), C.byref(maj), C.byref(mnr)), "trs_ctx_device_info")
        self.sm_count, self.smem_optin, self.cc = sm.value, smem.value, (maj.value, mnr.value)

    def close(self):
        if self.handle:
            self.lib.trs_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


def probe_fp64(device: int = 0):
    """(DFMA TFLOP/s, 10^12 DADD lane-instructions/s) measured on `device` (bench.py: denominator of the waypoint lookup's roofline)."""
    ctx = Context(device)
    try:
        a, b = C.c_double(), C.c_double()
        check(ctx.lib.trs_probe_fp64(ctx.handle, C.byref(a), C.byref(b)), "trs_probe_fp64")
        return a.value, b.value
    finally:
        ctx.close()


def kernel_launches() -> int:
    return int(load().trs_kernel_launches())


def preproc_params_from_cfg(cfg: dict) -> PreprocParams:
    """Reference key names (core/config.py:15-28); bounds may be lists after the JSON round trip (img_preprocessing.py:71)."""
    p = PreprocParams()
    p.contrast_ratio = float(cfg['preprocessing_contrast_enhancement_ratio'])
    p.contrast_offset = float(cfg['preprocessing_contrast_enhancement_offset'])
    p.brightness_baseline = float(cfg['preprocessing_brightness_baseline'])
    p.dynamic_brightness = int(bool(cfg['preprocessing_dynamic_brightness_enabled']))
    p.color_filter_enabled = int(bool(cfg['preprocessing_color_filter_enabled']))
    p.edge_enabled = int(bool(cfg['preprocessing_edge_detection_enabled']))
    if p.color_filter_enabled:
        hsvs = cfg['preprocessing_color_filter_hsvs']
        dests = cfg['preprocessing_color_filter_destination_channels']
        assert len(hsvs) == len(dests)          # img_preprocessing.py:59 (the reference asserts in __merge)
        if len(hsvs) > MAX_HSV:
            raise ValueError(f"at most {MAX_HSV} colour ranges are supported, got {len(hsvs)}")
        p.n_hsv = len(hsvs)
        for k, (lo, hi) in enumerate(hsvs):
            lo, hi = tuple(lo), tuple(hi)
            for c in range(3):
                p.hsv_lo[k][c] = float(lo[c])
                p.hsv_hi[k][c] = float(hi[c])
            p.color_dest[k] = int(dests[k])
    p.edge_dest = int(cfg['preprocessing_edge_detection_destination_channel'])
    p.canny_a = float(cfg['preprocessing_edge_detection_threshold_a'])
    p.canny_b = float(cfg['preprocessing_edge_detection_threshold_b'])
    return p


def ctl_params_from_cfg(cfg: dict, locks: bool = True, assist: bool = False) -> CtlParams:
    """Reference key names (core/config.py:57-63,104-106)."""
    p = CtlParams()
    if locks:
        p.throttle_lock_enabled = int(bool(cfg['ai_launch_boost_throttle_enabled']))
        p.throttle_lock_value = float(cfg['ai_launch_boost_throttle_value'])
        p.throttle_lock_duration = float(cfg['ai_launch_boost_throttle_duration'])
        p.steering_lock_enabled = int(bool(cfg['ai_launch_lock_steering_enabled']))
        p.steering_lock_value = float(cfg['ai_launch_lock_steering_value'])
        p.steering_lock_duration = float(cfg['ai_launch_lock_steering_duration'])
    if assist:
        mode = cfg['drive_assist_limit_mode']
        p.assist_mode = {'steering': 1, 'speed': 2}.get(mode, 0)          # any other string: neither branch of driver_assistance.py:16,25
        p.assist_k = float(cfg['drive_assist_limit_k'])
    return p


def spd_params_from_cfg(cfg: dict) -> SpdParams:
    p = SpdParams()
    p.threshold = float(cfg['spd_ctl_threshold'])
    p.reverse_multiplier = float(cfg['spd_ctl_reverse_multiplier'])
    p.break_multiplier = float(cfg['spd_ctl_break_multiplier'])
    p.use_break = int(bool(cfg['spd_ctl_break']))
    p.smooth_steering = int(bool(cfg['smooth_steering_enabled']))
    p.smooth_threshold = float(cfg['smooth_steering_threshold'])
    # not a reference key: which NumPy scalar promotion the caller's stack has (INTEGRATION.md, "NumPy promotion"); default NumPy >= 2
    p.numpy_legacy_promotion = int(bool(cfg.get('spd_ctl_numpy_legacy_promotion', False)))
    return p
