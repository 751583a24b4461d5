"""CPU-side check of the tub-recording arithmetic: csrc/jpeg_enc_core.cuh (pure host/device functions, the same source the encoder
kernels compile) built with g++ and compared byte for byte with Pillow's ``Image.save`` — the encoder the reference's recorder calls
(datastorage.py:78) — with OpenCV's ``imencode`` (utils/post_process.py) and with the files the reference's recorder wrote into
tests/golden/tub.npz."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest
from PIL import Image

from tests.conftest import ROOT
from triton_racer_sim_b200 import synth

SIZES = [(1, 1), (2, 3), (7, 9), (17, 33), (24, 32), (120, 160), (121, 163), (240, 320)]
QUALITIES = [1, 10, 30, 50, 75, 95, 100]


@pytest.fixture(scope="module")
def enc_lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("jpe") / "libjpecheck.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", str(out), os.path.join(ROOT, "tests", "host_jpeg_encode_check.cpp")])
    lib = C.CDLL(str(out))
    lib.jpe_encode_host.restype = C.c_ulonglong
    lib.jpe_encode_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_ulonglong]
    lib.jpe_max_bytes_host.restype = C.c_ulonglong
    lib.jpe_max_bytes_host.argtypes = [C.c_int, C.c_int]
    return lib


@pytest.fixture(scope="module")
def dec_lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("jpd") / "libjpgcheck.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", str(out), os.path.join(ROOT, "tests", "host_jpeg_check.cpp")])
    lib = C.CDLL(str(out))
    lib.jpg_decode_rgb_host.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    return lib


def host_encode(lib, frame, quality):
    f = np.ascontiguousarray(frame, np.uint8)
    h, w, _ = f.shape
    cap = lib.jpe_max_bytes_host(h, w)
    out = np.zeros(cap, np.uint8)
    n = lib.jpe_encode_host(f.ctypes.data, h, w, quality, out.ctypes.data, cap)
    assert n > 0
    return out[:n].tobytes()


def pil_encode(frame, quality=None):
    buf = io.BytesIO()
    kw = {} if quality is None else dict(quality=quality)
    Image.fromarray(frame).save(buf, format="JPEG", **kw)
    return buf.getvalue()


def adversarial_frames(h, w, seed=0):
    """All 0, all 255, 1-px checkerboards (grey and colour), uniform noise: category-11 DC differences, 16-bit AC codes, ZRL runs,
    0xFF bytes to stuff."""
    y, x = np.mgrid[:h, :w]
    cb = (((x + y) & 1) * 255).astype(np.uint8)
    rng = np.random.default_rng(seed)
    return [np.zeros((h, w, 3), np.uint8), np.full((h, w, 3), 255, np.uint8), np.repeat(cb[..., None], 3, axis=2),
            np.stack([cb, 255 - cb, cb], axis=2), rng.integers(0, 256, (h, w, 3), dtype=np.uint8)]


@pytest.mark.parametrize("h,w", SIZES)
def test_host_encoder_matches_pillow(enc_lib, h, w):
    for q in QUALITIES:
        for f in synth.frame_pool(3, h, w, seed=h * 7 + w + q):
            assert host_encode(enc_lib, f, q) == pil_encode(f, q), (h, w, q)


def test_default_quality_is_pillows():
    f = synth.frame_pool(1, 24, 32, seed=4)[0]
    assert pil_encode(f) == pil_encode(f, 75)                    # save() without quality: what the recorder calls


@pytest.mark.parametrize("h,w", [(24, 32), (17, 33), (120, 160)])
def test_host_encoder_adversarial_frames(enc_lib, h, w):
    stuffed = 0
    for q in (1, 10, 50, 100):
        for f in adversarial_frames(h, w, seed=q):
            got = host_encode(enc_lib, f, q)
            assert got == pil_encode(f, q), (h, w, q)
            stuffed += got.count(b"\xff\x00")
    assert stuffed > 100                                          # the stuffing path is exercised


def test_host_encoder_matches_opencv_default_quality(enc_lib):
    cv2 = pytest.importorskip("cv2")
    for h, w in ((120, 160), (121, 163), (7, 9)):
        for f in synth.frame_pool(3, h, w, seed=h + w):
            ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(f[..., ::-1]))          # OpenCV's default: quality 95
            assert ok and host_encode(enc_lib, f, 95) == buf.tobytes(), (h, w)
            ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(f[..., ::-1]), [cv2.IMWRITE_JPEG_QUALITY, 75])
            assert ok and host_encode(enc_lib, f, 75) == buf.tobytes(), (h, w)


def test_host_encoder_reproduces_the_recorders_files(enc_lib):
    g = np.load(os.path.join(ROOT, "tests", "golden", "tub.npz"))
    blob = g["jpeg_blob"].tobytes()
    s = np.concatenate([[0], np.cumsum(g["jpeg_sizes"])])
    frames = g["recorded_frames_u8"]
    assert len(frames) == 8
    for i, f in enumerate(frames):
        assert host_encode(enc_lib, f, 75) == blob[s[i]:s[i + 1]], i


def test_host_round_trip_through_the_host_decoder(enc_lib, dec_lib):
    for h, w in ((120, 160), (121, 163), (2, 3)):
        for q in (30, 75, 100):
            for f in synth.frame_pool(2, h, w, seed=q + h):
                data = host_encode(enc_lib, f, q)
                out = np.zeros((h, w, 3), np.uint8)
                arr = np.frombuffer(data, np.uint8).copy()
                assert dec_lib.jpg_decode_rgb_host(arr.ctypes.data, len(data), h, w, out.ctypes.data) == 0
                assert np.array_equal(out, np.asarray(Image.open(io.BytesIO(data)))), (h, w, q)


def test_quantisation_reciprocals_and_header_length(enc_lib):
    """The reciprocal quantisation equals the division for every divisor 8q and every numerator below 2^16, and the header builder
    writes exactly JPE_HEADER_BYTES (the kernels place the entropy-coded data behind that many bytes)."""
    assert enc_lib.jpe_self_check_host() == 0
    f = np.zeros((5, 5, 3), np.uint8)
    data = pil_encode(f, 75)
    sos = data.index(b"\xff\xda")
    assert sos + 14 == 623


def test_host_encoder_under_address_and_ub_sanitizers(tmp_path):
    """Random sizes (1x1 up to 260x330), qualities and frames through the encoder built with -fsanitize=address,undefined, into a
    buffer of exactly the worst-case size, then through the product's parser and entropy decoder."""
    exe = tmp_path / "jpe_fuzz"
    build = subprocess.run(["g++", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer",
                            "-o", str(exe), os.path.join(ROOT, "tests", "host_jpeg_encode_fuzz.cpp")], capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("no sanitizer runtime in this toolchain: " + build.stderr[-200:])
    run = subprocess.run([str(exe), "400"], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-3000:]
    assert run.stdout.startswith("runs 400")
