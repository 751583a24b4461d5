"""Tub recording: the CUDA JPEG encoder against Pillow's ``Image.save`` (the encoder the reference's recorder calls, datastorage.py:78),
byte for byte, and its round trips through the GPU decoder and the tub reader."""
import io
import json
import os

import numpy as np
import pytest
import torch
from PIL import Image

from tests.test_jpeg_encode_host import QUALITIES, SIZES, adversarial_frames, pil_encode
from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200 import synth, tub

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def files_of(blob, offsets):
    return [blob[int(offsets[k]):int(offsets[k + 1])].tobytes() for k in range(len(offsets) - 1)]


@pytest.mark.parametrize("h,w", SIZES)
def test_encoder_matches_pillow(h, w):
    frames = synth.frame_pool(6, h, w, seed=h * 5 + w)
    dev = torch.from_numpy(frames).cuda(0)
    for q in QUALITIES:
        blob, offsets = tub.encode_jpeg_batch(dev, quality=q, device=0)
        assert offsets.dtype == np.uint64 and len(offsets) == 7 and offsets[0] == 0
        assert files_of(blob, offsets) == [pil_encode(f, q) for f in frames], (h, w, q)


def test_default_quality_and_recorder_fixture():
    g = np.load(os.path.join(ROOT, "tests", "golden", "tub.npz"))
    blob, offsets = tub.encode_jpeg_batch(torch.from_numpy(g["recorded_frames_u8"]).cuda(0))       # quality 75: save()'s default
    assert blob.tobytes() == g["jpeg_blob"].tobytes()
    assert np.array_equal(np.diff(offsets).astype(np.int64), g["jpeg_sizes"])


def test_large_mixed_batch_at_quality_100():
    """20,003 records: maximum-entropy (noise, checkerboards) and ordinary frames in random order at quality 100, where a record can
    be several times its usual size.  Every offset and every packed file is checked."""
    uniq = adversarial_frames(120, 160, seed=3) + list(synth.frame_pool(11, 120, 160, seed=29))
    want_u = [pil_encode(f, 100) for f in uniq]
    n = 20003
    order = np.random.default_rng(4).integers(0, len(uniq), n)
    dev = torch.from_numpy(np.stack(uniq)).cuda(0)[torch.from_numpy(order).cuda(0)].contiguous()
    blob, offsets = tub.encode_jpeg_batch(dev, quality=100, device=0)
    sizes = np.asarray([len(want_u[i]) for i in order], np.uint64)
    assert np.array_equal(np.diff(offsets), sizes) and int(offsets[-1]) == blob.size
    want = b"".join(want_u[i] for i in order)
    assert blob.tobytes() == want
    assert max(len(f) for f in want_u) > 2 * min(len(f) for f in want_u[5:])        # the noise frame: over twice an ordinary file


def test_round_trip_through_the_gpu_decoder():
    frames = synth.frame_pool(40, 121, 163, seed=5)
    for q in (50, 95):
        packed = tub.encode_jpeg_batch(torch.from_numpy(frames).cuda(0), quality=q)
        got = tub.decode_jpeg_batch(packed, device=0).cpu().numpy()
        want = np.stack([np.asarray(Image.open(io.BytesIO(pil_encode(f, q)))) for f in frames])
        assert np.array_equal(got, want)


def test_full_chain_then_encode():
    """What the recorder stores (cam/processed_img, manage.py:103-104): the chain on the GPU, then the encoder, against Pillow applied
    to the oracle chain's output."""
    import oracle
    from triton_racer_sim_b200 import ImgPreprocessing
    from triton_racer_sim_b200.config import full_house_config
    cfg = full_house_config()
    frames = synth.frame_pool(64, 120, 160, seed=8)
    comp = ImgPreprocessing(cfg, device=0)
    u8, _ = comp.process_device(torch.from_numpy(frames).cuda(0))
    blob, offsets = tub.encode_jpeg_batch(u8)
    comp.onShutdown()
    assert files_of(blob, offsets) == [pil_encode(f) for f in oracle.process_batch(frames, cfg)]


def test_tub_writer_then_reader(tmp_path):
    frames = synth.frame_pool(9, 120, 160, seed=12)
    records = [{"mux/steering": 0.1 * i, "mux/throttle": 0.5, "gym/speed": 2.0 * i} for i in range(9)]
    wr = tub.TubWriter(str(tmp_path), device=0)
    assert wr.write(torch.from_numpy(frames[:5]).cuda(0), records[:5]) == [0, 1, 2, 3, 4]
    assert wr.write(torch.from_numpy(frames[5:]).cuda(0), records[5:]) == [5, 6, 7, 8]
    wr.close()
    names = sorted(os.listdir(tmp_path))
    assert names == sorted([f"img_{i}.jpg" for i in range(9)] + [f"record_{i}.json" for i in range(9)])
    for i in range(9):
        with open(os.path.join(tmp_path, f"img_{i}.jpg"), "rb") as f:
            assert f.read() == pil_encode(frames[i])
        with open(os.path.join(tmp_path, f"record_{i}.json")) as f:
            rec = json.load(f)
        assert rec["cam/img"] == f"img_{i}.jpg" and rec["gym/speed"] == 2.0 * i
    # the fixture's records name their files the same way, from 0
    g = np.load(os.path.join(ROOT, "tests", "golden", "tub.npz"))
    assert [r["cam/img"] for r in json.loads(bytes(g["records_json"]).decode())] == [f"img_{i}.jpg" for i in range(8)]
    # the loaders read from 1 (keras_train.py:36): record 0 is written but never loaded
    assert tub.count_records(str(tmp_path)) == 8
    rd = tub.TubReader(str(tmp_path), device=0)
    got, recs = rd.load(range(1, 9))
    want = np.stack([np.asarray(Image.open(io.BytesIO(pil_encode(f)))) for f in frames[1:]])
    assert np.array_equal(got.cpu().numpy(), want) and [r["mux/steering"] for r in recs] == [0.1 * i for i in range(1, 9)]
    rd.close()


def test_stream_ordered_behind_the_chain():
    """The encoder reads the chain's output on the same stream with no host synchronisation in between."""
    from triton_racer_sim_b200 import ImgPreprocessing
    from triton_racer_sim_b200.config import full_house_config
    import oracle
    cfg = full_house_config()
    frames = synth.frame_pool(2000, 120, 160, seed=14)
    src = torch.from_numpy(frames).pin_memory()
    comp = ImgPreprocessing(cfg, device=0)
    s = torch.cuda.Stream(0)
    with torch.cuda.stream(s):
        dev = src.cuda(0, non_blocking=True)
        u8, _ = comp.process_device(dev)
        blob, offsets = tub.encode_jpeg_batch(u8)
    comp.onShutdown()
    want = oracle.process_batch(frames[:200], cfg)
    assert files_of(blob, offsets)[:200] == [pil_encode(f) for f in want]


def test_caller_device_and_staging_growth():
    torch.cuda.set_device(0)
    ctx = nat.Context(0)
    try:
        for n, (h, w), q in ((3, (24, 32), 75), (50, (120, 160), 90), (400, (240, 320), 100), (7, (17, 33), 10), (1200, (120, 160), 100)):
            frames = synth.frame_pool(min(n, 16), h, w, seed=n)
            frames = np.concatenate([frames] * ((n + 15) // 16))[:n]
            blob, offsets = tub.encode_jpeg_batch(torch.from_numpy(frames).cuda(0), quality=q, ctx=ctx)
            assert torch.cuda.current_device() == 0
            assert files_of(blob, offsets) == [pil_encode(f, q) for f in frames], (n, h, w, q)
    finally:
        ctx.close()
    if torch.cuda.device_count() > 1:
        torch.cuda.set_device(1)
        try:
            f = torch.from_numpy(synth.frame_pool(2, 24, 32, seed=1)).cuda(0)
            blob, offsets = tub.encode_jpeg_batch(f)
            assert torch.cuda.current_device() == 1
            assert files_of(blob, offsets) == [pil_encode(x) for x in f.cpu().numpy()]
        finally:
            torch.cuda.set_device(0)


def test_bad_arguments_are_rejected():
    import ctypes as C
    f = torch.from_numpy(synth.frame_pool(2, 24, 32, seed=2)).cuda(0)
    with pytest.raises(TypeError):
        tub.encode_jpeg_batch(f.cpu())
    with pytest.raises(ValueError):
        tub.encode_jpeg_batch(f.float())
    with pytest.raises(ValueError):
        tub.encode_jpeg_batch(f[..., :2].contiguous())
    with pytest.raises(ValueError):
        tub.encode_jpeg_batch(f[:, :, ::2])
    for q in (0, 101, -5):
        with pytest.raises(ValueError):
            tub.encode_jpeg_batch(f, quality=q)
    ctx = nat.Context(0)
    try:
        lib, hnd = ctx.lib, ctx.handle
        offs = np.zeros(3, np.uint64)
        st = C.c_void_p(0)
        p = C.c_void_p(f.data_ptr())
        assert lib.trs_jpeg_encode_copy(hnd, C.c_void_p(0), 0, st) == -2                     # no encode yet
        assert lib.trs_jpeg_encode(hnd, p, 2, 0, 32, 75, C.c_void_p(offs.ctypes.data), st) == -1
        assert lib.trs_jpeg_encode(hnd, p, 2, 24, 65536, 75, C.c_void_p(offs.ctypes.data), st) == -1
        assert lib.trs_jpeg_encode(hnd, p, -1, 24, 32, 75, C.c_void_p(offs.ctypes.data), st) == -1
        assert lib.trs_jpeg_encode(hnd, p, 2, 24, 32, 75, C.c_void_p(0), st) == -1
        assert lib.trs_jpeg_encode(hnd, C.c_void_p(0), 2, 24, 32, 75, C.c_void_p(offs.ctypes.data), st) == -1
        assert lib.trs_jpeg_encode(C.c_void_p(0), p, 2, 24, 32, 75, C.c_void_p(offs.ctypes.data), st) == -1
        assert lib.trs_jpeg_encode(hnd, p, 2, 24, 32, 75, C.c_void_p(offs.ctypes.data), st) == 0
        blob = np.zeros(int(offs[2]) + 1, np.uint8)
        assert lib.trs_jpeg_encode_copy(hnd, C.c_void_p(blob.ctypes.data), int(offs[2]) + 1, st) == -1      # wrong byte count
        assert b"bytes" in lib.trs_last_error()
        assert lib.trs_jpeg_encode_copy(hnd, C.c_void_p(0), int(offs[2]), st) == -1
        assert lib.trs_jpeg_encode_copy(hnd, C.c_void_p(blob.ctypes.data), int(offs[2]), st) == 0
        assert blob[:int(offs[1])].tobytes() == pil_encode(f[0].cpu().numpy())
    finally:
        ctx.close()
    empty = tub.encode_jpeg_batch(torch.empty((0, 24, 32, 3), dtype=torch.uint8, device="cuda:0"))
    assert empty[0].size == 0 and list(empty[1]) == [0]
