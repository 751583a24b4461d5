"""Both tub codecs at the sizes where their long-range arithmetic matters: the decoder past its first chunk of records and past 2^32
output bytes, the encoder past 2^32 input bytes and at the 240x320 batch DESIGN.md §4.7a measures.

The other decoder tests stay inside one chunk (at most 20,003 records of 120x160, 1.15 GB of output), so the record offset of the
second chunk's launches, the output offset c0 * h * w * 3 and the reuse of the plane staging between chunks never run there.  The
chunk rule is restated from trs_jpeg_decode_host (csrc/trs_api.cu); the chunk test asserts the trips it claims and fails by name if
the rule changes under it.  Every output is compared with Pillow on the device, in slices, against the Pillow decodes of the few
distinct files the batch is drawn from; nothing of the size of the batch is copied back."""
import io
import threading

import numpy as np
import pytest
import torch
from PIL import Image

from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200 import synth, tub

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]
DEV = "cuda:0"
DECODE_STAGING_BYTES = 8 << 30          # trs_api.cu trs_jpeg_decode_host: plane staging per chunk of records
SLICE = 2048                            # records per comparison on the device


def decode_chunk(h, w, hs, vs):
    """Records per chunk of trs_jpeg_decode_host: the staging bytes over the MCU-padded Y + Cb + Cr planes of one record."""
    mw, mh = -(-w // (8 * hs)), -(-h // (8 * vs))
    ybytes, cbytes = mw * 8 * hs * mh * 8 * vs, mw * 8 * mh * 8
    return DECODE_STAGING_BYTES // (ybytes + 2 * cbytes)


def need_free(nbytes):
    free, _ = torch.cuda.mem_get_info(0)
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 1e9:.0f} GB of free device memory, {free / 1e9:.0f} GB free")


@pytest.fixture
def ctx(record_property):
    """A context of its own, closed afterwards (its staging is gigabytes); the device memory in use is sampled every 50 ms and its
    peak recorded as a test property (device-wide: other processes on the GPU count too)."""
    torch.cuda.empty_cache()
    c = nat.Context(0)
    peak, stop = [0], threading.Event()

    def sample():
        while not stop.is_set():
            free, total = torch.cuda.mem_get_info(0)
            peak[0] = max(peak[0], total - free)
            stop.wait(0.05)
    t = threading.Thread(target=sample, daemon=True)
    t.start()
    yield c
    stop.set()
    t.join()
    record_property("peak_device_gb_in_use", round(peak[0] / 1e9, 1))
    c.close()
    torch.cuda.empty_cache()


def pil_files(frames, **kw):
    out = []
    for f in frames:
        buf = io.BytesIO()
        Image.fromarray(f).save(buf, format="JPEG", **kw)
        out.append(buf.getvalue())
    return out


def assert_decoded(got, want_dev, order):
    """Record k of `got` equals the Pillow decode of file order[k] (want_dev: those decodes on the device), slice by slice."""
    order_dev = torch.from_numpy(order).to(got.device)
    for s in range(0, got.shape[0], SLICE):
        e = min(got.shape[0], s + SLICE)
        bad = (got[s:e] != want_dev[order_dev[s:e]]).flatten(1).any(1).nonzero().flatten()
        assert bad.numel() == 0, f"{bad.numel()} of records {s}..{e - 1} differ; first {(bad[:5] + s).tolist()}"


def test_decoder_three_chunks_at_480x640(ctx):
    """4:4:4 480x640: 921,600 plane bytes per record, so a chunk is 9,320 records.  2 x 9,320 + 17 records (17.2 GB of output) make
    three chunks, the last one ragged; 8 files at two qualities (two table sets) in random order."""
    h, w = 480, 640
    chunk = decode_chunk(h, w, 1, 1)
    assert chunk == 9320, f"the decoder's chunk at {h}x{w} 4:4:4 is {chunk} records, the test is sized for 9,320"
    n = 2 * chunk + 17
    assert -(-n // chunk) == 3 and n % chunk, f"{n} records make {-(-n // chunk)} chunks of {chunk} (last {n % chunk})"
    need_free(n * h * w * 3 + DECODE_STAGING_BYTES + (6 << 30))
    pool = synth.frame_pool(8, h, w, seed=480)
    smooth = pool[np.arange(8) % 4 != 0][:4]                                # 35-70 KB files at these qualities
    files = pil_files(smooth, quality=40, subsampling=0) + pil_files(smooth, quality=50, subsampling=0)
    want = torch.from_numpy(np.stack([np.asarray(Image.open(io.BytesIO(f))) for f in files])).to(DEV)
    order = np.random.default_rng(480).integers(0, len(files), n)
    order[chunk - 1:chunk + 1] = [0, 7]                                     # different files on both sides of each chunk boundary
    order[2 * chunk - 1:2 * chunk + 1] = [3, 4]
    got = tub.decode_jpeg_batch([files[i] for i in order], ctx=ctx)
    assert got.shape == (n, h, w, 3) and got.numel() > 2 ** 34
    assert_decoded(got, want, order)
    del got
    # the same context again with the order reversed: the staging is reused, nothing may be left from the call before
    order = order[::-1].copy()
    got = tub.decode_jpeg_batch([files[i] for i in order], ctx=ctx)
    assert_decoded(got, want, order)


def test_decoder_past_4_gib_at_the_tub_shape(ctx):
    """75,000 records of 120x160 4:2:0 (4.32 GB of output, one chunk of 279,620): offsets past 2^32 bytes where a 32-bit product
    would wrap.  96 files at two qualities in random order."""
    h, w, n = 120, 160, 75000
    assert decode_chunk(h, w, 2, 2) == 279620 and n * h * w * 3 > 2 ** 32
    need_free(n * h * w * 3 + n * 30720 + (4 << 30))
    uniq = synth.frame_pool(96, h, w, seed=75)
    files = pil_files(uniq[:48]) + pil_files(uniq[48:], quality=92)
    want = torch.from_numpy(np.stack([np.asarray(Image.open(io.BytesIO(f))) for f in files])).to(DEV)
    order = np.random.default_rng(75).integers(0, len(files), n)
    got = tub.decode_jpeg_batch([files[i] for i in order], ctx=ctx)
    assert_decoded(got, want, order)


@pytest.mark.parametrize("h,w,n,decode", [(120, 160, 75000, True), (240, 320, 16384, False)])
def test_encoder_past_4_gib(ctx, h, w, n, decode):
    """75,000 x 120x160 (4.32 GB of input) and 16,384 x 240x320 (3.77 GB, the batch of DESIGN.md §4.7a) at quality 75, drawn from a
    pool of 64 frames: every offset and every file equal Pillow's bytes for its frame.  The 120x160 blob then goes back through the
    decoder."""
    need_free(2 * n * h * w * 3 + n * 30720 + (4 << 30))
    pool = synth.frame_pool(64, h, w, seed=h + w)
    ref = pil_files(pool, quality=75)
    order = np.random.default_rng(n).integers(0, 64, n)
    frames = torch.from_numpy(pool).to(DEV)[torch.from_numpy(order).to(DEV)]
    if (h, w) == (120, 160):
        assert frames.numel() > 2 ** 32
    blob, offsets = tub.encode_jpeg_batch(frames, 75, ctx=ctx)
    del frames
    sizes = np.asarray([len(f) for f in ref], np.uint64)
    bad = np.nonzero(np.diff(offsets) != sizes[order])[0]
    assert bad.size == 0, f"{bad.size} of {n} file sizes differ; first {bad[:5].tolist()}"
    want = np.frombuffer(b"".join(ref[i] for i in order), np.uint8)
    assert blob.size == want.size
    if not np.array_equal(blob, want):
        first = int(np.argmax(blob != want))
        raise AssertionError(f"files differ from Pillow's from byte {first} (record {int(np.searchsorted(offsets, first, 'right')) - 1})")
    if decode:
        got = tub.decode_jpeg_batch((blob, offsets), hw=(h, w), ctx=ctx)
        want_dev = torch.from_numpy(np.stack([np.asarray(Image.open(io.BytesIO(f))) for f in ref])).to(DEV)
        assert_decoded(got, want_dev, order)
