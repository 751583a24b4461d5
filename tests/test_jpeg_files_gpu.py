"""The GPU JPEG decoder on every file family it accepts (tests/jpeg_files.py), against Pillow bit for bit, and its refusals.

The rest of the suite feeds the kernels Pillow's default files: Annex K Huffman tables, one or a few table sets per batch.  Here the
device-only code meets what else the parser lets through: optimised tables (code-length distributions unlike Annex K, one-symbol
tables at 1x1) in the bit reader's look-ahead and maxcode paths, one CTA staging 64 table sets in turn, segments the parser skips
next to plain files (both branches of the "same header bytes as the previous file" reuse), the byte path of the upsampler, and the
threaded host stages (header parse, base64) with their first-bad-record reductions.

Launch and thread rules restated from csrc/trs_api.cu / jpeg_kernels.cuh; a test that depends on one states it and fails by name if
the rule changes under it."""
import base64
import os

import numpy as np
import pytest
import torch

from tests import jpeg_files as J
from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200 import synth, tub

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
JPG_THREADS = 64                      # jpeg_kernels.cuh: records per k_jpeg_entropy CTA
MAX_TABLE_SETS = 64                   # trs_api.cu trs_jpeg_decode_host: distinct table sets per batch
PARSE_THREADS = min(16, os.cpu_count() or 1)      # trs_api.cu: host threads for the header parse and base64 stages ...
THREADED_FROM = 64 * PARSE_THREADS                # ... used from 64 records per thread on


@pytest.fixture(scope="module")
def ctx():
    c = nat.Context(0)
    yield c
    c.close()


def thread_ranges(n):
    """The record range of every host thread for a batch of n (trs_api.cu: ceil(n / threads) records each)."""
    assert n >= THREADED_FROM and PARSE_THREADS >= 2, \
        f"{n} records on {PARSE_THREADS} threads: the test needs the threaded host stage (n >= {THREADED_FROM}, >= 2 threads)"
    per = -(-n // PARSE_THREADS)
    return [(k0, min(n, k0 + per)) for k0 in range(0, n, per)]


def check(got, files, label=""):
    got = got.cpu().numpy()
    for k, data in enumerate(files):
        want = J.pil_decode(data)
        assert np.array_equal(got[k], want), f"{label} record {k}: {int((got[k] != want).sum())} of {want.size} bytes differ"


@pytest.mark.parametrize("h,w", J.SIZES)
def test_every_accepted_family(ctx, tmp_path, h, w):
    """Optimised tables (Pillow at three qualities and every subsampling, OpenCV), OpenCV's defaults, separate luma / chroma
    qualities and sampling factors, EXIF / ICC / comment / fill bytes / DRI 0 / bytes after EOI: each file alone, and every
    subsampling's files as one batch with several table sets in one CTA."""
    fam = J.accepted(tmp_path, h, w)
    for name, _, data in fam:
        check(tub.decode_jpeg_batch([data], hw=(h, w), ctx=ctx), [data], name)
    for sub in (0, 1, 2):
        files = [data for _, s, data in fam if s == sub]
        assert len({J.table_bytes(f) for f in files}) >= 2
        check(tub.decode_jpeg_batch(files, hw=(h, w), ctx=ctx), files, f"subsampling {sub}")


def test_segments_next_to_plain_files_in_runs_and_alternating(ctx, tmp_path):
    """Files with skipped segments in runs (three frames each with equal header bytes: the reuse branch) and alternating with plain
    files (a new parse per file), 120x160 4:2:0 q75."""
    frames = synth.frame_pool(12, 120, 160, seed=41)
    plain = [J.pil_file(tmp_path, f) for f in frames]
    seg = [J.with_segments(tmp_path, f) for f in frames[1:4]]                # 3 frames x 6 kinds
    kinds = len(seg[0])
    runs = plain[:3] + [seg[j][i][1] for i in range(kinds) for j in range(3)] + plain[3:6]
    header = lambda d: d[:J.segments(d)[-1][0] + 2 + J.segments(d)[-1][2]]                 # up to the end of the SOS segment
    assert all(header(seg[0][i][1]) == header(seg[j][i][1]) for i in range(kinds) for j in (1, 2))
    alternating = [f for i in range(kinds) for f in (plain[i], seg[i % 3][i][1])]
    for files in (runs, alternating, runs + alternating):
        check(tub.decode_jpeg_batch(files, ctx=ctx), files)


@pytest.fixture(scope="module")
def optimised_64(tmp_path_factory):
    """64 optimised 120x160 files of 64 different frames: 64 distinct DQT + DHT byte strings."""
    tmp = tmp_path_factory.mktemp("opt64")
    frames = synth.frame_pool(65, 120, 160, seed=64)
    files = [J.pil_file(tmp, f, optimize=True) for f in frames]
    assert len({J.table_bytes(f) for f in files}) == 65, "the files do not carry 65 distinct table sets"
    return files, np.stack([J.pil_decode(f) for f in files])


def test_one_cta_walks_64_table_sets(ctx, optimised_64):
    files, want = optimised_64
    files, want = files[:MAX_TABLE_SETS], want[:MAX_TABLE_SETS]
    assert len(files) == JPG_THREADS, "64 records must fill exactly one k_jpeg_entropy CTA"
    got = tub.decode_jpeg_batch(files, ctx=ctx).cpu().numpy()
    for k in range(len(files)):
        assert np.array_equal(got[k], want[k]), f"record {k} (table set {k} of the CTA)"
    order = np.random.default_rng(5).integers(0, MAX_TABLE_SETS, 5000)
    got = tub.decode_jpeg_batch([files[i] for i in order], ctx=ctx)
    want_dev = torch.from_numpy(want).to(got.device)
    bad = (got != want_dev[torch.from_numpy(order).to(got.device)]).flatten(1).any(1).nonzero().flatten().tolist()
    assert not bad, f"{len(bad)} of 5000 records differ; first {bad[:5]} (files {order[bad[:5]].tolist()})"


def test_65_table_sets_are_refused_and_the_context_recovers(ctx, optimised_64):
    files, want = optimised_64
    with pytest.raises(ValueError, match="more than 64 distinct"):
        tub.decode_jpeg_batch(files, ctx=ctx)
    with pytest.raises(ValueError, match="more than 64 distinct"):
        tub.decode_jpeg_batch(files[1:] + files[:1] * 200, ctx=ctx)
    got = tub.decode_jpeg_batch(files[1:], ctx=ctx).cpu().numpy()
    assert np.array_equal(got, want[1:])


@pytest.mark.parametrize("kind", ["cv-411", "cv-440", "cv-restart", "pil-restart", "pil-three-qtables"])
def test_refusals_name_the_first_bad_record(ctx, tmp_path, kind):
    """A refused file at the end of the first parse thread's range and another at the start of the second's: the error names the
    lower record, whichever thread finds its record first."""
    frames = synth.frame_pool(16, 120, 160, seed=77)
    plain = [J.pil_file(tmp_path, f) for f in frames]
    bad = dict(J.refused(tmp_path, frames[5]))[kind]
    n = 2048
    (_, lo_end), (hi, _) = thread_ranges(n)[:2]
    lo = lo_end - 1
    files = [plain[k % 16] for k in range(n)]
    files[lo] = files[hi] = bad
    with pytest.raises(ValueError, match=f"record {lo}: not a baseline"):
        tub.decode_jpeg_batch(files, ctx=ctx)
    with pytest.raises(ValueError, match=f"record {hi}: not a baseline"):
        tub.decode_jpeg_batch(files[:lo] + [plain[0]] + files[lo + 1:], ctx=ctx)
    check(tub.decode_jpeg_batch(plain, ctx=ctx), plain)


def test_upsampler_byte_path_on_an_odd_address(ctx, tmp_path):
    """120x160 4:2:0 into an out= view 1 byte into its allocation: w % 4 == 0 alone would take the word path, the address does not
    allow it; the bytes around the view stay untouched."""
    frames = synth.frame_pool(300, 120, 160, seed=88)
    files = [J.pil_file(tmp_path, f, quality=q) for f, q in zip(frames, [75, 92] * 150)]
    n, h, w = len(files), 120, 160
    buf = torch.full((n * h * w * 3 + 2,), 0xA5, dtype=torch.uint8, device="cuda:0")
    out = buf[1:-1].view(n, h, w, 3)
    assert out.data_ptr() % 4 == 1
    tub.decode_jpeg_batch(files, ctx=ctx, out=out)
    assert buf[0].item() == 0xA5 and buf[-1].item() == 0xA5
    check(out, files, "byte path")
    aligned = tub.decode_jpeg_batch(files, ctx=ctx)
    assert torch.equal(aligned, out)


def telemetry_text(data, k):
    """A base64 string the way a client may send it: MIME (76) or CRLF (64) line breaks, no padding, runs of white space."""
    t = base64.b64encode(data).decode()
    if k % 3 == 0:
        t = "\n".join(t[i:i + 76] for i in range(0, len(t), 76))
    elif k % 3 == 1:
        t = "\r\n".join(t[i:i + 64] for i in range(0, len(t), 64))
    if k % 5 == 0:
        t = t.rstrip("=")
    if k % 7 == 0:
        t = " \t  ".join(t[i:i + 100] for i in range(0, len(t), 100))
    if k % 11 == 0:
        t = "\n  " + t + " \r\n\t"
    return t


def test_telemetry_on_the_threaded_base64_decoder(ctx, tmp_path):
    """3,000 packets through the threaded base64 stage (the slots are sized from the text length, so every file is moved when the
    slots are compacted), all equal to Pillow; two corrupt strings in different threads' ranges: the error names the first."""
    frames = synth.frame_pool(96, 120, 160, seed=99)
    files = [J.pil_file(tmp_path, f, quality=q) for f, q in zip(frames, [75, 60, 92] * 32)]
    want = torch.from_numpy(np.stack([J.pil_decode(f) for f in files])).cuda()
    n = 3000
    order = np.random.default_rng(6).integers(0, len(files), n)
    packets = [{"image": telemetry_text(files[i], k), "pos_x": 0.0, "pos_y": 1.0, "pos_z": float(k), "speed": 2.0, "cte": "0.5"}
               for k, i in enumerate(order)]
    got = tub.decode_telemetry_batch(packets, ctx=ctx)
    img = got["cam/img"]
    bad = (img != want[torch.from_numpy(order).cuda()]).flatten(1).any(1).nonzero().flatten().tolist()
    assert not bad, f"{len(bad)} of {n} packets differ; first {bad[:5]}"
    assert np.array_equal(got["gym/z"].cpu().numpy(), np.arange(n, dtype=np.float64))
    ranges = thread_ranges(n)
    lo, hi = ranges[0][1] - 1, ranges[-1][0]
    for k in (lo, hi):
        s = packets[k]["image"]
        packets[k] = dict(packets[k], image=s[:300] + "*" + s[301:])
    with pytest.raises(ValueError, match=f"packet {lo}: the image string is not valid base64"):
        tub.decode_telemetry_batch(packets, hw=(120, 160), ctx=ctx)
