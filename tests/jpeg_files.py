"""JPEG file families for the tub decoder's tests: what Pillow and OpenCV write besides Pillow's default files, the hand edits a
parser has to skip, and the files the decoder refuses.  Shared by the host build (test_jpeg_files_host.py) and the GPU path
(test_jpeg_files_gpu.py), so that both tiers see the same bytes.

Every family is a list of (name, bytes).  `accepted` adds each file's subsampling as Pillow codes it (0: 4:4:4, 1: 4:2:2, 2: 4:2:0),
read from its frame header: the decoder takes one subsampling per batch, and OpenCV picks 4:4:4 by itself when the luma and
chroma qualities are set."""
import io
import os

import numpy as np
from PIL import Image

from triton_racer_sim_b200 import synth

SIZES = [(1, 1), (2, 3), (7, 9), (121, 163), (120, 160), (240, 320)]
SUBSAMPLINGS = {0: "444", 1: "422", 2: "420"}


def pil_file(tmp_path, frame, **kw):
    """Pillow's file for `frame`, written through a path: to a BytesIO Pillow 12.2 stops some optimised-table files with
    "Suspension not allowed here" (even 120x160 4:4:4 q95).  Through a path it still refuses a noise frame at 240x320 4:4:4 q95
    optimised, so the families below are written from the pool's smooth and track-like frames, which it writes at every size."""
    p = os.path.join(str(tmp_path), "pil.jpg")
    Image.fromarray(frame).save(p, format="JPEG", **kw)
    with open(p, "rb") as f:
        return f.read()


def cv_file(frame, params):
    import cv2
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(frame[..., ::-1]), params)
    assert ok, params
    return buf.tobytes()


def pil_decode(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


def segments(data):
    """[(offset, marker, length)] of the marker segments before the scan data (SOS included); skips 0xFF fill bytes."""
    out, i = [], 2
    while i + 4 <= len(data):
        assert data[i] == 0xFF, i
        m = data[i + 1]
        if m == 0xFF:
            i += 1
            continue
        L = (data[i + 2] << 8) | data[i + 3]
        out.append((i, m, L))
        if m == 0xDA:
            break
        i += 2 + L
    return out


def table_bytes(data, markers=(0xDB, 0xC4)):
    """The DQT and DHT segments of a file, concatenated: two files with equal strings share one decoder table set."""
    return b"".join(data[i:i + 2 + L] for i, m, L in segments(data) if m in markers)


def subsampling(data):
    """Pillow's subsampling code of a file from the luma sampling factors in its SOF0 segment."""
    i = next(i for i, m, _ in segments(data) if m == 0xC0)
    return {0x11: 0, 0x21: 1, 0x22: 2}[data[i + 11]]


def huffman_symbol_counts(data):
    """Number of symbols of every Huffman table the file defines."""
    counts = []
    for i, m, L in segments(data):
        o, end = i + 4, i + 2 + L
        while m == 0xC4 and o + 17 <= end:
            n = sum(data[o + 1:o + 17])
            counts.append(n)
            o += 17 + n
    return counts


def insert_before(data, marker, extra):
    """`extra` inserted in front of the first segment with `marker`."""
    i = next(i for i, m, _ in segments(data) if m == marker)
    return data[:i] + extra + data[i:]


def optimised(tmp_path, frame):
    """Pillow optimize=True at every subsampling and three qualities, OpenCV IMWRITE_JPEG_OPTIMIZE (4:2:0, q95).  Optimised tables
    follow the file's own symbol counts: code-length distributions unlike Annex K, down to one-symbol tables at 1x1."""
    import cv2
    out = []
    for sub in (2, 1, 0):
        for q in (30, 75, 95):
            out.append((f"pil-opt-{SUBSAMPLINGS[sub]}-q{q}", pil_file(tmp_path, frame, quality=q, subsampling=sub, optimize=True)))
    out.append(("cv-opt", cv_file(frame, [cv2.IMWRITE_JPEG_OPTIMIZE, 1])))
    return out


def opencv(frame):
    """OpenCV's own files: the default (q95, 4:2:0), separate luma / chroma qualities and the 4:2:2 / 4:4:4 sampling factors."""
    import cv2
    return [("cv-default", cv_file(frame, [])),
            ("cv-luma40-chroma90", cv_file(frame, [cv2.IMWRITE_JPEG_LUMA_QUALITY, 40, cv2.IMWRITE_JPEG_CHROMA_QUALITY, 90])),
            ("cv-luma90-chroma20", cv_file(frame, [cv2.IMWRITE_JPEG_LUMA_QUALITY, 90, cv2.IMWRITE_JPEG_CHROMA_QUALITY, 20])),
            ("cv-422", cv_file(frame, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422])),
            ("cv-444", cv_file(frame, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]))]


def icc_profile(size=70000):
    """Opaque profile bytes; past 65,519 bytes Pillow splits the profile over several APP2 segments."""
    return b"\x00\x00\x00\x00not-a-real-profile" + np.random.default_rng(4).integers(0, 256, size, dtype=np.uint8).tobytes()


def with_segments(tmp_path, frame, quality=75, sub=2):
    """Files with segments the parser skips: EXIF (APP1), an ICC profile (APP2 x 2), a comment (COM), 0xFF fill bytes in front of
    two markers, a DRI segment with interval 0 and bytes after EOI.  All at the recorder's defaults otherwise."""
    exif = Image.Exif()
    exif[0x010F] = "maker"
    exif[0x010E] = "d" * 3000                                        # ImageDescription: a larger APP1
    kw = dict(quality=quality, subsampling=sub)
    plain = pil_file(tmp_path, frame, **kw)
    return [("exif", pil_file(tmp_path, frame, exif=exif.tobytes(), **kw)),
            ("icc", pil_file(tmp_path, frame, icc_profile=icc_profile(), **kw)),
            ("comment", pil_file(tmp_path, frame, comment=b"recorded by a test", **kw)),
            ("fill-bytes", insert_before(insert_before(plain, 0xC0, b"\xff" * 3), 0xDA, b"\xff" * 7)),
            ("dri-0", insert_before(plain, 0xDB, b"\xff\xdd\x00\x04\x00\x00")),
            ("after-eoi", plain + b"\x00\x01trailing bytes\xff\xd9\xff")]


def accepted(tmp_path, h, w, seed=0):
    """Every accepted family at (h, w): a noise-free synthetic frame for the optimised and OpenCV files, a second frame for the
    segment edits."""
    frames = synth.frame_pool(4, h, w, seed=seed + 31 * h + w)
    files = optimised(tmp_path, frames[1]) + opencv(frames[3]) + with_segments(tmp_path, frames[2])
    return [(name, subsampling(data), data) for name, data in files]


def refused(tmp_path, frame):
    """Files the parser refuses as unsupported (100 + JPG_E_UNSUPPORTED on the host build): 4:1:1 and 4:4:0 sampling factors,
    restart intervals from OpenCV and Pillow, and separate Cb / Cr quantisation tables (Pillow with three qtables)."""
    import cv2
    return [("cv-411", cv_file(frame, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])),
            ("cv-440", cv_file(frame, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440])),
            ("cv-restart", cv_file(frame, [cv2.IMWRITE_JPEG_RST_INTERVAL, 4])),
            ("pil-restart", pil_file(tmp_path, frame, restart_marker_blocks=2)),
            ("pil-three-qtables", pil_file(tmp_path, frame, qtables=[list(range(1, 65)), [2] * 64, [3] * 64]))]
