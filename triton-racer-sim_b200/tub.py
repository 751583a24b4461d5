"""Tub ingestion on the GPU (SURVEY.md §8(f) rank 1): the step before the observation path in "N tub records" mode.

The reference's trainers read a tub folder record by record (components/keras_train.py:33-57, 301-325):
``img_{i}.jpg`` through ``np.asarray(Image.open(path), dtype=np.float32)`` then ``/= 255`` and ``record_{i}.json`` through
``json.load``; the recorder writes them with ``Image.fromarray(img).save(path)`` (components/datastorage.py:67-79).  Here the JPEG
files of a batch are decoded by the CUDA kernels behind ``trs_jpeg_decode_host`` straight into the ``(N,H,W,3)`` uint8 device tensor
the rest of the path reads (bit-exact with Pillow's decoder), so only the ~5 KB files cross the PCIe link, not 57.6 KB of pixels.
The write side is the same trade in the other direction: ``encode_jpeg_batch`` / ``TubWriter`` encode device frames behind
``trs_jpeg_encode`` (byte-identical with Pillow's ``save``) and only the files come back to the host.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np
import torch

from . import _native as nat


def jpeg_size(data: bytes):
    """(height, width) from the SOF0 header of a baseline JPEG (no decoding)."""
    i = 2
    n = len(data)
    while i + 4 <= n:
        if data[i] != 0xFF:
            break
        m = data[i + 1]
        if m == 0xFF:
            i += 1
            continue
        seg_len = (data[i + 2] << 8) | data[i + 3]
        if 0xC0 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            return (data[i + 5] << 8) | data[i + 6], (data[i + 7] << 8) | data[i + 8]
        i += 2 + seg_len
    raise ValueError("not a JPEG file (no frame header found)")


def pack_files(files):
    """list of bytes -> (blob uint8 array, offsets uint64 array of N + 1 entries)."""
    sizes = np.fromiter((len(f) for f in files), dtype=np.uint64, count=len(files))
    offsets = np.zeros(len(files) + 1, np.uint64)
    np.cumsum(sizes, out=offsets[1:])
    blob = np.frombuffer(b"".join(files), dtype=np.uint8)
    return blob, offsets


def decode_jpeg_batch(files, hw=None, device=None, ctx=None, out=None) -> torch.Tensor:
    """Decode N baseline-JPEG tub images (bytes objects, or a (blob, offsets) pair) into a CUDA uint8 tensor (N,H,W,3)."""
    blob, offsets = files if isinstance(files, tuple) else pack_files(list(files))
    n = len(offsets) - 1
    if hw is None:
        if n == 0:
            raise ValueError("hw is required for an empty batch")
        hw = jpeg_size(bytes(blob[int(offsets[0]):int(offsets[1])]))
    h, w = int(hw[0]), int(hw[1])
    own = ctx is None
    dev = torch.cuda.current_device() if device is None else int(device if not isinstance(device, torch.device) else device.index)
    ctx = nat.Context(dev) if own else ctx
    try:
        if out is None:
            out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=f"cuda:{ctx.device}")
        blob = np.ascontiguousarray(blob, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        nat.check(ctx.lib.trs_jpeg_decode_host(ctx.handle, C.c_void_p(blob.ctypes.data), C.c_void_p(offsets.ctypes.data), n, h, w,
                                               C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream(ctx.device).cuda_stream)),
                  "trs_jpeg_decode_host")
    finally:
        if own:
            ctx.close()
    return out


def encode_jpeg_batch(frames: torch.Tensor, quality: int = 75, device=None, ctx=None):
    """Encode a CUDA uint8 (N,H,W,3) RGB tensor into N baseline-JPEG files, byte-identical with
    ``Image.fromarray(frame).save(f, "JPEG", quality=quality)`` (the recorder's call, datastorage.py:78; Pillow's default quality is 75,
    ``cv2.imencode``'s 95).  Returns ``(blob uint8 array, offsets uint64 array of N + 1 entries)``, the form ``decode_jpeg_batch``
    takes.  The encoding runs on the frames' stream-ordered position on the current stream; only the files are copied back."""
    if not isinstance(frames, torch.Tensor) or not frames.is_cuda:
        raise TypeError("frames must be a CUDA tensor")
    if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError(f"frames must be uint8 (N,H,W,3), got {tuple(frames.shape)} {frames.dtype}")
    if not frames.is_contiguous():
        raise ValueError("frames must be contiguous")
    quality = int(quality)
    n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    own = ctx is None
    dev = frames.device.index if device is None else int(device if not isinstance(device, torch.device) else device.index)
    if dev != frames.device.index:
        raise ValueError(f"frames are on cuda:{frames.device.index}, the encoder runs on cuda:{dev}")
    ctx = nat.Context(dev) if own else ctx
    try:
        if ctx.device != frames.device.index:
            raise ValueError(f"frames are on cuda:{frames.device.index}, the context on cuda:{ctx.device}")
        offsets = np.zeros(n + 1, np.uint64)
        stream = C.c_void_p(torch.cuda.current_stream(ctx.device).cuda_stream)
        nat.check(ctx.lib.trs_jpeg_encode(ctx.handle, C.c_void_p(frames.data_ptr() if n else 0), n, h, w, quality,
                                          C.c_void_p(offsets.ctypes.data), stream), "trs_jpeg_encode")
        blob = np.empty(int(offsets[n]), np.uint8)
        nat.check(ctx.lib.trs_jpeg_encode_copy(ctx.handle, C.c_void_p(blob.ctypes.data if blob.size else 0), C.c_ulonglong(blob.size), stream),
                  "trs_jpeg_encode_copy")
    finally:
        if own:
            ctx.close()
    return blob, offsets


class TubWriter:
    """The write side of ``TubReader``: a batch of records in the layout and numbering of the reference's recorder
    (components/datastorage.py:67-79, :98-112): ``img_{i}.jpg`` + ``record_{i}.json`` with ``'cam/img'`` holding the file name,
    numbered from 0 (the loaders read from 1, ``count_records``).  The frames are encoded on the GPU (``encode_jpeg_batch``), the
    files and JSON records are written by the host.  The recorder's thread, toggle and delete handling are not part of this."""

    def __init__(self, tub_path: str, device=None, quality: int = 75):
        self.path = tub_path
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.quality = int(quality)
        self.index = 0                                   # next record number (datastorage.py: the file thread counts from 0)
        self.ctx = nat.Context(self.device)
        os.makedirs(tub_path, exist_ok=True)

    def write(self, frames: torch.Tensor, records):
        """frames: CUDA uint8 (N,H,W,3) (the recorder's ``cam/img`` input); records: N dicts of the other values.  Returns the record
        numbers written."""
        records = list(records)
        if len(records) != int(frames.shape[0]):
            raise ValueError(f"{int(frames.shape[0])} frames but {len(records)} records")
        blob, offsets = encode_jpeg_batch(frames, self.quality, device=self.device, ctx=self.ctx)
        written = []
        for k, rec in enumerate(records):
            i = self.index + k
            name = f"img_{i}.jpg"
            with open(os.path.join(self.path, name), "wb") as f:
                f.write(blob[int(offsets[k]):int(offsets[k + 1])].tobytes())
            row = {"cam/img": name}
            row.update({key: v for key, v in rec.items() if key != "cam/img"})
            with open(os.path.join(self.path, f"record_{i}.json"), "w") as f:
                json.dump(row, f)
            written.append(i)
        self.index += len(records)
        return written

    def close(self):
        self.ctx.close()


# The reference's loader classes differ only in what they take from a record (keras_train.py:113-119, 264-299):
#   name -> (labels(record), features(record) or None); values become float32 as in keras_train.py:48-49.
LOADERS = {
    "DataLoader": (lambda r: (r['mux/steering'], r['mux/throttle']), None),                                   # :113-119
    "SpeedFeatureDataLoader": (lambda r: (r['mux/steering'], r['mux/throttle']), lambda r: (r['gym/speed'] / 20,)),   # :264-269
    "SpeedCtlDataLoader": (lambda r: (r['mux/steering'], r['gym/speed'] / 20), None),                         # :271-276
    "FullHouseDataLoader": (lambda r: (r['mux/steering'], r['gym/speed'] / 20),                                # :292-299
                            lambda r: (r['gym/speed'] / 20, r['loc/segment'])),
}
# the loader train() picks for each model type (keras_train.py:384-395)
LOADER_OF_MODEL = {"cnn_2d": "DataLoader", "cnn_2d_speed_as_feature": "SpeedFeatureDataLoader",
                   "cnn_2d_speed_control": "SpeedCtlDataLoader", "cnn_2d_full_house": "FullHouseDataLoader"}


def labels_and_features(records, loader="DataLoader"):
    """What the reference's ``DataLoader.load`` keeps of each record, gathered for a batch:
    labels (N, 2) float32 and features (N, k) float32 or None (keras_train.py:48-52)."""
    get_labels, get_features = LOADERS[LOADER_OF_MODEL.get(loader, loader)]
    labels = np.asarray([get_labels(r) for r in records], dtype=np.float32).reshape(len(records), -1)
    feats = None
    if get_features is not None:
        feats = np.asarray([get_features(r) for r in records], dtype=np.float32).reshape(len(records), -1)
    return labels, feats


def count_records(tub_path: str) -> int:
    """Number of complete records, counted as the reference does: consecutive indices from 1, the first missing file ends the folder
    (keras_train.py:36-39, 54-56)."""
    i = 1
    while os.path.exists(os.path.join(tub_path, f"record_{i}.json")) and os.path.exists(os.path.join(tub_path, f"img_{i}.jpg")):
        i += 1
    return i - 1


class TubReader:
    """A tub folder as the reference's loaders see it: records 1..N, ``img_{i}.jpg`` + ``record_{i}.json`` (keras_train.py:36-46)."""

    def __init__(self, tub_path: str, device=None):
        self.path = tub_path
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.ctx = nat.Context(self.device)

    def count(self) -> int:
        """Number of complete records, counted as the reference does: consecutive indices from 1 (keras_train.py:36-39)."""
        return count_records(self.path)

    def load(self, indices):
        """-> (frames (N,H,W,3) uint8 CUDA tensor, list of record dicts) for the given record indices."""
        files, records = [], []
        for i in indices:
            with open(os.path.join(self.path, f"img_{i}.jpg"), "rb") as f:
                files.append(f.read())
            with open(os.path.join(self.path, f"record_{i}.json")) as f:
                records.append(json.load(f))
        return decode_jpeg_batch(files, device=self.device, ctx=self.ctx), records

    def load_examples(self, indices, loader="DataLoader"):
        """One batch the way ``DataLoader.load`` builds its examples (keras_train.py:33-57): frames stay uint8 on the GPU (the `/255`
        is fused into the consumers), labels and feature vectors come back as float32 CUDA tensors."""
        frames, records = self.load(indices)
        labels, feats = labels_and_features(records, loader)
        dev = frames.device
        return frames, torch.from_numpy(labels).to(dev), None if feats is None else torch.from_numpy(feats).to(dev)

    def close(self):
        self.ctx.close()


def decode_telemetry_batch(packets, hw=None, device=None, ctx=None):
    """N simulator telemetry packets (the dicts ``GymInterface.on_msg_recv`` receives, components/gyminterface.py:95-104) ->
    ``{'cam/img': (N,H,W,3) uint8 CUDA tensor, 'gym/x', 'gym/y', 'gym/z', 'gym/speed', 'gym/cte': (N,) float64 CUDA tensors}``
    (the keys GymInterface publishes, gyminterface.py:52).  The base64 image strings are decoded and the JPEGs decompressed behind
    ``trs_telemetry_decode_host``."""
    n = len(packets)
    texts = [p["image"].encode("ascii") if isinstance(p["image"], str) else bytes(p["image"]) for p in packets]
    text, offsets = pack_files(texts)
    if hw is None:
        import base64
        head = b"".join(texts[0].split())[:2048]                       # the frame header sits in the first few hundred bytes
        head = head[:len(head) // 4 * 4]
        hw = jpeg_size(base64.b64decode(head + b"=" * (-len(head) % 4)))
    h, w = int(hw[0]), int(hw[1])
    own = ctx is None
    dev = torch.cuda.current_device() if device is None else int(device if not isinstance(device, torch.device) else device.index)
    ctx = nat.Context(dev) if own else ctx
    try:
        out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=f"cuda:{ctx.device}")
        text = np.ascontiguousarray(text, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        nat.check(ctx.lib.trs_telemetry_decode_host(ctx.handle, C.c_void_p(text.ctypes.data), C.c_void_p(offsets.ctypes.data), n, h, w,
                                                    C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream(ctx.device).cuda_stream)),
                  "trs_telemetry_decode_host")
    finally:
        if own:
            ctx.close()
    res = {"cam/img": out}
    for key, field in (("gym/x", "pos_x"), ("gym/y", "pos_y"), ("gym/z", "pos_z"), ("gym/speed", "speed"), ("gym/cte", "cte")):
        res[key] = torch.as_tensor(np.asarray([float(p[field]) for p in packets], np.float64), device=out.device)      # gyminterface.py:100-104
    return res
