"""Drop-ins for the compute of the reference's data_read.py that sits next to the hot path:

    outlier_removal(lidar)        data_read.py:103-128   (SURVEY.md section 8 f-2)
    read_depth_pngs(files)        data_read.py:215 / :223 `np.array(Image.open(f))`, a batch of files at once
    write_depth_pngs(batch)       its mirror: uint16 samples or depth in metres -> 16-bit grayscale PNG files

numpy in, numpy out; the 7 x 7 diamond filter runs on the GPU (kernel k6_outlier_removal), the PNG files are decoded on
the GPU (kernels k8_png_inflate, k8_png_unfilter) and encoded there (kernels k9_png_*).  The h5 reader of NYU is out of scope.
"""
from __future__ import annotations

import struct

import numpy as np

from . import _lib


def outlier_removal(lidar, device: int | None = None):
    """data_read.py:103-128: zero every depth that is more than 1.0 m farther than the average of the valid depths
    inside its 7 x 7 diamond.  A dropped depth becomes a zero of its own sign, as the reference's float64
    ``x * (1 - 1)`` gives (-0.0 for a negative depth).  Any shape that squeezes to [H,W]; returns float32 [H,W]."""
    sparse_lidar = np.squeeze(np.asarray(lidar))                              # :114
    if sparse_lidar.ndim != 2:
        raise ValueError(f"outlier_removal: input must squeeze to 2-D, got {np.shape(lidar)}")
    if sparse_lidar.dtype != np.float32:
        raise TypeError(f"outlier_removal: dtype {sparse_lidar.dtype} not supported by the CUDA path (float32 only)")
    return _lib.get_handle(device).outlier_removal(np.ascontiguousarray(sparse_lidar)[None])[0]


def _file_bytes(f) -> bytes:
    if isinstance(f, (bytes, bytearray, memoryview)):
        return bytes(f)
    with open(f, "rb") as fh:
        return fh.read()


def pack_png_files(files):
    """Files (paths or bytes) -> (data uint8, offsets int64 [B+1], H, W), the size read from the first file's IHDR."""
    blobs = [_file_bytes(f) for f in files]
    if not blobs:
        raise ValueError("read_depth_pngs: no files")
    head = blobs[0]
    if len(head) < 24 or head[:8] != b"\x89PNG\r\n\x1a\n" or head[12:16] != b"IHDR":
        raise ValueError("read_depth_pngs: file 0 is not a PNG file")
    W, H = struct.unpack(">II", head[16:24])
    offsets = np.zeros(len(blobs) + 1, np.int64)
    np.cumsum([len(b) for b in blobs], out=offsets[1:])
    return np.frombuffer(b"".join(blobs), np.uint8), offsets, int(H), int(W)


def read_depth_pngs(files, device: int | None = None) -> np.ndarray:
    """The reference's `np.array(Image.open(f))` of 16-bit grayscale PNGs (KITTI depth maps and ground truth,
    data_read.py:215, :223) for a batch of files, decoded on the GPU: uint16 [B,H,W].  files: paths or the files' bytes,
    all of the size the first file's IHDR gives.  Raises ValueError naming the first file that is not an intact 16-bit
    grayscale PNG of that size."""
    data, offsets, H, W = pack_png_files(files)
    out = _lib.output_empty((offsets.size - 1, H, W), np.uint16)
    return _lib.get_handle(device).png_decode(data, offsets, H, W, out=out)[0]


def write_depth_pngs(batch, paths=None, device: int | None = None) -> list:
    """The mirror of read_depth_pngs: a batch of depth maps encoded on the GPU as 16-bit grayscale PNG files (KITTI's
    depth format).  batch: uint16 samples [B,H,W], or float32 depth in metres [B,H,W] / [B,H,W,1], whose samples are

        sample = clip(nan_to_num(fl32(d * 256), nan=0, posinf=65535), 0, 65535) truncated toward zero,

    which equals (d * 256).astype(np.uint16) for every d in [0, 65535/256] (the usual way KITTI predictions are
    written) and is the identity on depths read from such files (d = k/256).  Returns the files' bytes; with ``paths``
    (one per frame) it also writes them.  Other dtypes raise TypeError, other shapes ValueError."""
    x = np.asarray(batch)
    if x.dtype not in (np.uint16, np.float32):
        raise TypeError(f"write_depth_pngs: uint16 samples or float32 depth expected, got {x.dtype}")
    if x.ndim == 4 and x.shape[-1] == 1 and x.dtype == np.float32:
        x = x[..., 0]
    if x.ndim != 3 or 0 in x.shape:
        raise ValueError(f"write_depth_pngs: expected [B,H,W] (or float32 [B,H,W,1]), got shape {np.shape(batch)}")
    if paths is not None:
        paths = list(paths)
        if len(paths) != x.shape[0]:
            raise ValueError(f"write_depth_pngs: {len(paths)} paths for {x.shape[0]} frames")
    h = _lib.get_handle(device)
    x = np.ascontiguousarray(x)
    files = h.png_encode(x) if x.dtype == np.uint16 else h.png_encode_depth(x)
    for p, f in zip(paths or (), files):
        with open(p, "wb") as fh:
            fh.write(f)
    return files
