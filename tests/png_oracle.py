"""Test oracle of the PNG decoder (csrc/dtfill_k8_png.cuh): a pure-Python writer of 16-bit grayscale PNGs that can
produce every kind of file the decoder must accept (any row filters, any zlib level and strategy, the stream split over
IDAT chunks of any size, ancillary chunks in between), and a zlib + numpy reader.  Never imported by the package."""
from __future__ import annotations

import struct
import zlib

import numpy as np

SIGNATURE = b"\x89PNG\r\n\x1a\n"
STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman": zlib.Z_HUFFMAN_ONLY,
              "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}


def chunk(ctype: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + ctype + data + struct.pack(">I", zlib.crc32(ctype + data) & 0xffffffff)


def ihdr(H: int, W: int, bit_depth: int = 16, colour: int = 0, interlace: int = 0) -> bytes:
    return chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, bit_depth, colour, 0, 0, interlace))


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(samples: np.ndarray, filters="msad", seed: int = 0) -> bytes:
    """The filtered scanlines of uint16 [H,W] samples.  filters: an int 0..4 for every row, a sequence of one per
    row, "random" (a random mix) or "msad" (per row the filter of least sum of absolute signed differences, the
    heuristic of libpng)."""
    H, W = samples.shape
    raw = samples.astype(">u2").view(np.uint8).reshape(H, 2 * W).astype(np.int32)
    up = np.vstack([np.zeros((1, 2 * W), np.int32), raw[:-1]])
    left = np.hstack([np.zeros((H, 2), np.int32), raw[:, :-2]])
    ul = np.hstack([np.zeros((H, 2), np.int32), up[:, :-2]])
    cand = np.stack([raw, raw - left, raw - up, raw - (left + up) // 2, raw - _paeth(left, up, ul)]) & 255
    if isinstance(filters, str) and filters == "msad":
        cost = np.minimum(cand, 256 - cand).sum(axis=2)
        ft = np.argmin(cost, axis=0)
    elif isinstance(filters, str) and filters == "random":
        ft = np.random.default_rng(seed).integers(0, 5, H)
    elif np.isscalar(filters):
        ft = np.full(H, int(filters))
    else:
        ft = np.asarray(filters)
    rows = cand[ft, np.arange(H)]
    return np.hstack([ft[:, None], rows]).astype(np.uint8).tobytes()


def compress(raw: bytes, level: int = 6, strategy: str = "default") -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 9, STRATEGIES[strategy])
    return c.compress(raw) + c.flush()


def split(z: bytes, idat="one", seed: int = 0) -> list:
    """IDAT payloads: "one" chunk, int n (n-byte chunks), "random" sizes with some empty chunks."""
    if idat == "one":
        return [z]
    if isinstance(idat, int):
        return [z[i:i + idat] for i in range(0, len(z), idat)] or [b""]
    rng = np.random.default_rng(seed)
    parts, i = [], 0
    while i < len(z):
        n = int(rng.integers(0, 4000)) if rng.random() < 0.8 else 0
        parts.append(z[i:i + n])
        i += n
    return parts or [b""]


def assemble(H: int, W: int, payloads, ancillary: bool = False, header: bytes | None = None) -> bytes:
    out = [SIGNATURE, header if header is not None else ihdr(H, W)]
    if ancillary:
        out.append(chunk(b"tEXt", b"Comment\x00between chunks"))
        out.append(chunk(b"gAMA", struct.pack(">I", 45455)))
    for i, p in enumerate(payloads):
        out.append(chunk(b"IDAT", p))
        if ancillary and i % 3 == 1:
            out.append(chunk(b"tIME", b"\x07\xea\x01\x02\x03\x04\x05"))
    out.append(chunk(b"IEND", b""))
    return b"".join(out)


def encode(samples: np.ndarray, filters="msad", level: int = 6, strategy: str = "default", idat="one",
           ancillary: bool = False, seed: int = 0) -> bytes:
    """uint16 [H,W] -> the bytes of a 16-bit grayscale PNG file."""
    samples = np.asarray(samples, np.uint16)
    H, W = samples.shape
    z = compress(filter_rows(samples, filters, seed), level, strategy)
    return assemble(H, W, split(z, idat, seed), ancillary)


def chunks(png: bytes):
    """[(type, payload)] of a well-formed file."""
    assert png[:8] == SIGNATURE
    out, pos = [], 8
    while pos < len(png):
        n, t = struct.unpack(">I4s", png[pos:pos + 8])
        out.append((t, png[pos + 8:pos + 8 + n]))
        pos += 12 + n
        if t == b"IEND":
            break
    return out


def decode(png: bytes) -> np.ndarray:
    """zlib + numpy reader of a 16-bit grayscale PNG -> uint16 [H,W]."""
    cs = chunks(png)
    W, H, depth, colour, _, _, interlace = struct.unpack(">IIBBBBB", cs[0][1])
    assert (depth, colour, interlace) == (16, 0, 0)
    raw = np.frombuffer(zlib.decompress(b"".join(p for t, p in cs if t == b"IDAT")), np.uint8)
    rows = raw.reshape(H, 1 + 2 * W)
    out = np.zeros((H, 2 * W), np.int32)
    prev = np.zeros(2 * W, np.int32)
    for r in range(H):
        ft, x = rows[r, 0], rows[r, 1:].astype(np.int32)
        if ft == 0:
            cur = x
        elif ft == 1:
            cur = np.cumsum(x.reshape(W, 2), axis=0).reshape(-1) & 255
        elif ft == 2:
            cur = (x + prev) & 255
        elif ft in (3, 4):
            cur = np.zeros(2 * W, np.int32)
            for c in range(0, 2 * W, 2):
                a = cur[c - 2:c] if c else np.zeros(2, np.int32)
                b = prev[c:c + 2]
                if ft == 3:
                    cur[c:c + 2] = (x[c:c + 2] + (a + b) // 2) & 255
                else:
                    cc = prev[c - 2:c] if c else np.zeros(2, np.int32)
                    cur[c:c + 2] = (x[c:c + 2] + _paeth(a, b, cc)) & 255
        else:
            raise ValueError(f"filter type {ft}")
        out[r] = cur
        prev = cur
    return out.astype(np.uint8).reshape(H, W, 2).view(">u2")[..., 0].astype(np.uint16)


def kitti_png_samples(seed: int, beams: int = 64) -> np.ndarray:
    """uint16 [448,1216]: a synthetic KITTI depth map as its PNG holds it (the 96 rows above the crop empty)."""
    from distancetransform_depthcompletion_b200 import synth
    x = synth.kitti_frame(seed, beam_step=64 // beams)
    out = np.zeros((448, 1216), np.uint16)
    out[96:] = np.round(x * 256).astype(np.uint16)
    return out
