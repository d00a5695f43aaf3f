"""The PNG encoder (csrc/dtfill_k9_png_encode.cuh) run serially on the CPU through dtfill_debug_png_encode_host, which
writes the bytes the device writes: the files decode to the samples through four independent readers, the filter bytes
are libpng's heuristic, every checksum is right, the size stays within the bound, and the compression is close to zlib
level 1.  The depth -> sample rule is checked against its numpy expression.  No GPU needed."""
import io
import struct
import zlib

import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib, data_read, synth

SHAPES = [(1, 1), (3, 2), (1, 1216), (448, 1), (448, 37), (352, 1216), (448, 1216)]


@pytest.fixture(scope="module")
def lib(dtfill_lib):
    return _lib.load()


def _filled(seed, beams):
    from oracle import oracle as O
    d = O.dt_fill(synth.kitti_frame(seed, beam_step=64 // beams))["depth"]
    return (d * 256).astype(np.uint16)


def _cases(H, W):
    rng = np.random.default_rng(H * 10007 + W)
    yield "zeros", np.zeros((H, W), np.uint16)
    yield "max", np.full((H, W), 65535, np.uint16)
    yield "extremes", np.where((np.arange(H)[:, None] + np.arange(W)) % 2 == 0, 0, 65535).astype(np.uint16)
    yield "noise", rng.integers(0, 65536, (H, W)).astype(np.uint16)
    yield "sparse", ((rng.random((H, W)) < 0.1) * rng.integers(0, 65536, (H, W))).astype(np.uint16)
    if (H, W) == (448, 1216):
        yield "kitti64", P.kitti_png_samples(1)
        yield "kitti16", P.kitti_png_samples(2, beams=16)
    if (H, W) == (352, 1216):
        yield "filled64", _filled(3, 64)
        yield "filled16", _filled(4, 16)


ALL = [(f"{H}x{W}-{name}", x) for H, W in SHAPES for name, x in _cases(H, W)]


def _idat(png):
    return b"".join(p for t, p in P.chunks(png) if t == b"IDAT")


@pytest.mark.parametrize("name,x", ALL, ids=[n for n, _ in ALL])
def test_round_trip_through_every_reader(lib, name, x):
    from PIL import Image
    import cv2
    f = _lib.png_encode_host(x)
    assert np.array_equal(P.decode(f), x)
    im = Image.open(io.BytesIO(f))
    assert im.size == (x.shape[1], x.shape[0])
    assert np.array_equal(np.array(im).astype(np.uint16), x)
    assert np.array_equal(cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_UNCHANGED), x)
    st, got = _lib.png_decode_host(f, *x.shape)
    assert st == 0 and np.array_equal(got, x)


@pytest.mark.parametrize("name,x", ALL, ids=[n for n, _ in ALL])
def test_filter_bytes_checksums_and_bound(lib, name, x):
    H, W = x.shape
    f = _lib.png_encode_host(x)
    assert len(f) <= _lib.png_encode_bound(H, W)
    raw = zlib.decompress(_idat(f))
    assert raw == P.filter_rows(x, "msad")
    assert struct.unpack(">I", _idat(f)[-4:])[0] == zlib.adler32(raw)
    pos, types = 8, []
    while pos < len(f):
        n, t = struct.unpack(">I4s", f[pos:pos + 8])
        assert struct.unpack(">I", f[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(f[pos + 4:pos + 8 + n]), (t, pos)
        types.append(t)
        pos += 12 + n
    assert pos == len(f)
    nseg = (H + 15) // 16
    assert types == [b"IHDR"] + [b"IDAT"] * (nseg + 2) + [b"IEND"]
    cs = P.chunks(f)
    assert cs[1][1] == b"\x78\x01" and len(cs[-2][1]) == 4


def test_noise_takes_the_stored_fallback_within_the_bound(lib):
    x = np.random.default_rng(5).integers(0, 65536, (448, 1216)).astype(np.uint16)
    f = _lib.png_encode_host(x)
    assert len(f) == _lib.png_encode_bound(448, 1216)          # every segment stored
    segs = [p for t, p in P.chunks(f) if t == b"IDAT"][1:-1]
    for s in segs:
        assert s[0] & 6 == 0                                   # BTYPE 00
    assert np.array_equal(P.decode(f), x)


def test_segments_end_byte_aligned_with_an_empty_stored_block(lib):
    x = P.kitti_png_samples(6)
    segs = [p for t, p in P.chunks(_lib.png_encode_host(x)) if t == b"IDAT"][1:-1]
    for i, s in enumerate(segs):
        assert s[-4:] == b"\x00\x00\xff\xff", i
        assert s[0] & 7 == 2                                   # BFINAL 0, BTYPE 01
    # each segment alone is a sync-flushed stream: it inflates to its 16 rows
    d = zlib.decompressobj(-15)
    assert len(d.decompress(segs[0])) == 16 * 2433


def test_size_within_bound_for_small_shapes(lib):
    for H in range(1, 40):
        for W in (1, 2, 3, 7, 64):
            x = np.random.default_rng(H * 100 + W).integers(0, 65536, (H, W)).astype(np.uint16)
            f = _lib.png_encode_host(x)
            assert len(f) <= _lib.png_encode_bound(H, W)
            assert np.array_equal(P.decode(f), x)


@pytest.mark.parametrize("beams", [64, 16])
def test_compression_close_to_zlib_level1(lib, beams):
    ours, z1 = 0, 0
    for seed in range(8):
        x = _filled(seed, beams)
        ours += len(_lib.png_encode_host(x))
        z1 += len(zlib.compress(P.filter_rows(x, "msad"), 1))
    assert ours <= 1.25 * z1, ours / z1


def test_bound_and_arguments(lib):
    assert _lib.png_encode_bound(1, 1) == 8 + 25 + 14 + 12 + 3 + 5 + 5 + 16 + 12
    assert lib.dtfill_png_encode_bound(0, 5) < 0 and lib.dtfill_png_encode_bound(1 << 14, 1 << 14) < 0
    x = np.zeros((4, 4), np.uint16)
    out = np.empty(_lib.png_encode_bound(4, 4) - 1, np.uint8)
    assert lib.dtfill_debug_png_encode_host(_lib._ptr(x), 4, 4, _lib._ptr(out), out.size) == -1
    with pytest.raises(TypeError):
        _lib.png_encode_host(x.astype(np.int32))


def _rule(d):
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.nan_to_num(np.float32(256) * d.astype(np.float32), nan=0, posinf=65535, neginf=0)
        return np.trunc(np.clip(v, 0, 65535)).astype(np.uint16)


def test_depth_rule_matches_numpy(lib):
    tiny = np.float32(1e-45)
    special = np.array([np.nan, 0.0, -0.0, -1.0, -1e-30, -np.inf, np.inf, tiny, -tiny, np.float32(1e-39), 255.99609375,
                        np.nextafter(np.float32(255.99609375), np.float32(300)), 256.0, 1e30, 1e-3, 0.00390625,
                        0.0039062, 80.0, 85.123], np.float32)
    ks = np.arange(65536, dtype=np.float32) / np.float32(256)
    d = np.concatenate([special, ks, ks + np.float32(0.001)])
    got = _lib.depth_samples_host(d)
    assert np.array_equal(got, _rule(d))
    assert np.array_equal(_lib.depth_samples_host(ks), np.arange(65536, dtype=np.uint16))       # identity on k/256
    inside = (d >= 0) & (d <= 65535 / 256)
    assert np.array_equal(got[inside], (d[inside] * 256).astype(np.uint16))
    assert got[10] == 65535 and got[11] == 65535                        # 255.99609375 and the float above it


def test_write_depth_pngs_checks_on_the_host():
    with pytest.raises(TypeError):
        data_read.write_depth_pngs(np.zeros((1, 4, 4), np.float64))
    with pytest.raises(TypeError):
        data_read.write_depth_pngs(np.zeros((1, 4, 4), np.int32))
    with pytest.raises(ValueError):
        data_read.write_depth_pngs(np.zeros((4, 4), np.uint16))
    with pytest.raises(ValueError):
        data_read.write_depth_pngs(np.zeros((1, 4, 4, 2), np.float32))
    with pytest.raises(ValueError):
        data_read.write_depth_pngs(np.zeros((2, 4, 4), np.uint16), paths=["a.png"])
