"""The PNG decoder (csrc/dtfill_k8_png.cuh) run serially on the CPU through dtfill_debug_png_decode_host: the bit
reader, Huffman tables and token decoder are the code the device runs.  Exact samples on every kind of file the decoder
accepts, and the exact status code on every kind it must reject.  No GPU needed."""
import io
import os
import struct
import zlib

import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib


@pytest.fixture(scope="module")
def lib(dtfill_lib):
    return _lib.load()


def _decode(png, H, W):
    return _lib.png_decode_host(png, H, W)


def _frames():
    rng = np.random.default_rng(7)
    yield "kitti64", P.kitti_png_samples(3)
    yield "kitti16", P.kitti_png_samples(4, beams=16)
    yield "noise", rng.integers(0, 65536, (448, 1216)).astype(np.uint16)
    yield "zeros", np.zeros((448, 1216), np.uint16)
    yield "extremes", rng.choice(np.array([0, 65535], np.uint16), (448, 1216))


@pytest.mark.parametrize("name,x", list(_frames()), ids=lambda v: v if isinstance(v, str) else "")
@pytest.mark.parametrize("filters", [0, 1, 2, 3, 4, "random", "msad"])
def test_filters_kitti_sized(lib, name, x, filters):
    st, got = _decode(P.encode(x, filters=filters, seed=hash(name) & 0xffff), *x.shape)
    assert st == 0 and np.array_equal(got, x)


@pytest.mark.parametrize("level", range(10))
@pytest.mark.parametrize("strategy", sorted(P.STRATEGIES))
def test_levels_and_strategies(lib, level, strategy):
    rng = np.random.default_rng(level * 7 + len(strategy))
    x = P.kitti_png_samples(level, beams=16)[90:150]
    x[:4] = rng.integers(0, 65536, (4, 1216))            # a few dense rows: literals, long codes
    st, got = _decode(P.encode(x, filters="random", level=level, strategy=strategy, seed=level), *x.shape)
    assert st == 0 and np.array_equal(got, x)


@pytest.mark.parametrize("H", [1, 3, 448])
@pytest.mark.parametrize("W", [1, 2, 37, 1216])
def test_shapes(lib, H, W):
    rng = np.random.default_rng(H * 10000 + W)
    x = ((rng.random((H, W)) < 0.1) * rng.integers(0, 65536, (H, W))).astype(np.uint16)
    x.flat[0] = 65535
    for filters in ("random", 4):
        st, got = _decode(P.encode(x, filters=filters, seed=W), H, W)
        assert st == 0 and np.array_equal(got, x)


@pytest.mark.parametrize("idat", [1, 7, "random"])
@pytest.mark.parametrize("ancillary", [False, True])
def test_idat_splits_and_ancillary_chunks(lib, idat, ancillary):
    x = P.kitti_png_samples(11)[:160] if idat == 1 else P.kitti_png_samples(11)
    png = P.encode(x, filters="random", idat=idat, ancillary=ancillary, seed=3)
    st, got = _decode(png, *x.shape)
    assert st == 0 and np.array_equal(got, x)


def test_empty_idat_chunks(lib):
    x = P.kitti_png_samples(12)
    z = P.compress(P.filter_rows(x, "msad"))
    png = P.assemble(448, 1216, [b"", z[:100], b"", b"", z[100:], b""], ancillary=True)
    st, got = _decode(png, 448, 1216)
    assert st == 0 and np.array_equal(got, x)


def test_oracle_agrees_with_pil_and_cv2():
    x = P.kitti_png_samples(5)[80:200]
    for png in (P.encode(x, filters="random"), P.encode(x, level=9, strategy="fixed", idat="random")):
        assert np.array_equal(P.decode(png), x)
        try:
            from PIL import Image
        except ImportError:
            Image = None
        if Image is not None:
            im = Image.open(io.BytesIO(png))
            assert np.array_equal(np.array(im).astype(np.uint16), x)
            buf = io.BytesIO()
            Image.fromarray(x).save(buf, format="PNG")                      # libpng's writer through PIL
            assert np.array_equal(P.decode(buf.getvalue()), x)
        try:
            import cv2
        except ImportError:
            cv2 = None
        if cv2 is not None:
            assert np.array_equal(cv2.imdecode(np.frombuffer(png, np.uint8), cv2.IMREAD_UNCHANGED), x)
            ok, enc = cv2.imencode(".png", x)
            assert ok and np.array_equal(P.decode(enc.tobytes()), x)


def test_golden_libpng_files(lib, golden_dir):
    """Files written by libpng (through PIL and cv2, several settings), committed with the samples they hold."""
    z = np.load(os.path.join(golden_dir, "png_frames.npz"))
    names = sorted(k[:-4] for k in z.files if k.endswith("/png"))
    assert len(names) >= 6
    for n in names:
        x = z[n + "/samples"]
        st, got = _decode(z[n + "/png"].tobytes(), *x.shape)
        assert st == 0 and np.array_equal(got, x), n


# ---- malformed files: the exact status, never a crash ---------------------------------------------------------------
SMALL = np.arange(5 * 6, dtype=np.uint16).reshape(5, 6) * 2000


def _small(**kw):
    return P.encode(SMALL, **kw)


def test_every_prefix(lib):
    png = _small(filters="random")
    for n in range(len(png)):
        st, got = _decode(png[:n], 5, 6)
        assert st == (1 if n < 8 else 4), n
        assert not got.any()
    assert _decode(png, 5, 6)[0] == 0


def _with_zlib(z, H=5, W=6):
    return P.assemble(H, W, [z])


def test_adler_flip(lib):
    z = bytearray(P.compress(P.filter_rows(SMALL, "random")))
    for i in (-1, -4):
        zz = bytearray(z)
        zz[i] ^= 0x10
        assert _decode(_with_zlib(bytes(zz)), 5, 6)[0] == 9


def test_truncated_zlib_stream(lib):
    z = P.compress(P.filter_rows(SMALL, "random"))
    for cut in (1, 3, 10, len(z) - 6):
        assert _decode(_with_zlib(z[:cut]), 5, 6)[0] == (5 if cut < 2 else 6), cut


def test_zlib_header(lib):
    raw = P.filter_rows(SMALL, 0)
    z = P.compress(raw)
    assert _decode(_with_zlib(b"\x79" + z[1:]), 5, 6)[0] == 5            # CM 9
    assert _decode(_with_zlib(z[:1] + bytes([z[1] ^ 1]) + z[2:]), 5, 6)[0] == 5    # FCHECK
    flg = 0x20 | 0x1e                                                       # FDICT set, FCHECK fixed up
    flg += (31 - ((0x78 << 8) | flg) % 31) % 31
    assert _decode(_with_zlib(b"\x78" + bytes([flg]) + z[2:]), 5, 6)[0] == 5


def _stored(raw, final=True, nlen_xor=0):
    n = len(raw)
    return bytes([1 if final else 0]) + struct.pack("<HH", n, (~n & 0xffff) ^ nlen_xor) + raw


def _zwrap(deflate, raw):
    return b"\x78\x01" + deflate + struct.pack(">I", zlib.adler32(raw) & 0xffffffff)


def test_stored_blocks_and_bad_nlen(lib):
    raw = P.filter_rows(SMALL, "random")
    ok = _zwrap(_stored(raw[:20], final=False) + _stored(b"", final=False) + _stored(raw[20:]), raw)
    st, got = _decode(_with_zlib(ok), 5, 6)
    assert st == 0 and np.array_equal(got, SMALL)
    assert _decode(_with_zlib(_zwrap(_stored(raw, nlen_xor=1), raw)), 5, 6)[0] == 6


class _BitWriter:
    def __init__(self):
        self.bits, self.n = 0, 0

    def put(self, v, n):
        self.bits |= v << self.n
        self.n += n

    def huff(self, code, n):                  # Huffman codes go MSB first
        self.put(int(format(code, f"0{n}b")[::-1], 2), n)

    def bytes(self):
        return self.bits.to_bytes((self.n + 7) // 8, "little")


def _fixed_lit(w, v):
    if v < 144:
        w.huff(0x30 + v, 8)
    else:
        w.huff(0x190 + v - 144, 9)


def test_distance_before_start(lib):
    raw = P.filter_rows(SMALL, 0)
    w = _BitWriter()
    w.put(1, 1); w.put(1, 2)                   # final, fixed Huffman
    _fixed_lit(w, raw[0])
    w.huff(0b0000001, 7)                       # length 3 (symbol 257)
    w.huff(1, 5)                               # distance 2 > 1 byte of output
    w.huff(0, 7)                               # end of block
    assert _decode(_with_zlib(_zwrap(w.bytes(), raw)), 5, 6)[0] == 6


def test_fixed_symbols_286_and_distance_30(lib):
    raw = P.filter_rows(SMALL, 0)
    for sym_code, dist in ((0xc0 + 286 - 280, None), (0b0000001, 30)):
        w = _BitWriter()
        w.put(1, 1); w.put(1, 2)
        _fixed_lit(w, raw[0]); _fixed_lit(w, raw[1])
        w.huff(sym_code, 8 if dist is None else 7)
        if dist is not None:
            w.huff(dist, 5)
        w.huff(0, 7)
        assert _decode(_with_zlib(_zwrap(w.bytes(), raw)), 5, 6)[0] == 6


def test_oversubscribed_code_length_set(lib):
    raw = P.filter_rows(SMALL, 0)
    w = _BitWriter()
    w.put(1, 1); w.put(2, 2)                   # final, dynamic
    w.put(0, 5); w.put(0, 5); w.put(15, 4)     # 257 lit/len, 1 dist, 19 code-length codes
    for _ in range(19):
        w.put(1, 3)                            # nineteen codes of length 1
    assert _decode(_with_zlib(_zwrap(w.bytes() + b"\0" * 8, raw)), 5, 6)[0] == 6


def test_incomplete_code_length_set(lib):
    raw = P.filter_rows(SMALL, 0)
    w = _BitWriter()
    w.put(1, 1); w.put(2, 2)
    w.put(0, 5); w.put(0, 5); w.put(0, 4)      # 4 code-length codes: lengths 2, 2, 2, 0 (incomplete)
    for v in (2, 2, 2, 0):
        w.put(v, 3)
    assert _decode(_with_zlib(_zwrap(w.bytes() + b"\0" * 8, raw)), 5, 6)[0] == 6


def test_output_too_long_and_too_short(lib):
    raw = P.filter_rows(SMALL, 0)
    assert _decode(_with_zlib(P.compress(raw + b"\0")), 5, 6)[0] == 7
    assert _decode(_with_zlib(P.compress(raw[:-1])), 5, 6)[0] == 7
    assert _decode(_with_zlib(_zwrap(_stored(raw + b"\0\0"), raw)), 5, 6)[0] == 7


def test_filter_type_5(lib):
    raw = bytearray(P.filter_rows(SMALL, 2))
    raw[3 * 13] = 5
    assert _decode(_with_zlib(P.compress(bytes(raw))), 5, 6)[0] == 8


@pytest.mark.parametrize("depth,colour,interlace", [(8, 0, 0), (16, 2, 0), (16, 0, 1), (16, 4, 0), (16, 3, 0)])
def test_unsupported_ihdr(lib, depth, colour, interlace):
    z = P.compress(P.filter_rows(SMALL, 0))
    png = P.assemble(5, 6, [z], header=P.ihdr(5, 6, depth, colour, interlace))
    assert _decode(png, 5, 6)[0] == 2


def test_size_mismatch_and_broken_chunks(lib):
    png = _small()
    assert _decode(png, 5, 7)[0] == 3
    assert _decode(png, 4, 6)[0] == 3
    assert _decode(b"\x89PNG\r\n\x1a\x0b" + png[8:], 5, 6)[0] == 1
    no_idat = P.assemble(5, 6, [])
    assert _decode(no_idat, 5, 6)[0] == 4
    bad_len = bytearray(png)
    bad_len[33:37] = struct.pack(">I", 0x7fffffff)
    assert _decode(bytes(bad_len), 5, 6)[0] == 4
    crit = png[:33] + P.chunk(b"XXXX", b"abc") + png[33:]                     # unknown critical chunk
    assert _decode(crit, 5, 6)[0] == 4
    bad_crc = bytearray(png)
    bad_crc[29] ^= 0xff                                                       # CRCs are not checked (IHDR's)
    assert _decode(bytes(bad_crc), 5, 6)[0] == 0
