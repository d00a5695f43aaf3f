"""GPU tests of the PNG decoder (k8_png_inflate, k8_png_unfilter) and of the entry points built on it: dtfill_png_decode
against the host hook and the oracle in mixed batches, per-frame status of malformed files inside valid batches,
DT_complete_batch_png_files against DT_complete_batch_png, and DTFillEngine.decode_png + fill_png.
Run on the B200 box:  python -m pytest tests -m gpu"""
import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib, data_read, tools

pytestmark = pytest.mark.gpu

STRATS = sorted(P.STRATEGIES)


@pytest.fixture(scope="module")
def handle(dtfill_lib):
    return _lib.get_handle()


def _pack(files):
    offsets = np.zeros(len(files) + 1, np.int64)
    np.cumsum([len(f) for f in files], out=offsets[1:])
    return np.frombuffer(b"".join(files), np.uint8), offsets


def _kinds(i, x):
    """The i-th kind of encoding of the test matrix."""
    filters = [0, 1, 2, 3, 4, "random", "msad"][i % 7]
    level = i % 10
    strategy = STRATS[(i // 10) % len(STRATS)]
    idat = ["one", 1 if x.size < 40000 else 4096, "random", 7][(i // 3) % 4]
    return P.encode(x, filters=filters, level=level, strategy=strategy, idat=idat, ancillary=i % 5 == 0, seed=i)


def _frame(i, H, W):
    rng = np.random.default_rng(i)
    k = i % 4
    if H == 448 and W == 1216 and k < 2:
        return P.kitti_png_samples(i, beams=64 if k == 0 else 16)
    if k == 2:
        return rng.integers(0, 65536, (H, W)).astype(np.uint16)
    if k == 3:
        return np.zeros((H, W), np.uint16) if i % 8 == 3 else rng.choice(np.array([0, 65535], np.uint16), (H, W))
    return ((rng.random((H, W)) < 0.1) * rng.integers(0, 65536, (H, W))).astype(np.uint16)


@pytest.mark.parametrize("H,W", [(1, 1), (3, 2), (448, 37), (3, 1216), (448, 1216)])
def test_mixed_batches_equal_host_hook_and_oracle(handle, H, W):
    B = 96 if H * W > 100000 else 64
    xs = [_frame(i, H, W) for i in range(B)]
    files = [_kinds(i, x) for i, x in enumerate(xs)]
    data, offsets = _pack(files)
    got, status = handle.png_decode(data, offsets, H, W)
    assert not status.any()
    for i in range(B):
        assert np.array_equal(got[i], xs[i]), i
        if i % 8 == 0:
            st, hh = _lib.png_decode_host(files[i], H, W)
            assert st == 0 and np.array_equal(hh, got[i])


def test_1024_kitti_frames(handle):
    """A batch of the benchmarked size: every frame against the host hook."""
    base = [P.kitti_png_samples(s, beams=64 if s % 2 else 16) for s in range(16)]
    files = [P.encode(base[i % 16], filters="msad" if i % 3 else "random", level=6 if i % 2 else 1, seed=i)
             for i in range(1024)]
    data, offsets = _pack(files)
    got, status = handle.png_decode(data, offsets, 448, 1216)
    assert not status.any()
    for i in range(1024):
        assert np.array_equal(got[i], base[i % 16]), i


def _malformed():
    x = _frame(1, 448, 1216)
    good = P.encode(x, filters="random")
    raw = P.filter_rows(x, "random")
    z = P.compress(raw)
    adler = bytearray(z)
    adler[-1] ^= 1
    bad_filter = bytearray(raw)
    bad_filter[7 * 2433] = 5
    return [
        (good[:5], 1),
        (P.assemble(448, 1216, [z], header=P.ihdr(448, 1216, 8)), 2),
        (P.encode(x[:, :1000]), 3),
        (good[:len(good) // 2], 4),
        (P.assemble(448, 1216, [b"\x79" + z[1:]]), 5),
        (P.assemble(448, 1216, [z[:len(z) // 2]]), 6),
        (P.assemble(448, 1216, [P.compress(raw[:-3])]), 7),
        (P.assemble(448, 1216, [P.compress(bytes(bad_filter))]), 8),
        (P.assemble(448, 1216, [bytes(adler)]), 9),
    ]


def test_malformed_files_inside_a_valid_batch(handle):
    bad = _malformed()
    xs, files, want = [], [], []
    for i in range(40):
        if i % 4 == 1:
            f, st = bad[(i // 4) % len(bad)]
            xs.append(np.zeros((448, 1216), np.uint16))
        else:
            xs.append(_frame(i, 448, 1216))
            f, st = _kinds(i, xs[-1]), 0
        files.append(f)
        want.append(st)
    for f, st in zip(files, want):
        assert _lib.png_decode_host(f, 448, 1216)[0] == st
    data, offsets = _pack(files)
    out = np.empty((40, 448, 1216), np.uint16)
    status = np.empty(40, np.int32)
    bad_frame = __import__("ctypes").c_int(-1)
    L = _lib.load()
    rc = L.dtfill_png_decode(handle._h, _lib._ptr(data), _lib._ptr(offsets), 0, 40, 448, 1216, _lib._ptr(out),
                             _lib._ptr(status), 0, __import__("ctypes").byref(bad_frame))
    assert rc == _lib.E_DATA and bad_frame.value == 1
    assert status.tolist() == want
    for i in range(40):
        assert np.array_equal(out[i], xs[i]), i
    with pytest.raises(ValueError, match="frame 1: bad PNG signature"):
        handle.png_decode(data, offsets, 448, 1216)


def _kitti_files(n, seed=0):
    xs = [P.kitti_png_samples(seed + i, beams=64 if i % 2 == 0 else 16) for i in range(n)]
    return xs, [P.encode(x, filters="msad" if i % 2 else "random", seed=i) for i, x in enumerate(xs)]


def test_dt_complete_batch_png_files_equals_samples_path(handle, tmp_path):
    xs, files = _kitti_files(12)
    paths = []
    for i, f in enumerate(files[:6]):
        p = tmp_path / f"{i:010d}.png"
        p.write_bytes(f)
        paths.append(str(p))
    lidar, refined = tools.DT_complete_batch_png_files(paths + files[6:])
    lidar0, refined0 = tools.DT_complete_batch_png(np.stack(xs))
    assert lidar.shape == lidar0.shape == (12, 352, 1216, 1)
    assert np.array_equal(lidar, lidar0) and np.array_equal(refined, refined0)
    assert np.array_equal(data_read.read_depth_pngs(paths + files[6:]), np.stack(xs))


def test_dt_complete_batch_png_files_errors(handle):
    zero = P.encode(np.zeros((448, 1216), np.uint16))
    xs, files = _kitti_files(2)
    with pytest.raises(IndexError):
        tools.DT_complete_batch_png_files([files[0], zero])
    with pytest.raises(ValueError):
        tools.DT_complete_batch_png_files(files, crop_top=95)
    with pytest.raises(ValueError, match="frame 1"):
        tools.DT_complete_batch_png_files([files[0], files[1][:100], zero])     # a decode failure wins over IndexError


@pytest.mark.parametrize("depth", [1, 4])
def test_engine_decode_then_fill(handle, depth):
    torch = pytest.importorskip("torch")
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    eng = DTFillEngine(pipeline_depth=depth)
    xs, files = _kitti_files(24, seed=100)
    results = []
    for lo, hi in ((0, 8), (8, 24), (0, 3), (3, 24), (10, 12)):      # batch sizes that grow and shrink
        data, offsets = _pack(files[lo:hi])
        d = torch.from_numpy(data.copy()).cuda()
        o = torch.from_numpy(offsets).cuda()
        samples, status = eng.decode_png(d, o, 448, 1216)
        r = eng.fill_png(samples)
        results.append((lo, hi, samples, status, r))
    eng.flush()
    torch.cuda.synchronize()
    for lo, hi, samples, status, r in results:
        assert not status.cpu().numpy().any()
        s = samples.cpu().view(torch.int16).numpy().view(np.uint16)
        assert np.array_equal(s, np.stack(xs[lo:hi]))
        lidar0, refined0 = tools.DT_complete_batch_png(np.stack(xs[lo:hi]))
        assert np.array_equal(r["lidar"].cpu().numpy(), lidar0[..., 0])
        assert np.array_equal(r["depth"].cpu().numpy(), refined0[..., 0])
    eng.close()
