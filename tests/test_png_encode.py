"""GPU tests of the PNG encoder (k9_png_filter, k9_png_deflate, k9_png_offsets, k9_png_pack) and of the entry points
built on it: dtfill_png_encode byte for byte against the host hook in mixed batches, encode -> dtfill_png_decode on the
device, the float32 depth path, DT_complete_batch_png_files_to_png against DT_complete_batch_png_files, the engine, and
the capacity check.  Run on the B200 box:  python -m pytest tests -m gpu"""
import ctypes

import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib, data_read, tools

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle(dtfill_lib):
    return _lib.get_handle()


def _frame(i, H, W):
    rng = np.random.default_rng(i)
    k = i % 6
    if H == 448 and W == 1216 and k < 2:
        x = P.kitti_png_samples(i % 24, beams=64 if k == 0 else 16)
        return np.roll(x, i // 24, axis=1)
    if k == 2:
        return rng.integers(0, 65536, (H, W)).astype(np.uint16)
    if k == 3:
        return np.zeros((H, W), np.uint16) if i % 12 == 3 else np.full((H, W), 65535, np.uint16)
    if k == 4:
        return rng.choice(np.array([0, 65535], np.uint16), (H, W))
    return ((rng.random((H, W)) < 0.1) * rng.integers(0, 65536, (H, W))).astype(np.uint16)


@pytest.mark.parametrize("H,W,B", [(1, 1, 64), (3, 2, 64), (1, 1216, 64), (448, 1, 64), (448, 37, 128),
                                   (352, 1216, 96), (448, 1216, 1024)])
def test_device_bytes_equal_host_hook(handle, H, W, B):
    xs = np.stack([_frame(i, H, W) for i in range(B)])
    files = handle.png_encode(xs)
    assert len(files) == B
    step = 1 if B <= 128 else 7
    for i in range(0, B, step):
        assert files[i] == _lib.png_encode_host(xs[i]), i
    for i in range(0, B, 31):
        assert np.array_equal(P.decode(files[i]), xs[i]), i


def test_device_round_trip_through_the_decoder(handle):
    import torch
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    B, H, W = 256, 448, 1216
    xs = np.stack([_frame(i, H, W) for i in range(B)])
    eng = DTFillEngine()
    t = torch.from_numpy(xs.view(np.int16)).cuda().view(torch.uint16)
    data, offsets = eng.encode_png(t)
    samples, status = eng.decode_png(data, offsets, H, W)
    torch.cuda.synchronize()
    assert not status.cpu().numpy().any()
    assert np.array_equal(samples.cpu().view(torch.int16).numpy().view(np.uint16), xs)
    eng.close()


def test_float_path_equals_samples_of_the_rule(handle):
    rng = np.random.default_rng(3)
    B, H, W = 64, 352, 1216
    d = (rng.random((B, H, W)) * 90).astype(np.float32) * (rng.random((B, H, W)) < 0.5)
    d[0, 0, :8] = [np.nan, np.inf, -np.inf, -1, 255.99609375, 300, 1e-40, 0.00390625]
    d[1] = np.arange(H * W, dtype=np.float32).reshape(H, W) % 65536 / 256
    got = handle.png_encode_depth(d)
    want = handle.png_encode(_lib.depth_samples_host(d))
    assert got == want
    assert data_read.write_depth_pngs(d[..., None]) == want
    assert np.array_equal(P.decode(got[1]), (d[1] * 256).astype(np.uint16))


def test_write_depth_pngs_writes_files(handle, tmp_path):
    xs = np.stack([P.kitti_png_samples(i) for i in range(3)])
    paths = [tmp_path / f"{i:010d}.png" for i in range(3)]
    files = data_read.write_depth_pngs(xs, paths=paths)
    for p, f, x in zip(paths, files, xs):
        assert p.read_bytes() == f
        assert np.array_equal(data_read.read_depth_pngs([str(p)])[0], x)


@pytest.fixture(scope="module")
def kitti_files():
    return [P.encode(P.kitti_png_samples(i % 32, beams=64 if i % 2 == 0 else 16), level=1 + i % 9) for i in range(256)]


def test_files_to_files_equal_files_to_numpy(handle, kitti_files):
    out = tools.DT_complete_batch_png_files_to_png(kitti_files)
    _, ref = tools.DT_complete_batch_png_files(kitti_files)
    want = (ref[..., 0] * 256).astype(np.uint16)
    assert len(out) == len(kitti_files)
    got = data_read.read_depth_pngs(out)
    assert np.array_equal(got, want)
    for i in range(0, 256, 37):
        assert np.array_equal(P.decode(out[i]), want[i])
        assert out[i] == _lib.png_encode_host(want[i])


def test_files_to_files_errors(handle, kitti_files):
    files = list(kitti_files[:8])
    files[5] = files[5][:200]
    with pytest.raises(ValueError, match="frame 5"):
        tools.DT_complete_batch_png_files_to_png(files)
    files = list(kitti_files[:8])
    files[3] = P.encode(np.zeros((448, 1216), np.uint16))
    with pytest.raises(IndexError):
        tools.DT_complete_batch_png_files(files)
    with pytest.raises(IndexError):
        tools.DT_complete_batch_png_files_to_png(files)
    with pytest.raises(ValueError):
        tools.DT_complete_batch_png_files_to_png([P.encode(np.zeros((400, 1216), np.uint16))])
    assert tools.DT_complete_batch_png_files_to_png([]) == []


@pytest.mark.parametrize("depth", [1, 4])
def test_engine_decode_fill_encode(handle, kitti_files, depth):
    import torch
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    files = kitti_files[:64]
    data, offsets, Hin, W = data_read.pack_png_files(files)
    eng = DTFillEngine(pipeline_depth=depth)
    d = torch.from_numpy(np.array(data)).cuda()
    o = torch.from_numpy(offsets).cuda()
    outs = []
    for _ in range(3):
        samples, status = eng.decode_png(d, o, Hin, W)
        r = eng.fill_png(samples, crop_top=96, want_lidar=False)
        outs.append(eng.encode_png(r["depth"]))
    eng.flush()
    torch.cuda.synchronize()
    want = tools.DT_complete_batch_png_files_to_png(files)
    for buf, off in outs:
        off = off.cpu().numpy()
        buf = buf.cpu().numpy()
        assert [buf[off[b]:off[b + 1]].tobytes() for b in range(len(files))] == want
    eng.close()


def test_capacity_below_bound_is_refused_without_writing(handle):
    L = _lib.load()
    B, H, W = 4, 352, 1216
    x = np.stack([P.kitti_png_samples(i)[96:] for i in range(B)])
    cap = B * _lib.png_encode_bound(H, W) - 1
    out = np.full(cap, 0xAB, np.uint8)
    off = np.full(B + 1, -7, np.int64)
    rc = L.dtfill_png_encode(handle._h, _lib._ptr(x), 0, B, H, W, _lib._ptr(out), cap, _lib._ptr(off), 0)
    assert rc == _lib.E_ARG
    assert (out == 0xAB).all() and (off == -7).all()
    bad = ctypes.c_int(0)
    data, offsets, Hin, W2 = data_read.pack_png_files([P.encode(P.kitti_png_samples(i)) for i in range(B)])
    rc = L.dtfill_run_png_to_png(handle._h, _lib._ptr(data), _lib._ptr(offsets), 0, B, Hin, W2, 96, 0.1, 0.1,
                                 _lib._ptr(out), cap, _lib._ptr(off), 0, ctypes.byref(bad))
    assert rc == _lib.E_ARG
    assert (out == 0xAB).all() and (off == -7).all()
