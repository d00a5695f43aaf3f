"""Handle.transfer_bytes (dtfill_transfer_bytes): every synchronous call with an in_is_device / out_is_device flag, and
every eval_* call, starts the link ledger at 0 and counts each copy between host and device it issues, so the values
below follow from the shapes alone -- with host buffers, host in / device out and device in / host out, and right after
a call of another kind.  Run on the B200 box:  python -m pytest tests -m gpu"""
import ctypes

import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib

gpu = pytest.mark.gpu
B, H, W = 3, 64, 96
NPX = B * H * W


def _frames(seed, density=0.1):
    """Sparse float32 depth frames [B,H,W]: values in [1, 60) metres, k / 256 as a PNG sample gives them; each one is
    a source and valid, so the sparse upload keeps exactly the non-zero pixels."""
    rng = np.random.default_rng(seed)
    x = np.zeros((B, H, W), np.float32)
    m = rng.random((B, H, W)) < density
    x[m] = np.round(rng.uniform(1.0, 60.0, int(m.sum())) * 256) / 256
    return x


def _files(frames):
    """Frames -> (packed 16-bit PNG files, offsets [B+1], total file bytes)."""
    files = [P.encode(np.rint(f * 256).astype(np.uint16)) for f in frames]
    off = np.zeros(len(files) + 1, np.int64)
    off[1:] = np.cumsum([len(f) for f in files])
    return np.frombuffer(b"".join(files), np.uint8).copy(), off, int(off[-1])


def _staged(nbytes, nfiles):
    """What one upload of host PNG files sends: the bytes rounded up to 16, then the rebased offsets."""
    return ((nbytes + 15) & ~15) + 8 * (nfiles + 1)


def _p(a):
    return ctypes.c_void_p(a if isinstance(a, int) else a.ctypes.data) if a is not None else None


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture
def h(dtfill_lib):
    h = _lib.Handle(0)
    yield h
    h.close()


@gpu
def test_run_host_with_and_without_counts(h):
    x = _frames(1)
    h.set_sparse_upload(False)
    h.run_host(x, 0.1, 0.1, want_dt=True, want_lbl=True, want_mask=True)
    assert h.transfer_bytes() == (x.nbytes, NPX * 13 + B * 8)          # depth, dt, lbl, mask, counts
    h.run_host(x, 0.1, 0.1, want_counts=False)
    assert h.transfer_bytes() == (x.nbytes, NPX * 4)
    h.set_sparse_upload(True)
    h.run_host(x, 0.1, 0.1)
    assert h.transfer_bytes() == (8 * np.count_nonzero(x), NPX * 4 + B * 8)    # (index, value) pairs up


@gpu
def test_run_with_device_buffers_on_one_side(h, torch):
    x = _frames(2)
    xd = torch.from_numpy(x).cuda()
    depth_d = torch.empty((B, H, W), dtype=torch.float32, device="cuda")
    counts_d = torch.empty((B, 2), dtype=torch.int32, device="cuda")
    depth = np.empty((B, H, W), np.float32)
    counts = np.empty((B, 2), np.int32)
    bad = ctypes.c_int(-1)
    L = h._L
    assert L.dtfill_run(h._h, _p(x), 0, B, H, W, 0.1, 0.1, _p(depth_d.data_ptr()), None, None, None,
                        _p(counts_d.data_ptr()), 1, ctypes.byref(bad)) == 0
    assert h.transfer_bytes() == (x.nbytes, 0)
    assert L.dtfill_run(h._h, _p(xd.data_ptr()), 1, B, H, W, 0.1, 0.1, _p(depth), None, None, None, _p(counts), 0,
                        ctypes.byref(bad)) == 0
    assert h.transfer_bytes() == (0, NPX * 4 + B * 8)
    assert np.array_equal(depth, depth_d.cpu().numpy()) and np.array_equal(counts, counts_d.cpu().numpy())


@gpu
def test_png_decode_host_and_device_files(h, torch):
    data, off, nbytes = _files(_frames(3))
    samples, _ = h.png_decode(data, off, H, W)
    assert h.transfer_bytes() == (_staged(nbytes, B), NPX * 2 + B * 4)
    h.outlier_removal(_frames(4))                     # a call that moves other amounts first
    out = np.empty((B, H, W), np.uint16)
    status = np.empty(B, np.int32)
    bad = ctypes.c_int(-1)
    data_d, off_d = torch.from_numpy(data).cuda(), torch.from_numpy(off).cuda()
    assert h._L.dtfill_png_decode(h._h, _p(data_d.data_ptr()), _p(off_d.data_ptr()), 1, B, H, W, _p(out), _p(status),
                                  0, ctypes.byref(bad)) == 0
    assert h.transfer_bytes() == (0, NPX * 2 + B * 4)
    assert np.array_equal(out, samples)


@gpu
def test_run_host_png_and_png_to_png(h):
    data, off, nbytes = _files(_frames(5))
    h.run_host_png(data, off, H, W, 0, 0.1, 0.1)
    assert h.transfer_bytes() == (_staged(nbytes, B), B * 4 + NPX * 4 + B * 8)     # status, depth, counts
    r = h.run_host_png_to_png(data, off, H, W, 0, 0.1, 0.1)
    out_bytes = sum(len(f) for f in r["files"])
    assert h.transfer_bytes() == (_staged(nbytes, B), B * 4 + 8 * (B + 1) + out_bytes)    # status, offsets, files


@gpu
def test_png_encode(h):
    samples = np.rint(_frames(6) * 256).astype(np.uint16)
    files = h.png_encode(samples)
    assert h.transfer_bytes() == (samples.nbytes, 8 * (B + 1) + sum(len(f) for f in files))


@gpu
def test_metrics_on_either_side(h, torch):
    pred = _frames(7, density=0.9)
    gt = _frames(8, density=0.3).astype(np.float64)
    h.metrics(pred, gt, B, H, W, _lib.METRICS_KITTI, True)
    assert h.transfer_bytes() == (pred.nbytes + gt.nbytes, B * 72 + 80)
    pf_d = torch.empty((B, 9), dtype=torch.float64, device="cuda")
    sums_d = torch.empty(10, dtype=torch.float64, device="cuda")
    pred_d, gt_d = torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda()
    h.metrics(pred, gt, B, H, W, _lib.METRICS_KITTI, True)          # non-zero counts before the device-only call
    h.metrics(pred_d.data_ptr(), gt_d.data_ptr(), B, H, W, _lib.METRICS_KITTI, True, on_device=True,
              per_frame_ptr=pf_d.data_ptr(), sums_ptr=sums_d.data_ptr())
    assert h.transfer_bytes() == (0, 0)
    pf, sums = np.empty((B, 9)), np.empty(10)
    assert h._L.dtfill_metrics(h._h, _p(pred_d.data_ptr()), _p(gt_d.data_ptr()), 1, 1, B, H, W, _lib.METRICS_KITTI,
                               _p(pf), _p(sums), 0) == 0
    assert h.transfer_bytes() == (0, B * 72 + 80)
    assert np.array_equal(pf, pf_d.cpu().numpy()) and np.array_equal(sums, sums_d.cpu().numpy())


@gpu
def test_dt_pool_outlier_and_edt(h):
    x, m = _frames(9), (_frames(10) > 0).astype(np.float32)
    h.dt_pool(x, m, B, H, W, 3, 3, want_masks=True)
    assert h.transfer_bytes() == (2 * NPX * 4, 2 * NPX * 4 + 2 * NPX)          # data and mask up; 2 levels and masks
    h.dt_pool_demo(x, B, H, W, 5, 3)
    assert h.transfer_bytes() == (NPX * 4 + 5 * 5 * 4, 2 * NPX * 4)            # data and the weight table up
    h.outlier_removal(x)
    assert h.transfer_bytes() == (NPX * 4, NPX * 4)
    h.edt(x, 0.1, want_idx=True)
    assert h.transfer_bytes() == (NPX * 4, 2 * NPX * 4)


@gpu
def test_eval_after_another_call_and_async_calls_leave_it(h, torch):
    lidar, lidar_off, nl = _files(_frames(11))
    gt, gt_off, ng = _files(_frames(12, density=0.4))
    h.edt(_frames(13), 0.1)                            # much larger counts than the evaluation's
    h.eval_png(lidar, lidar_off, gt, gt_off, H, W, 0.1, 0.1)
    want = (_staged(nl + ng, 2 * B), B * (4 + 4 + 8 + 72) + 80)      # two statuses, counts, rows, sums
    assert h.transfer_bytes() == want
    xd = torch.from_numpy(_frames(14)).cuda()
    depth_d = torch.empty_like(xd)
    h.run_device_async(xd.data_ptr(), B, H, W, 0.1, 0.1, depth_d.data_ptr())
    h.status()
    assert h.transfer_bytes() == want
