"""The metrics in numpy's summation order (kernels k4x_*, dtfill_metrics / dtfill_metrics_ex) at the edges that random
depths in [0.5, 80] never reach, compared with evaluation.py restated in numpy (oracle.result_kitti / result_nyu) with
assert_array_equal, which holds NaN equal to NaN: outputs and ground truth one float step either side of the validity
threshold 0.01, NYU ratios exactly at the delta bounds 1.25, 1.5625 and 1.953125 and one step either side, infinite,
NaN and overflowing values, the valid counts at which numpy's pairwise sum changes shape, a float64 batch large enough
to be split into two scratch groups, and running totals accumulated on the device."""
import warnings

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib
from oracle import oracle as O

pytestmark = pytest.mark.gpu

f32 = np.float32
MODES = ((_lib.METRICS_KITTI, O.result_kitti), (_lib.METRICS_NYU, O.result_nyu))


@pytest.fixture(scope="module")
def handle(dtfill_lib):
    return _lib.get_handle()


def oracle_rows(ref, out, gt):
    rows = []
    for o, t in zip(out, gt):
        with warnings.catch_warnings():                     # overflow, inf - inf and the mean of an empty array
            warnings.simplefilter("ignore", RuntimeWarning)
            m = ref(o.ravel(), t.ravel())
        rows.append([m["mse"], m["rmse"], m["mae"], m["irmse"], m["imae"], m.get("delta1", 0.0), m.get("delta2", 0.0),
                     m.get("delta3", 0.0), m["count"]])
    return np.array(rows, np.float64)


def column_sums(rows):
    """The batch totals in the order the library adds them: frame after frame from 0, then the frame count."""
    s = np.zeros(9, np.float64)
    for r in rows:
        s = s + r
    return np.append(s, float(len(rows)))


def check(handle, out, gt, what):
    """Every frame's row and the totals, in both modes, against the oracle."""
    out = np.ascontiguousarray(out, np.float32)
    gt = np.ascontiguousarray(gt)
    B = out.shape[0]
    n = out[0].size
    rows = {}
    for mode, ref in MODES:
        per_frame, sums = handle.metrics(out, gt, B, 1, n, mode, gt.dtype == np.float64)
        want = oracle_rows(ref, out, gt)
        np.testing.assert_array_equal(per_frame, want, err_msg=f"{what}, {gt.dtype} ground truth, mode {mode}")
        np.testing.assert_array_equal(sums, column_sums(want), err_msg=f"{what} totals, {gt.dtype}, mode {mode}")
        rows[mode] = want
    return rows


def base_frames(rng, B, n, gt_dtype):
    """B frames of n valid pixels away from every edge, non-grid values."""
    out = rng.uniform(0.5, 80.0, (B, n)).astype(f32)
    gt = rng.uniform(0.5, 80.0, (B, n)).astype(gt_dtype)
    return out, gt


def planted(rng, pairs, gt_dtype, n=300):
    """One frame per (output, ground truth) pair, the pair at a different position in each."""
    out, gt = base_frames(rng, len(pairs), n, gt_dtype)
    for b, (o, t) in enumerate(pairs):
        k = (37 * b + 5) % n
        out[b, k] = f32(o)
        gt[b, k] = gt_dtype(t)
    return out, gt


def steps(v, dtype):
    """v rounded to dtype and its two neighbours."""
    v = dtype(v)
    return [np.nextafter(v, dtype(0)), v, np.nextafter(v, dtype(1e9))]


@pytest.mark.parametrize("gt_dtype", [np.float32, np.float64])
def test_validity_threshold(handle, gt_dtype):
    """`output > 0.01` is a float32 comparison, `target > 0.01` one in the ground truth's dtype: 0.01 rounded to float32
    is not valid, the next float32 up is, and a float64 ground truth of 0.01 rounded to float32 is not."""
    rng = np.random.default_rng(1)
    os_, ts = steps(0.01, f32), steps(0.01, gt_dtype)
    if gt_dtype == np.float64:
        ts += [np.float64(f32(0.01)), np.float64(np.nextafter(f32(0.01), f32(1)))]
    pairs = [(o, 5.0) for o in os_] + [(5.0, t) for t in ts] + [(o, t) for o in os_ for t in ts]
    out, gt = planted(rng, pairs, gt_dtype)
    rows = check(handle, out, gt, "validity threshold")
    counts = rows[_lib.METRICS_KITTI][:, 8]
    assert counts[:3].tolist() == [299, 299, 300]
    assert counts[3:6].tolist() == [299, 299, 300]


@pytest.mark.parametrize("gt_dtype", [np.float32, np.float64])
def test_nyu_delta_bounds(handle, gt_dtype):
    """max(o / t, t / o) < 1.25, 1.5625, 1.953125 (evaluation.py:218-220) with the ratio exactly on each bound, in both
    directions, and one step of the output or of the ground truth either side."""
    rng = np.random.default_rng(2)
    pairs = []
    for r in (1.25, 1.5625, 1.953125):
        for o in steps(4.0 * r, f32):
            pairs.append((o, 4.0))
        for t in steps(4.0, gt_dtype):
            pairs.append((4.0 * r, t))
        for t in steps(4.0 * r, gt_dtype):
            pairs.append((4.0, t))
        for o in steps(4.0, f32):
            pairs.append((o, 4.0 * r))
    out, gt = planted(rng, pairs, gt_dtype, n=200)
    # the planted pair is the frame's only pixel near a bound: a ratio below 1.1 everywhere else
    for b in range(len(pairs)):
        k = (37 * b + 5) % 200
        keep = out[b, k], gt[b, k]
        gt[b] = (out[b] * rng.uniform(0.95, 1.05, 200)).astype(gt_dtype)
        out[b, k], gt[b, k] = keep
    rows = check(handle, out, gt, "delta bounds")[_lib.METRICS_NYU]
    hits = np.rint(rows[:, 5:8] * 200).astype(int)
    assert len(set(map(tuple, hits))) >= 3                     # the bounds split the pairs


@pytest.mark.parametrize("gt_dtype", [np.float32, np.float64])
def test_special_values(handle, gt_dtype):
    """+inf, NaN and 3e38 outputs (1e3 * 3e38 overflows float32; 1 / 3e38 is a float32 denormal), NaN, -inf and +inf
    ground truth, -0.0, and both sides infinite (inf - inf is NaN): one frame each, with frames of no valid pixel."""
    rng = np.random.default_rng(3)
    big = float(f32(3e38))
    pairs = [(np.inf, 5.0), (np.nan, 5.0), (big, 5.0), (-np.inf, 5.0), (-0.0, 5.0), (5.0, np.nan), (5.0, -np.inf),
             (5.0, np.inf), (np.inf, np.inf), (big, big), (5.0, -0.0), (np.nan, np.nan), (big, 1e-2 * 1.5)]
    out, gt = planted(rng, pairs, gt_dtype)
    out[-1] = f32(big)
    check(handle, out, gt, "special values")
    empty_out = np.zeros((2, 50), f32)
    empty_out[1] = np.nan
    check(handle, empty_out, rng.uniform(1, 2, (2, 50)).astype(gt_dtype), "no valid pixel")


@pytest.mark.parametrize("gt_dtype", [np.float32, np.float64])
def test_valid_counts_at_leaf_sizes(handle, gt_dtype):
    """numpy's pairwise sum adds fewer than 8 elements one by one, up to 128 in eight running sums and splits longer
    arrays at a multiple of 8: frames with 0 (NaN rows and NaN totals), 1, 7, 8, 9, 127, 128, 129, 130 and more valid
    pixels, scattered among pixels that fail either test."""
    rng = np.random.default_rng(4)
    counts = (0, 1, 7, 8, 9, 127, 128, 129, 130, 136, 255, 256, 257, 1031)
    n = 2000
    out, gt = base_frames(rng, len(counts), n, gt_dtype)
    for b, c in enumerate(counts):
        bad = rng.permutation(n)[:n - c]
        half = len(bad) // 2
        out[b, bad[:half]] = rng.uniform(0, 0.01, half).astype(f32) * (rng.random(half) < 0.5)
        gt[b, bad[half:]] = 0
    rows = check(handle, out, gt, "leaf sizes")
    assert rows[_lib.METRICS_KITTI][:, 8].tolist() == list(counts)
    assert np.isnan(rows[_lib.METRICS_NYU][0, :8]).all()


def test_float64_batch_in_two_scratch_groups(handle):
    """320 KITTI frames with a float64 ground truth as device pointers: the per-pixel terms of 313 frames fill the ~4 GiB
    scratch, so the batch runs as two groups (313 + 7) and every row, the last of the first group and the first of the
    second included, must still be the oracle's."""
    import torch
    B, H, W = 320, 352, 1216
    g = torch.Generator(device="cuda").manual_seed(6)
    pred = torch.rand((B, H, W), generator=g, device="cuda", dtype=torch.float32) * 80
    gt = torch.rand((B, H, W), generator=g, device="cuda", dtype=torch.float64) * 80
    gt *= torch.rand((B, H, W), generator=g, device="cuda") < 0.2
    per_frame = torch.empty((B, _lib.METRIC_COLS), dtype=torch.float64, device="cuda")
    sums = torch.empty((_lib.METRIC_COLS + 1,), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    handle.metrics(pred.data_ptr(), gt.data_ptr(), B, H, W, _lib.METRICS_KITTI, True, on_device=True,
                   per_frame_ptr=per_frame.data_ptr(), sums_ptr=sums.data_ptr())
    handle.synchronize()
    got, got_sums = per_frame.cpu().numpy(), sums.cpu().numpy()
    p, t = pred.cpu().numpy(), gt.cpu().numpy()
    del pred, gt
    want = oracle_rows(O.result_kitti, p, t)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got_sums, column_sums(want))


@pytest.mark.parametrize("exact", [True, False])
def test_accumulated_totals(handle, exact):
    """metrics(accumulate=True) over two batches into one device vector: the first batch's totals plus the second's, in
    both modes and for both ground-truth dtypes, in numpy's order and in the one-pass order."""
    import torch
    rng = np.random.default_rng(7)
    handle.set_metrics_exact(exact)
    try:
        for gt_dtype in (np.float32, np.float64):
            o1, t1 = base_frames(rng, 5, 40 * 50, gt_dtype)
            o2, t2 = base_frames(rng, 7, 40 * 50, gt_dtype)
            t2[:, ::3] = 0
            for mode, _ in MODES:
                f64 = gt_dtype == np.float64
                _, s1 = handle.metrics(o1, t1, 5, 40, 50, mode, f64)
                _, s2 = handle.metrics(o2, t2, 7, 40, 50, mode, f64)
                tot = torch.zeros(_lib.METRIC_COLS + 1, dtype=torch.float64, device="cuda")
                dev = [torch.from_numpy(a).cuda() for a in (o1, t1, o2, t2)]
                torch.cuda.synchronize()
                handle.metrics(dev[0].data_ptr(), dev[1].data_ptr(), 5, 40, 50, mode, f64, sums_ptr=tot.data_ptr(),
                               accumulate=True)
                handle.metrics(dev[2].data_ptr(), dev[3].data_ptr(), 7, 40, 50, mode, f64, sums_ptr=tot.data_ptr(),
                               accumulate=True)
                handle.synchronize()
                np.testing.assert_array_equal(tot.cpu().numpy(), s1 + s2, err_msg=f"{gt_dtype} mode {mode}")
    finally:
        handle.set_metrics_exact(True)
