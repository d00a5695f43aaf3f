"""Drop-in for the two helper functions defined inside the reference's solution_DeepNet/eval_NYU.py:114-133, and the
script's evaluation loop on the GPU.

    nearest_point(refined_lidar)   -> (dt, lbl)          eval_NYU.py:114-117  (source threshold 0.001)
    Distance_Transform(lidar)      -> depth_map [H,W]    eval_NYU.py:120-133  (any size, dtype of the input)
    nyu_sample_coords(n)           -> (rows, cols)       data_read.py:360-364 (the random sample of one frame)
    evaluate_fill_sampled(gt, rows, cols) -> (per_frame [B,9], sums [10])   eval_NYU.py:138-254 from dense ground truth
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .tools import VALID_THR, _as_frames_f32, _gather_f64, _is_wide, _labels_f64
from .tools import nearest_point as _nearest_point

NYU_SRC_THR = 0.001     # eval_NYU.py:115
NYU_EVAL_CROP = (6, 234, 8, 312)      # eval_NYU.py:202-207: rows 6:234, columns 8:312 of the 240 x 320 frames are scored


def nearest_point(refined_lidar, device: int | None = None):
    return _nearest_point(refined_lidar, thr=NYU_SRC_THR, device=device)


def Distance_Transform(lidar, src_thr: float = NYU_SRC_THR, device: int | None = None):
    """eval_NYU.py:120-133.  The notebook copies of this function use src_thr=0.1."""
    lidar = np.squeeze(np.asarray(lidar))                                    # :122
    if lidar.ndim != 2:
        raise ValueError(f"not enough values to unpack (expected 2, got {lidar.ndim})"
                         if lidar.ndim < 2 else f"too many values to unpack (expected 2)")   # :123
    if _is_wide(lidar):
        # float64 input: predicates in float64, the result keeps the input's dtype (:126-133)
        _, lbl, val, r = _labels_f64(lidar[None], src_thr, device)
        if "index_error" in r:
            raise IndexError(r["index_error"])                               # :128
        if int(r["counts"][0, 1]) == 1:
            raise IndexError("too many indices for array: array is 0-dimensional, but 1 were indexed")
        return _gather_f64(lidar, val[0], lbl[0])
    x = _as_frames_f32(lidar, "Distance_Transform")
    r = _lib.get_handle(device).run_host(x[None], src_thr, VALID_THR)
    if "index_error" in r:
        raise IndexError(r["index_error"])                                   # :128
    if int(r["counts"][0, 1]) == 1:
        # :126 np.squeeze(lidar[with_value]) makes a single valid depth 0-dimensional; :128 then fails
        raise IndexError("too many indices for array: array is 0-dimensional, but 1 were indexed")
    return r["depth"][0]


def nyu_sample_coords(n: int, H: int = 240, W: int = 320, rng=np.random):
    """The sample of one NYU frame: (rows, cols) int arrays of length n such that ``Mask[rows, cols] = 1`` is the
    reference's mask.  The expression is the one SURVEY.md (section 8, row a-7) quotes from data_read.py:360-364, which is
    not part of this checkout:

        Mask[np.random.randint(H - 12, size=n) + 6, np.random.randint(W - 16, size=n) + 8] = 1

    Python evaluates the index tuple left to right, so the rows are drawn first; under the same seed (``np.random.seed``,
    or a ``np.random.RandomState`` passed as rng) this gives the reference's masks."""
    rows = rng.randint(H - 12, size=n) + 6
    cols = rng.randint(W - 16, size=n) + 8
    return rows, cols


def _index_array(a, what):
    """One frame's rows or cols as numpy's fancy index takes them: an integer array of any length, or a sequence (an
    empty list indexes nothing; an empty float array is refused, as numpy refuses it)."""
    if not isinstance(a, np.ndarray):
        a = np.asarray(a)
        if a.size == 0:
            a = a.astype(np.intp)
    if a.ndim != 1:
        raise ValueError(f"evaluate_fill_sampled: {what} of a frame must be one-dimensional, got shape {a.shape}")
    if a.dtype.kind == "b":
        raise IndexError(f"evaluate_fill_sampled: {what} must be integer arrays, not boolean masks")
    if a.dtype.kind not in "iu":
        raise IndexError("arrays used as indices must be of integer (or boolean) type")
    return a


def _sample_arrays(rows, cols, B: int, H: int, W: int):
    """rows / cols: [B,n] integer arrays or sequences of B per-frame integer arrays -> (rows int32, cols int32, offsets
    int64 [B+1]), negatives wrapped as numpy's fancy index wraps them.  IndexError with numpy's message for the first
    coordinate outside the frame (frames in order, rows before columns)."""
    rows_f = [_index_array(r, "rows") for r in rows]
    cols_f = [_index_array(c, "cols") for c in cols]
    if len(rows_f) != B or len(cols_f) != B:
        raise ValueError(f"evaluate_fill_sampled: {B} frames but {len(rows_f)} rows and {len(cols_f)} cols lists")
    for b, (r, c) in enumerate(zip(rows_f, cols_f)):
        if r.size != c.size:
            raise ValueError(f"evaluate_fill_sampled: frame {b} has {r.size} rows but {c.size} cols")
    counts = np.array([r.size for r in rows_f], np.int64)
    offsets = np.zeros(B + 1, np.int64)
    np.cumsum(counts, out=offsets[1:])
    out = []
    for arrs, size, axis in ((rows_f, H, 0), (cols_f, W, 1)):
        flat = np.concatenate([a.astype(np.int64, copy=False) for a in arrs]) if offsets[-1] else np.zeros(0, np.int64)
        out.append(flat)
    bad = (out[0] < -H) | (out[0] >= H) | (out[1] < -W) | (out[1] >= W)
    if bad.any():
        k = int(np.argmax(bad))
        b = int(np.searchsorted(offsets, k, side="right")) - 1
        lo, hi = offsets[b], offsets[b + 1]
        for flat, size, axis in ((out[0], H, 0), (out[1], W, 1)):
            sel = (flat[lo:hi] < -size) | (flat[lo:hi] >= size)
            if sel.any():
                v = int(flat[lo + int(np.argmax(sel))])
                raise IndexError(f"index {v} is out of bounds for axis {axis} with size {size}")
    r32 = np.where(out[0] < 0, out[0] + H, out[0]).astype(np.int32)
    c32 = np.where(out[1] < 0, out[1] + W, out[1]).astype(np.int32)
    if r32.size == 0:                      # the library takes non-NULL arrays; the offsets say that none is read
        r32, c32 = np.zeros(1, np.int32), np.zeros(1, np.int32)
    return r32, c32, offsets


def _check_crop(crop, H: int, W: int):
    r0, r1, c0, c1 = (int(v) for v in crop)
    if not (0 <= r0 < r1 <= H and 0 <= c0 < c1 <= W):
        raise ValueError(f"evaluate_fill_sampled: crop {tuple(crop)} is not a non-empty window of the {H} x {W} frames")
    return r0, r1, c0, c1


def evaluate_fill_sampled(gt, rows, cols, crop=NYU_EVAL_CROP, src_thr: float = NYU_SRC_THR, device: int | None = None):
    """The evaluation loop of eval_NYU.py:138-254 on B frames of dense ground truth, in one call on the GPU:

        for b in range(B):
            Mask = np.zeros((H, W), np.float32); Mask[rows[b], cols[b]] = 1        data_read.py:360-364
            pred = Distance_Transform(gt[b] * Mask)                                eval_NYU.py:120-133 (src_thr 0.001)
            r0, r1, c0, c1 = crop
            result.evaluate(pred[r0:r1, c0:c1], gt[b][r0:r1, c0:c1])               eval_NYU.py:202-207

    gt: float32 [B,H,W], a numpy array or a CUDA torch tensor (used in place: only the coordinates go up).  rows / cols:
    [B,n] integer arrays, or sequences of B per-frame integer arrays of different lengths (nyu_sample_coords draws one
    frame's); they index like numpy's fancy index (duplicates collapse, negatives in [-H, -1] / [-W, -1] wrap).  Returns
    (per_frame float64 [B,9], sums float64 [10]) in the layout of evaluation.evaluate_batch: row b is Result_NYU.evaluate's
    [mse, rmse, mae (= REL), irmse, imae, delta1, delta2, delta3, n_valid] bit for bit, sums the column sums followed by B.
    The division by the frame count (654 in the reference) stays with the caller: sharding.finalize_means(sums).
    device: the GPU that runs the call for a numpy ground truth; a CUDA tensor runs on its own device (a different
    device raises ValueError).

    Raises TypeError for a ground truth that is not float32, ValueError for an empty batch, rows / cols that do not match
    the batch or each other and a crop that is not a window of the frame, IndexError with numpy's message for a coordinate
    outside the frame -- all before the device is touched -- and IndexError for the first frame Distance_Transform rejects
    (no valid depth, exactly one valid depth, labels outside the list of valid depths)."""
    from .tools import VALID_THR
    is_tensor = type(gt).__module__.startswith("torch")
    if is_tensor:
        import torch
        if gt.dtype != torch.float32:
            raise TypeError(f"evaluate_fill_sampled: ground truth dtype {gt.dtype} not supported (float32 only)")
        if not gt.is_cuda:
            gt = gt.numpy()
            is_tensor = False
    if is_tensor and device is not None and int(device) != gt.device.index:
        raise ValueError(f"evaluate_fill_sampled: device={device} but the ground truth is on {gt.device}")
    if not is_tensor:
        gt = np.asarray(gt)
        if gt.dtype != np.float32:
            raise TypeError(f"evaluate_fill_sampled: ground truth dtype {gt.dtype} not supported (float32 only)")
    if gt.ndim != 3:
        raise ValueError(f"evaluate_fill_sampled: ground truth must be [B,H,W], got shape {tuple(gt.shape)}")
    B, H, W = (int(v) for v in gt.shape)
    if B == 0 or H == 0 or W == 0:
        raise ValueError("evaluate_fill_sampled: empty batch")
    crop = _check_crop(crop, H, W)
    r, c, off = _sample_arrays(rows, cols, B, H, W)
    if is_tensor:
        gt = _aligned(gt)
        torch.cuda.current_stream(gt.device).synchronize()      # the handle's stream reads gt
        h = _lib.get_handle(gt.device.index)
        return h.eval_sampled(gt.data_ptr(), B, H, W, r, c, off, crop, src_thr, VALID_THR, gt_is_device=True)
    return _lib.get_handle(device).eval_sampled(np.ascontiguousarray(gt), B, H, W, r, c, off, crop, src_thr, VALID_THR)


def _aligned(t):
    """A contiguous CUDA tensor whose data starts on a 16-byte boundary (the rows are read with 128-bit loads): t itself
    as a rule, else a copy."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()
