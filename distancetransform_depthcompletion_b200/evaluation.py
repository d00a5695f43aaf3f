"""Drop-in for the reference's evaluation.py result classes, reduced on the GPU (kernels k4_metrics_*).

    Result().evaluate(output, target)       evaluation.py:82-123   KITTI: mm and 1/km
    Result_NYU().evaluate(output, target)   evaluation.py:196-239  NYU: metres, REL, delta1..3

``evaluate`` sets the same attributes as the reference and returns None.  ``evaluate_batch`` is the batched form
the eval loops (eval.py:212-232, eval_NYU.py:207-229) reduce to: per-frame metrics and their running sums.
``evaluate_fill_png_files`` runs the KITTI ablation notebook's loop (PNG files -> Distance_Transform -> Result.evaluate)
from the files, decoding, filling and evaluating on the GPU.
"""
from __future__ import annotations

import numpy as np

from . import _lib


def _prep(output, target):
    output = np.asarray(output)
    target = np.asarray(target)
    if output.shape != target.shape:
        raise IndexError(f"boolean index did not match: output {output.shape} vs target {target.shape}")
    if output.dtype != np.float32:
        raise TypeError(f"evaluate: output dtype {output.dtype} not supported by the CUDA path (float32 only)")
    if target.dtype not in (np.float32, np.float64):
        raise TypeError(f"evaluate: target dtype {target.dtype} not supported (float32 or float64)")
    return np.ascontiguousarray(output), np.ascontiguousarray(target)


def evaluate_batch(output, target, mode: int, device: int | None = None):
    """output float32 / target float32|float64, both [B,...]: returns (per_frame [B,9], sums [10])."""
    output, target = _prep(output, target)
    B = output.shape[0]
    n = int(np.prod(output.shape[1:]))
    return _lib.get_handle(device).metrics(output, target, B, 1, n, mode, target.dtype == np.float64)


def evaluate_fill_png_files(lidar_files, gt_files, src_thr: float = 0.1, device: int | None = None):
    """The evaluation loop of the KITTI ablation notebook (SURVEY.md section 3 C), from the PNG files, in one call:

        for i in range(B):
            lidar = np.array(Image.open(lidar_files[i])).astype(np.float32) / 256    data_read.py:215
            gt = np.array(Image.open(gt_files[i])) / 256.                            data_read.py:223 (float64)
            pred = Distance_Transform(lidar, src_thr)                                 eval_NYU.py:120-133
            result.evaluate(pred, gt)                                                 evaluation.py:82-123

    lidar_files, gt_files: paths or the files' bytes, 16-bit grayscale PNGs all of the size of the first LiDAR file,
    evaluated at that size (no crop).  Returns (per_frame float64 [B,9], sums float64 [10]) in the layout of
    evaluate_batch: row b is [mse, rmse, mae, irmse, imae, 0, 0, 0, n_valid] of frame b, equal to Result.evaluate's bit for
    bit (a frame whose ground truth has no valid pixel gives numpy's mean of an empty array), and sums holds the column
    sums followed by B, ready for sharding.finalize_means.  The files are decoded, filled and evaluated on the GPU; only the
    files go up and only the metrics come back.

    Raises ValueError for lists of different lengths or empty lists, and for the first frame with a file that is not an
    intact 16-bit grayscale PNG of that size (naming the LiDAR or the ground-truth list and the frame; the LiDAR file wins
    at the same frame).  Otherwise raises IndexError for the first frame Distance_Transform rejects (no valid depth,
    exactly one valid depth, labels outside the list of valid depths)."""
    from .data_read import pack_png_files
    from .tools import VALID_THR
    lidar_files, gt_files = list(lidar_files), list(gt_files)
    if not lidar_files or not gt_files:
        raise ValueError("evaluate_fill_png_files: no files")
    if len(lidar_files) != len(gt_files):
        raise ValueError(f"evaluate_fill_png_files: {len(lidar_files)} LiDAR files but {len(gt_files)} ground-truth files")
    B = len(lidar_files)
    # one buffer for both lists; the size comes from the first LiDAR file's IHDR
    try:
        data, offsets, H, W = pack_png_files(lidar_files + gt_files)
    except ValueError:
        raise ValueError("evaluate_fill_png_files: LiDAR file 0 is not a PNG file") from None
    return _lib.get_handle(device).eval_png(data, offsets[:B + 1], data, offsets[B:], H, W, src_thr, VALID_THR)


class _ResultBase(object):
    _mode = _lib.METRICS_KITTI

    def __init__(self):
        # evaluation.py:12-27 / :126-141
        self.irmse = 0
        self.imae = 0
        self.mse = 0
        self.rmse = 0
        self.mae = 0
        self.absrel = 0
        self.squared_rel = 0
        self.lg10 = 0
        self.delta1 = 0
        self.delta2 = 0
        self.delta3 = 0
        self.data_time = 0
        self.gpu_time = 0
        self.silog = 0
        self.photometric = 0
        self.count = 0.0

    # the bookkeeping half of the reference classes (evaluation.py:29-80 / :143-194): plain host arithmetic
    _AVERAGED = ("irmse", "imae", "mse", "rmse", "mae", "absrel", "squared_rel", "lg10", "delta1", "delta2", "delta3",
                 "data_time", "gpu_time", "silog", "photometric")
    _WORST_INF = ("irmse", "imae", "mse", "rmse", "mae", "absrel", "squared_rel", "lg10", "silog")
    _WORST_ZERO = ("delta1", "delta2", "delta3", "data_time", "gpu_time")

    def set_to_worst(self):
        """evaluation.py:29-43."""
        for name in self._WORST_INF:
            setattr(self, name, np.inf)
        for name in self._WORST_ZERO:
            setattr(self, name, 0)

    def update(self, irmse, imae, mse, rmse, mae, absrel, squared_rel, lg10, delta1, delta2, delta3, gpu_time,
               data_time, silog, photometric=0):
        """evaluation.py:63-79: add one frame's metrics to the running sums."""
        self.count += 1.0
        given = dict(irmse=irmse, imae=imae, mse=mse, rmse=rmse, mae=mae, absrel=absrel, squared_rel=squared_rel,
                     lg10=lg10, delta1=delta1, delta2=delta2, delta3=delta3, gpu_time=gpu_time, data_time=data_time,
                     silog=silog, photometric=photometric)
        for name, v in given.items():
            setattr(self, name, getattr(self, name) + v)

    def finalize(self):
        """evaluation.py:46-61: running sums -> means over ``count`` frames."""
        for name in self._AVERAGED:
            setattr(self, name, getattr(self, name) / self.count)

    def evaluate(self, output, target, photometric=0):
        output, target = _prep(output, target)
        per_frame, _ = _lib.get_handle().metrics(output, target, 1, 1, int(output.size), self._mode,
                                                 target.dtype == np.float64)
        m = per_frame[0]
        self.mse, self.rmse, self.mae, self.irmse, self.imae = (float(v) for v in m[:5])
        if self._mode == _lib.METRICS_NYU:
            self.delta1, self.delta2, self.delta3 = (float(v) for v in m[5:8])
        self.photometric = float(photometric)


class Result(_ResultBase):
    """evaluation.py:11-123."""
    _mode = _lib.METRICS_KITTI


class Result_NYU(_ResultBase):
    """evaluation.py:125-239."""
    _mode = _lib.METRICS_NYU
