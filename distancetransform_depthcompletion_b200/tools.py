"""Drop-in for the reference's solution_DeepNet/tools.py (same names, arguments, shapes, dtypes, exceptions),
backed by the sm_100a kernels behind libdtfill.so.  numpy in, numpy out.

    nearest_point(refined_lidar)      -> (dt float32 [H,W], lbl int32 [H,W])      tools.py:7-10
    DT_complete_batch(lidar_batch)    -> float32 [B,352,1216,1]                     tools.py:13-35

and, for the uint16 samples of KITTI's depth PNGs or the PNG files themselves, DT_complete_batch_png and
DT_complete_batch_png_files (loader + crop + fill in one call), and DT_complete_batch_png_files_to_png (files in, the
refined frames as PNG files out).
"""
from __future__ import annotations

import numpy as np

from . import _lib

KITTI_SRC_THR = 0.1     # tools.py:8   value_mask = 1.0 - x > 0.1
VALID_THR = 0.1         # tools.py:22  with_value = x > 0.1
_H, _W = 352, 1216      # tools.py:25,27 hard-coded frame size


def _as_frames_f32(a: np.ndarray, what: str) -> np.ndarray:
    if a.dtype != np.float32:
        raise TypeError(f"{what}: dtype {a.dtype} is not supported by the CUDA path (float32, or float64 / integers "
                        "through the float64 route of tools.nearest_point / DT_complete_batch / Distance_Transform)")
    return np.ascontiguousarray(a)


def _is_wide(a: np.ndarray) -> bool:
    """float64 (or integer) input: the reference evaluates its predicates in float64 (tools.py:8, :22)."""
    return a.dtype == np.float64 or np.issubdtype(a.dtype, np.integer)


def _labels_f64(frames: np.ndarray, src_thr: float, device):
    """float64 / integer frames [B,H,W]: the reference's predicates evaluated in float64 on the host (tools.py:8
    ``1.0 - x > thr``, tools.py:22 ``x > 0.1``), handed to the kernels as a float32 surrogate frame that has exactly those
    predicates in float32 (1.0: source and valid, 0.5: valid only, NaN: source only, 0.0: neither), so distances and
    labels are the reference's; the depths are gathered on the host from the float64 values (tools.py:24-26), which the
    float32 kernels cannot carry.  Returns (dt, lbl, valid masks, the run's result dict)."""
    if not (0.0 <= float(src_thr) < 0.5):
        raise TypeError("float64 input needs a source threshold in [0, 0.5) (the reference uses 0.1 and 0.001)")
    x = frames.astype(np.float64, copy=False)
    with np.errstate(invalid="ignore"):
        src = ~((1.0 - x) > src_thr)
        val = x > VALID_THR
    sur = np.zeros(x.shape, np.float32)
    sur[val] = np.float32(0.5)
    sur[src & val] = np.float32(1.0)
    sur[src & ~val] = np.float32(np.nan)
    r = _lib.get_handle(device).run_host(sur, src_thr, VALID_THR, want_dt=True, want_lbl=True)
    return r["dt"], r["lbl"], val, r


def _gather_f64(frame: np.ndarray, val: np.ndarray, lbl: np.ndarray) -> np.ndarray:
    """tools.py:24-26 on the host: depth_list = x[valid]; depth_list[lbl - 1] (numpy's own IndexError / index -1)."""
    depth_list = frame[val]
    return depth_list[lbl.reshape(-1) - 1].reshape(frame.shape)


def nearest_point(refined_lidar, thr: float = KITTI_SRC_THR, device: int | None = None):
    """tools.py:7-10.  ``thr`` is the literal 0.1 of tools.py:8 (eval_NYU.py:115 uses 0.001)."""
    x = np.squeeze(np.asarray(refined_lidar))
    if x.ndim != 2:
        # cv2.distanceTransformWithLabels accepts only a single-channel 2-D image
        raise ValueError(f"nearest_point: input must squeeze to 2-D, got shape {np.shape(refined_lidar)}")
    if _is_wide(x):
        dt, lbl, _, _ = _labels_f64(x[None], thr, device)
        return dt[0], lbl[0]
    x = _as_frames_f32(x, "nearest_point")
    r = _lib.get_handle(device).run_host(x[None], thr, VALID_THR, want_dt=True, want_lbl=True, want_counts=False)
    return r["dt"][0], r["lbl"][0]


def DT_complete_batch(lidar_batch, device: int | None = None):
    """tools.py:13-35: per frame, fill every pixel with the depth of its chamfer-nearest source."""
    lidar_batch = np.asarray(lidar_batch)
    if lidar_batch.ndim != 4:
        raise IndexError(f"DT_complete_batch: expected [B,H,W,C], got shape {lidar_batch.shape}")   # tools.py:19
    B, H, W, _ = lidar_batch.shape
    if B == 0:
        return np.expand_dims(np.asarray([]), axis=-1).astype(np.float32)                           # tools.py:30-33
    if H * W != _H * _W:
        raise ValueError(f"cannot reshape array of size {H * W} into shape ({_H},{_W})")            # tools.py:25-27
    if min(H, W) < 2:
        raise ValueError("DT_complete_batch: frames must be 2-D after squeeze")
    if _is_wide(lidar_batch):
        # float64 frames: labels from the kernels, depths gathered in float64, cast at the end like tools.py:30-33
        frames = np.ascontiguousarray(lidar_batch[:, :, :, 0])
        _, lbl, val, r = _labels_f64(frames, KITTI_SRC_THR, device)
        if "index_error" in r:
            raise IndexError(r["index_error"])                                                      # tools.py:26
        out = np.stack([_gather_f64(frames[i], val[i], lbl[i]) for i in range(B)])
        return out.reshape(B, _H, _W, 1).astype(np.float32)
    frames = _as_frames_f32(lidar_batch[:, :, :, 0], "DT_complete_batch")                           # tools.py:19
    # the result is a new array the caller owns (tools.py:27-33); its memory is page-locked and pooled so that the
    # device-to-host copy lands in it directly
    out = {"depth": _lib.output_empty((B, _H, _W), np.float32)}
    r = _lib.get_handle(device).run_host(frames, KITTI_SRC_THR, VALID_THR, want_counts=False, out=out)
    if "index_error" in r:
        raise IndexError(r["index_error"])                                                          # tools.py:26
    return r["depth"].reshape(B, _H, _W, 1)                                                         # tools.py:27-33


def dt_fill_batch(frames, src_thr: float = KITTI_SRC_THR, val_thr: float = VALID_THR, want_lbl: bool = False,
                  device: int | None = None, out=None):
    """All outputs of the path for frames float32 [B,H,W]: filled depth, distance channel, validity
    (DT-pooling, net.py:131-132) mask, optional label map, per-frame (n_sources, n_valid)."""
    frames = _as_frames_f32(np.asarray(frames), "dt_fill_batch")
    if frames.ndim != 3:
        raise ValueError("dt_fill_batch: expected [B,H,W]")
    r = _lib.get_handle(device).run_host(frames, src_thr, val_thr, want_dt=True, want_lbl=want_lbl, want_mask=True,
                                         out=out)
    if "index_error" in r:
        raise IndexError(r["index_error"])
    return r


def euclidean_feature_transform(frames, thr: float = KITTI_SRC_THR, device: int | None = None):
    """EXTENSION, not part of the reference (its transform is the 5x5 chamfer of nearest_point): the exact Euclidean
    feature transform of the same source mask (tools.py:8 predicate).  frames float32 [B,H,W] or [H,W] ->
    (d2 int32: squared distance to the nearest source, idx int32: y' * W + x' of such a source, -1 if the frame has
    none).  ``np.sqrt(d2)`` is what scipy.ndimage.distance_transform_edt returns for the mask."""
    x = _as_frames_f32(np.asarray(frames), "euclidean_feature_transform")
    single = x.ndim == 2
    if single:
        x = x[None]
    if x.ndim != 3:
        raise ValueError("euclidean_feature_transform: expected [B,H,W] or [H,W]")
    d2, idx = _lib.get_handle(device).edt(np.ascontiguousarray(x), thr)
    return (d2[0], idx[0]) if single else (d2, idx)


def DT_complete_batch_png(depth_png_batch, crop_top: int = 96, device: int | None = None):
    """The reference's loader + crop + fill in one call on the raw PNG samples (SURVEY.md 8(f-3)):

        depth = depth_png.astype(np.float32) / 256.        data_read.py:215
        lidar = depth[:, crop_top:, :, None]                train.py:211, eval.py:156  (crop_top = 96)
        refined = DT_complete_batch(lidar)                  tools.py:13-35

    depth_png_batch: uint16 [B, H_in, W] with H_in - crop_top == 352 and W == 1216 (the size tools.py hard-codes).
    Returns (lidar float32 [B,352,1216,1], refined float32 [B,352,1216,1]); the uint16 -> float32 decode and the
    crop run inside the first CUDA kernel, so the device reads 2 bytes per pixel."""
    png = np.asarray(depth_png_batch)
    if png.dtype != np.uint16:
        raise TypeError(f"DT_complete_batch_png: expected uint16 PNG samples, got {png.dtype}")
    if png.ndim != 3:
        raise IndexError(f"DT_complete_batch_png: expected [B,H_in,W], got shape {png.shape}")
    B, Hin, W = png.shape
    H = Hin - int(crop_top)
    if B == 0:
        e = np.expand_dims(np.asarray([]), axis=-1).astype(np.float32)
        return e, e
    if crop_top < 0 or H <= 0:
        raise ValueError(f"DT_complete_batch_png: crop_top {crop_top} leaves no rows of {Hin}")
    if H * W != _H * _W:
        raise ValueError(f"cannot reshape array of size {H * W} into shape ({_H},{_W})")            # tools.py:25-27
    r = _lib.get_handle(device).run_host_u16(np.ascontiguousarray(png), crop_top, KITTI_SRC_THR, VALID_THR,
                                             want_lidar=True)
    if "index_error" in r:
        raise IndexError(r["index_error"])                                                          # tools.py:26
    return r["lidar"].reshape(B, H, W, 1), r["depth"].reshape(B, _H, _W, 1)


def DT_complete_batch_png_files(files, crop_top: int = 96, device: int | None = None):
    """DT_complete_batch_png on the PNG files themselves (paths or bytes), decoded on the GPU:

        depth_png = np.array(Image.open(f), dtype=int)      data_read.py:215, per file
        ... DT_complete_batch_png(depth_png batch)

    Only the compressed files cross the PCIe link; the decoded samples never leave the device.  Same shapes, checks
    and exceptions as DT_complete_batch_png, plus ValueError for a file that is not an intact 16-bit grayscale PNG of
    the first file's size."""
    from .data_read import pack_png_files
    files = list(files)
    if not files:
        e = np.expand_dims(np.asarray([]), axis=-1).astype(np.float32)
        return e, e
    data, offsets, Hin, W = pack_png_files(files)
    B = len(files)
    H = Hin - int(crop_top)
    if crop_top < 0 or H <= 0:
        raise ValueError(f"DT_complete_batch_png_files: crop_top {crop_top} leaves no rows of {Hin}")
    if H * W != _H * _W:
        raise ValueError(f"cannot reshape array of size {H * W} into shape ({_H},{_W})")            # tools.py:25-27
    out = {"lidar": _lib.output_empty((B, H, W), np.float32), "depth": _lib.output_empty((B, H, W), np.float32)}
    r = _lib.get_handle(device).run_host_png(data, offsets, Hin, W, crop_top, KITTI_SRC_THR, VALID_THR, want_lidar=True,
                                             want_counts=False, out=out)
    if "index_error" in r:
        raise IndexError(r["index_error"])                                                          # tools.py:26
    return r["lidar"].reshape(B, H, W, 1), r["depth"].reshape(B, _H, _W, 1)


def DT_complete_batch_png_files_to_png(files, crop_top: int = 96, device: int | None = None) -> list:
    """DT_complete_batch_png_files with the refined frames written as 16-bit grayscale PNG files (KITTI's depth format,
    sample = depth * 256), all on the GPU: only compressed bytes cross the PCIe link in either direction.  Returns one
    file (bytes) per input file; each decodes to (DT_complete_batch_png_files(files)[1][..., 0] * 256).astype(np.uint16).
    The depth -> sample rule is that of data_read.write_depth_pngs.  Same checks and exceptions as
    DT_complete_batch_png_files: ValueError for a size or a broken file (naming the frame), IndexError (tools.py:26)."""
    from .data_read import pack_png_files
    files = list(files)
    if not files:
        return []
    data, offsets, Hin, W = pack_png_files(files)
    H = Hin - int(crop_top)
    if crop_top < 0 or H <= 0:
        raise ValueError(f"DT_complete_batch_png_files_to_png: crop_top {crop_top} leaves no rows of {Hin}")
    if H * W != _H * _W:
        raise ValueError(f"cannot reshape array of size {H * W} into shape ({_H},{_W})")            # tools.py:25-27
    r = _lib.get_handle(device).run_host_png_to_png(data, offsets, Hin, W, crop_top, KITTI_SRC_THR, VALID_THR)
    if "index_error" in r:
        raise IndexError(r["index_error"])                                                          # tools.py:26
    return r["files"]
