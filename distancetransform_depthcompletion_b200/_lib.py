"""ctypes binding of libdtfill.so (include/dtfill.h) -- the only way Python reaches the CUDA kernels.

There is deliberately no fallback: if the shared library is missing or no CUDA device is usable, importing the
library or creating a handle raises, loudly.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DTFILL_LIB: another build of the same library (kernel experiments); the product is the in-tree libdtfill.so
LIB_PATH = os.environ.get("DTFILL_LIB") or os.path.join(_HERE, "libdtfill.so")

E_ARG, E_CUDA, E_INDEX, E_NOMEM, E_DATA = -1, -2, -3, -4, -5
METRICS_KITTI, METRICS_NYU = 0, 1
METRIC_COLS = 9
ABI_VERSION = 9          # DTFILL_ABI_VERSION of include/dtfill.h this module was written against
METRIC_NAMES = ("mse", "rmse", "mae", "irmse", "imae", "delta1", "delta2", "delta3", "count")

_c_float_p = ctypes.POINTER(ctypes.c_float)
_c_int_p = ctypes.POINTER(ctypes.c_int)
_lib = None
_lock = threading.Lock()


class DTFillError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load libdtfill.so and declare every symbol of include/dtfill.h."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise DTFillError(
                f"{LIB_PATH} is missing: build it with `python -m distancetransform_depthcompletion_b200.build` "
                "(needs nvcc; there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        vp, ci, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
        L.dtfill_abi_version.restype = ci
        if L.dtfill_abi_version() != ABI_VERSION:
            raise DTFillError(f"{LIB_PATH} has ABI version {L.dtfill_abi_version()}, this package needs {ABI_VERSION}: "
                              "rebuild it with `python -m distancetransform_depthcompletion_b200.build`")
        L.dtfill_last_error.restype = ctypes.c_char_p
        L.dtfill_create.argtypes = [ci, ctypes.POINTER(vp)]
        L.dtfill_destroy.argtypes = [vp]
        L.dtfill_destroy.restype = None
        L.dtfill_set_stream.argtypes = [vp, vp]
        L.dtfill_synchronize.argtypes = [vp]
        L.dtfill_run.argtypes = [vp, vp, ci, ci, ci, ci, cf, cf, vp, vp, vp, vp, vp, ci, _c_int_p]
        L.dtfill_run_async.argtypes = [vp, vp, ci, ci, ci, cf, cf, vp, vp, vp, vp, vp]
        L.dtfill_status.argtypes = [vp, _c_int_p, _c_int_p]
        L.dtfill_run_eval_async.argtypes = [vp, vp, vp, ci, ci, ci, ci, cf, cf, ci, vp, vp, vp, vp, vp]
        L.dtfill_eval_totals.argtypes = [vp, vp, ci]
        L.dtfill_metrics.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, vp, ci]
        L.dtfill_metrics_ex.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, vp, ci, ci]
        L.dtfill_nccl_unique_id.argtypes = [vp]
        L.dtfill_comm_create.argtypes = [vp, vp, ci, ci, ctypes.POINTER(vp)]
        L.dtfill_comm_destroy.argtypes = [vp]
        L.dtfill_allreduce_sums.argtypes = [vp, vp, vp, ci]
        L.dtfill_set_profiling.argtypes = [vp, ci]
        L.dtfill_set_band_cap.argtypes = [vp, ci]
        L.dtfill_set_subbatches.argtypes = [vp, ci]
        L.dtfill_run_u16.argtypes = [vp, vp, ci, ci, ci, ci, ci, cf, cf, vp, vp, vp, vp, vp, vp, ci, ctypes.POINTER(ci)]
        L.dtfill_run_u16_async.argtypes = [vp, vp, ci, ci, ci, ci, cf, cf, vp, vp, vp, vp, vp, vp]
        L.dtfill_set_sky_min.argtypes = [vp, ci]
        L.dtfill_debug_set_skip.argtypes = [vp, ci]
        L.dtfill_set_stage_threads.argtypes = [vp, ci]
        L.dtfill_set_sparse_upload.argtypes = [vp, ci]
        L.dtfill_debug_compact.argtypes = [vp, ctypes.c_long, cf, cf, vp, vp, ctypes.c_long]
        L.dtfill_debug_compact.restype = ctypes.c_long
        L.dtfill_set_metrics_exact.argtypes = [vp, ci]
        L.dtfill_transfer_bytes.argtypes = [vp, ctypes.POINTER(ctypes.c_ulonglong), ctypes.POINTER(ctypes.c_ulonglong)]
        L.dtfill_set_pipeline_depth.argtypes = [vp, ci]
        L.dtfill_flush.argtypes = [vp]
        L.dtfill_debug_get_tasks.argtypes = [vp, vp, ci]
        L.dtfill_debug_get_tasks.restype = ci
        L.dtfill_kernel_times.argtypes = [vp, _c_float_p]
        L.dtfill_dt_pool.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, ci]
        L.dtfill_dt_pool_ex.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, vp, ci]
        L.dtfill_outlier_removal.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci]
        L.dtfill_dt_pool_demo.argtypes = [vp, vp, ci, ci, ci, ci, ci, ci, vp, ci]
        L.dtfill_edt.argtypes = [vp, vp, ci, ci, ci, ci, cf, vp, vp, ci]
        L.dtfill_png_decode.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp, vp, ci, ctypes.POINTER(ci)]
        L.dtfill_run_png.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, cf, cf, vp, vp, vp, vp, vp, vp, ci, ctypes.POINTER(ci)]
        L.dtfill_debug_png_decode_host.argtypes = [vp, ctypes.c_long, ci, ci, vp]
        i64 = ctypes.c_int64
        L.dtfill_png_encode_bound.argtypes = [ci, ci]
        L.dtfill_png_encode_bound.restype = i64
        L.dtfill_png_encode.argtypes = [vp, vp, ci, ci, ci, ci, vp, i64, vp, ci]
        L.dtfill_png_encode_depth.argtypes = [vp, vp, ci, ci, ci, ci, vp, i64, vp, ci]
        L.dtfill_run_png_to_png.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, cf, cf, vp, i64, vp, ci, ctypes.POINTER(ci)]
        L.dtfill_debug_png_encode_host.argtypes = [vp, ci, ci, vp, ctypes.c_long]
        L.dtfill_debug_png_encode_host.restype = ctypes.c_long
        L.dtfill_eval_png.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, cf, cf, vp, vp, ctypes.POINTER(ci)]
        L.dtfill_eval_sampled.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, vp, ci, ci, ci, ci, ci, cf, cf, vp, vp, vp,
                                          ctypes.POINTER(ci)]
        L.dtfill_debug_depth_samples_host.argtypes = [vp, ctypes.c_long, vp]
        L.dtfill_debug_depth_samples_host.restype = ci
        L.dtfill_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
        L.dtfill_host_free.argtypes = [vp]
        L.dtfill_host_free.restype = None
        for name in ("dtfill_create", "dtfill_set_stream", "dtfill_synchronize", "dtfill_run", "dtfill_run_async",
                     "dtfill_status", "dtfill_run_u16", "dtfill_run_u16_async", "dtfill_metrics", "dtfill_host_alloc", "dtfill_set_profiling", "dtfill_set_band_cap", "dtfill_set_sky_min", "dtfill_set_subbatches", "dtfill_set_pipeline_depth",
                     "dtfill_flush", "dtfill_dt_pool", "dtfill_dt_pool_ex", "dtfill_outlier_removal",
                     "dtfill_kernel_times", "dtfill_metrics_ex", "dtfill_nccl_unique_id", "dtfill_comm_create",
                     "dtfill_comm_destroy", "dtfill_allreduce_sums", "dtfill_set_stage_threads", "dtfill_debug_set_skip",
                     "dtfill_run_eval_async", "dtfill_eval_totals", "dtfill_edt", "dtfill_set_sparse_upload",
                     "dtfill_transfer_bytes", "dtfill_set_metrics_exact", "dtfill_dt_pool_demo", "dtfill_png_decode",
                     "dtfill_run_png", "dtfill_debug_png_decode_host", "dtfill_png_encode", "dtfill_png_encode_depth",
                     "dtfill_run_png_to_png", "dtfill_eval_png", "dtfill_eval_sampled"):
            getattr(L, name).restype = ci
        _lib = L
        return L


def last_error() -> str:
    return load().dtfill_last_error().decode("utf-8", "replace")


def _check(rc: int, what: str):
    if rc == 0:
        return
    msg = last_error()
    if rc == E_INDEX:
        raise IndexError(msg)
    if rc in (E_ARG, E_DATA):
        raise ValueError(f"{what}: {msg}")
    if rc == E_NOMEM:
        raise MemoryError(f"{what}: {msg}")
    raise DTFillError(f"{what}: {msg}")


def _ptr(a):
    """Address of a numpy array's buffer, or an int device pointer, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return ctypes.c_void_p(a.ctypes.data)
    return ctypes.c_void_p(int(a))


class _Serialised:
    """The library's entry points behind one lock: a dtfill_t is used from one host thread at a time (include/dtfill.h)
    and ctypes releases the GIL during a call, so two Python threads sharing the per-device handle of get_handle()
    (a loader thread and an evaluation thread, say) would otherwise interleave on its staging buffers."""

    def __init__(self, lib, lock):
        self._lib, self._lock = lib, lock

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        lock = self._lock

        def call(*args):
            with lock:
                return fn(*args)
        setattr(self, name, call)
        return call


class Handle:
    """One dtfill_t: a CUDA device, a stream and a growing workspace (include/dtfill.h).  Calls are serialised per
    handle, so a Handle may be shared between Python threads."""

    def __init__(self, device: int = 0):
        self._lock = threading.RLock()
        self._L = _Serialised(load(), self._lock)
        h = ctypes.c_void_p()
        _check(self._L.dtfill_create(int(device), ctypes.byref(h)), "dtfill_create")
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.dtfill_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int | None):
        _check(self._L.dtfill_set_stream(self._h, ctypes.c_void_p(cuda_stream or 0)), "dtfill_set_stream")

    def synchronize(self):
        _check(self._L.dtfill_synchronize(self._h), "dtfill_synchronize")

    # ---- host (numpy) path -------------------------------------------------------------------------
    def run_host(self, frames: np.ndarray, src_thr: float, val_thr: float, want_dt=False, want_lbl=False,
                 want_mask=False, want_counts=True, out=None):
        """frames float32 [B,H,W] C-contiguous -> dict of numpy outputs.  Raises IndexError like numpy."""
        assert frames.dtype == np.float32 and frames.ndim == 3 and frames.flags.c_contiguous
        B, H, W = frames.shape
        out = out or {}
        depth = out.get("depth") if out.get("depth") is not None else np.empty((B, H, W), np.float32)
        dt = (out.get("dt") if out.get("dt") is not None else np.empty((B, H, W), np.float32)) if want_dt else None
        lbl = (out.get("lbl") if out.get("lbl") is not None else np.empty((B, H, W), np.int32)) if want_lbl else None
        mask = (out.get("mask") if out.get("mask") is not None else np.empty((B, H, W), np.uint8)) if want_mask else None
        counts = np.empty((B, 2), np.int32) if want_counts else None
        bad = ctypes.c_int(-1)
        rc = self._L.dtfill_run(self._h, _ptr(frames), 0, B, H, W, float(src_thr), float(val_thr), _ptr(depth),
                                _ptr(dt), _ptr(lbl), _ptr(mask), _ptr(counts), 0, ctypes.byref(bad))
        res = dict(depth=depth, dt=dt, lbl=lbl, mask=mask, counts=counts, first_bad=bad.value)
        if rc == E_INDEX:
            res["index_error"] = last_error()
            return res
        _check(rc, "dtfill_run")
        return res

    def run_host_u16(self, png: np.ndarray, crop_top: int, src_thr: float, val_thr: float, want_lidar=False,
                     want_dt=False, want_lbl=False, want_mask=False, want_counts=True):
        """png uint16 [B,H_in,W] (KITTI depth PNG samples, depth = sample / 256; data_read.py:215); rows
        [crop_top, H_in) are processed (train.py:211).  Outputs as run_host, plus the decoded frames on request."""
        assert png.dtype == np.uint16 and png.ndim == 3 and png.flags.c_contiguous
        B, Hin, W = png.shape
        H = Hin - int(crop_top)
        lidar = np.empty((B, H, W), np.float32) if want_lidar else None
        depth = np.empty((B, H, W), np.float32)
        dt = np.empty((B, H, W), np.float32) if want_dt else None
        lbl = np.empty((B, H, W), np.int32) if want_lbl else None
        mask = np.empty((B, H, W), np.uint8) if want_mask else None
        counts = np.empty((B, 2), np.int32) if want_counts else None
        bad = ctypes.c_int(-1)
        rc = self._L.dtfill_run_u16(self._h, _ptr(png), 0, B, Hin, W, int(crop_top), float(src_thr), float(val_thr),
                                    _ptr(lidar), _ptr(depth), _ptr(dt), _ptr(lbl), _ptr(mask), _ptr(counts), 0,
                                    ctypes.byref(bad))
        res = dict(lidar=lidar, depth=depth, dt=dt, lbl=lbl, mask=mask, counts=counts, first_bad=bad.value)
        if rc == E_INDEX:
            res["index_error"] = last_error()
            return res
        _check(rc, "dtfill_run_u16")
        return res

    def png_decode(self, data: np.ndarray, offsets: np.ndarray, H: int, W: int, out=None):
        """16-bit grayscale PNG files packed back to back in data (uint8), file b = data[offsets[b]:offsets[b+1]] ->
        (samples uint16 [B,H,W], status int32 [B]).  Raises ValueError naming the first failed frame and the reason
        (the other frames are still decoded; a failed frame's samples are zero)."""
        data, offsets = _png_args(data, offsets)
        B = offsets.size - 1
        out = np.empty((B, H, W), np.uint16) if out is None else out
        assert out.dtype == np.uint16 and out.shape == (B, H, W) and out.flags.c_contiguous
        status = np.empty(B, np.int32)
        bad = ctypes.c_int(-1)
        _check(self._L.dtfill_png_decode(self._h, _ptr(data), _ptr(offsets), 0, B, int(H), int(W), _ptr(out),
                                         _ptr(status), 0, ctypes.byref(bad)), "dtfill_png_decode")
        return out, status

    def run_host_png(self, data: np.ndarray, offsets: np.ndarray, H_in: int, W: int, crop_top: int, src_thr: float,
                     val_thr: float, want_lidar=False, want_counts=True, out=None):
        """PNG files (as png_decode) decoded on the device and filled like run_host_u16, the samples never leaving the
        device.  Outputs as run_host_u16; a decode failure raises ValueError, an IndexError is reported in the dict."""
        data, offsets = _png_args(data, offsets)
        B = offsets.size - 1
        H = H_in - int(crop_top)
        out = out or {}
        lidar = (out.get("lidar") if out.get("lidar") is not None else np.empty((B, H, W), np.float32)) if want_lidar else None
        depth = out.get("depth") if out.get("depth") is not None else np.empty((B, H, W), np.float32)
        counts = np.empty((B, 2), np.int32) if want_counts else None
        bad = ctypes.c_int(-1)
        rc = self._L.dtfill_run_png(self._h, _ptr(data), _ptr(offsets), 0, B, int(H_in), int(W), int(crop_top),
                                    float(src_thr), float(val_thr), _ptr(lidar), _ptr(depth), None, None, None,
                                    _ptr(counts), 0, ctypes.byref(bad))
        res = dict(lidar=lidar, depth=depth, counts=counts, first_bad=bad.value)
        if rc == E_INDEX:
            res["index_error"] = last_error()
            return res
        _check(rc, "dtfill_run_png")
        return res

    def png_decode_device_async(self, data_ptr: int, offsets_ptr: int, B: int, H: int, W: int, out_ptr: int,
                                status_ptr: int):
        """Device files and offsets -> device samples and status, enqueued on the handle's stream only."""
        bad = ctypes.c_int(-1)
        _check(self._L.dtfill_png_decode(self._h, _ptr(data_ptr), _ptr(offsets_ptr), 1, int(B), int(H), int(W),
                                         _ptr(out_ptr), _ptr(status_ptr), 1, ctypes.byref(bad)), "dtfill_png_decode")

    def png_encode(self, samples: np.ndarray) -> list:
        """uint16 samples [B,H,W] -> B 16-bit grayscale PNG files (list of bytes), encoded on the device."""
        return self._png_encode(samples, np.uint16, "dtfill_png_encode")

    def png_encode_depth(self, depth: np.ndarray) -> list:
        """float32 depth in metres [B,H,W] -> B 16-bit grayscale PNG files (list of bytes), encoded on the device with
        sample = clip(nan_to_num(fl32(d * 256), nan=0, posinf=65535), 0, 65535) truncated toward zero, which is
        (d * 256).astype(np.uint16) for d in [0, 65535/256] and the identity on d = k/256."""
        return self._png_encode(depth, np.float32, "dtfill_png_encode_depth")

    def _png_encode(self, x, dtype, fn):
        x = np.ascontiguousarray(x)
        assert x.dtype == dtype and x.ndim == 3, (x.dtype, x.shape)
        B, H, W = x.shape
        cap = B * png_encode_bound(H, W)
        # pageable and untouched beyond offsets[B]: only the bytes of the files are copied into it
        out = np.empty(cap, np.uint8)
        offsets = np.empty(B + 1, np.int64)
        _check(getattr(self._L, fn)(self._h, _ptr(x), 0, B, H, W, _ptr(out), cap, _ptr(offsets), 0), fn)
        return _split_files(out, offsets)

    def run_host_png_to_png(self, data: np.ndarray, offsets: np.ndarray, H_in: int, W: int, crop_top: int,
                            src_thr: float, val_thr: float):
        """PNG files (as png_decode) decoded, filled like run_host_png and the filled depth encoded, all on the device ->
        dict(files=list of bytes, first_bad).  A decode failure raises ValueError; an IndexError is reported in the dict
        under "index_error" (the files of all frames are still returned)."""
        data, offsets = _png_args(data, offsets)
        B = offsets.size - 1
        H = H_in - int(crop_top)
        cap = B * png_encode_bound(H, W)
        out = np.empty(cap, np.uint8)
        out_off = np.empty(B + 1, np.int64)
        bad = ctypes.c_int(-1)
        rc = self._L.dtfill_run_png_to_png(self._h, _ptr(data), _ptr(offsets), 0, B, int(H_in), int(W), int(crop_top),
                                           float(src_thr), float(val_thr), _ptr(out), cap, _ptr(out_off), 0,
                                           ctypes.byref(bad))
        res = dict(first_bad=bad.value)
        if rc == E_INDEX:
            res["index_error"] = last_error()
        else:
            _check(rc, "dtfill_run_png_to_png")
        res["files"] = _split_files(out, out_off)
        return res

    def eval_png(self, lidar_data: np.ndarray, lidar_off: np.ndarray, gt_data: np.ndarray, gt_off: np.ndarray, H: int,
                 W: int, src_thr: float, val_thr: float):
        """B LiDAR and B ground-truth PNG files (each set packed as for png_decode) decoded, the LiDAR frames filled and
        KITTI-mode metrics taken against the ground truth, all on the device -> (per_frame [B,9], sums [10]) float64,
        bit-exact with Result.evaluate.  A decode failure raises ValueError naming the list and the frame; a frame
        Distance_Transform rejects raises IndexError."""
        lidar_data, lidar_off = _png_args(lidar_data, lidar_off)
        gt_data, gt_off = _png_args(gt_data, gt_off)
        B = lidar_off.size - 1
        if gt_off.size - 1 != B:
            raise ValueError(f"dtfill_eval_png: {B} LiDAR files but {gt_off.size - 1} ground-truth files")
        per_frame = np.empty((B, METRIC_COLS), np.float64)
        sums = np.empty(METRIC_COLS + 1, np.float64)
        bad = ctypes.c_int(-1)
        _check(self._L.dtfill_eval_png(self._h, _ptr(lidar_data), _ptr(lidar_off), _ptr(gt_data), _ptr(gt_off), B,
                                       int(H), int(W), float(src_thr), float(val_thr), _ptr(per_frame), _ptr(sums),
                                       ctypes.byref(bad)), "dtfill_eval_png")
        return per_frame, sums

    def eval_sampled(self, gt, B: int, H: int, W: int, rows, cols, offsets, crop, src_thr: float, val_thr: float,
                     gt_is_device: bool = False, coords_are_device: bool = False, want_lidar: bool = False):
        """The NYU evaluation loop on B frames of dense float32 ground truth gt [B,H,W] (a numpy array, or a device pointer
        with gt_is_device): frame b keeps the pixels rows[k], cols[k] for k in [offsets[b], offsets[b+1]) (int32 / int64
        numpy arrays, or device pointers with coords_are_device), is filled, and the crop window (r0, r1, c0, c1) is scored
        in NYU mode, all on the device -> (per_frame [B,9], sums [10]) float64, plus the sparse frames gt * Mask float32
        [B,H,W] with want_lidar.  Coordinates outside the frame and decreasing offsets raise ValueError, a frame
        Distance_Transform rejects raises IndexError."""
        r0, r1, c0, c1 = (int(v) for v in crop)
        if not gt_is_device:
            assert gt.dtype == np.float32 and gt.shape == (B, H, W) and gt.flags.c_contiguous
        if not coords_are_device:
            assert rows.dtype == np.int32 and cols.dtype == np.int32 and offsets.dtype == np.int64 and offsets.size == B + 1
        per_frame = np.empty((B, METRIC_COLS), np.float64)
        sums = np.empty(METRIC_COLS + 1, np.float64)
        lidar = np.empty((B, H, W), np.float32) if want_lidar else None
        bad = ctypes.c_int(-1)
        _check(self._L.dtfill_eval_sampled(self._h, _ptr(gt), int(bool(gt_is_device)), int(B), int(H), int(W), _ptr(rows),
                                           _ptr(cols), _ptr(offsets), int(bool(coords_are_device)), r0, r1, c0, c1,
                                           float(src_thr), float(val_thr), _ptr(lidar), _ptr(per_frame), _ptr(sums),
                                           ctypes.byref(bad)), "dtfill_eval_sampled")
        return (per_frame, sums, lidar) if want_lidar else (per_frame, sums)

    def png_encode_device_async(self, in_ptr: int, is_float: bool, B: int, H: int, W: int, out_ptr: int,
                                capacity: int, offsets_ptr: int):
        """Device frames (uint16, or float32 depth when is_float) -> device files + offsets [B+1], enqueued on the
        handle's stream only."""
        fn = "dtfill_png_encode_depth" if is_float else "dtfill_png_encode"
        _check(getattr(self._L, fn)(self._h, _ptr(in_ptr), 1, int(B), int(H), int(W), _ptr(out_ptr), int(capacity),
                                    _ptr(offsets_ptr), 1), fn)

    # ---- device path (raw pointers, e.g. torch tensors' data_ptr()) ------------------------------------
    def run_device_u16_async(self, in_ptr: int, B: int, H_in: int, W: int, crop_top: int, src_thr: float,
                             val_thr: float, depth_ptr: int, lidar_ptr: int | None = None, dt_ptr: int | None = None,
                             lbl_ptr: int | None = None, mask_ptr: int | None = None, counts_ptr: int | None = None):
        _check(self._L.dtfill_run_u16_async(self._h, _ptr(in_ptr), B, H_in, W, int(crop_top), float(src_thr),
                                            float(val_thr), _ptr(lidar_ptr), _ptr(depth_ptr), _ptr(dt_ptr),
                                            _ptr(lbl_ptr), _ptr(mask_ptr), _ptr(counts_ptr)), "dtfill_run_u16_async")

    def run_device_async(self, in_ptr: int, B: int, H: int, W: int, src_thr: float, val_thr: float, depth_ptr: int,
                         dt_ptr: int | None = None, lbl_ptr: int | None = None, mask_ptr: int | None = None,
                         counts_ptr: int | None = None):
        _check(self._L.dtfill_run_async(self._h, _ptr(in_ptr), B, H, W, float(src_thr), float(val_thr), _ptr(depth_ptr),
                                        _ptr(dt_ptr), _ptr(lbl_ptr), _ptr(mask_ptr), _ptr(counts_ptr)),
               "dtfill_run_async")

    def run_eval_async(self, in_ptr: int, gt_ptr: int, gt_is_f64: bool, B: int, H: int, W: int, src_thr: float,
                       val_thr: float, mode: int, depth_ptr: int, dt_ptr=None, lbl_ptr=None, mask_ptr=None,
                       counts_ptr=None):
        """Fill + per-frame metrics of the filled depth against gt, added to the handle's running totals."""
        _check(self._L.dtfill_run_eval_async(self._h, _ptr(in_ptr), _ptr(gt_ptr), int(bool(gt_is_f64)), B, H, W,
                                             float(src_thr), float(val_thr), int(mode), _ptr(depth_ptr), _ptr(dt_ptr),
                                             _ptr(lbl_ptr), _ptr(mask_ptr), _ptr(counts_ptr)), "dtfill_run_eval_async")

    def eval_totals(self, sums_ptr: int, accumulate: bool = False):
        """Join the calls in flight and write / add the running totals [10] to the device vector at sums_ptr."""
        _check(self._L.dtfill_eval_totals(self._h, _ptr(sums_ptr), int(bool(accumulate))), "dtfill_eval_totals")

    def status(self):
        """Synchronise; returns (first_bad_frame or -1, kernel launches of the last run)."""
        bad, launches = ctypes.c_int(-1), ctypes.c_int(0)
        rc = self._L.dtfill_status(self._h, ctypes.byref(bad), ctypes.byref(launches))
        if rc not in (0, E_INDEX):
            _check(rc, "dtfill_status")
        return bad.value, launches.value

    KERNEL_NAMES = ("k1_mask_rows", "k1b_scan_compact", "k2_chamfer", "k2_chamfer_wide", "k3_sky")

    def set_band_cap(self, cap: int):
        """Band planner target (row steps per task): >0 explicit, 0 never split frames, -1 automatic."""
        _check(self._L.dtfill_set_band_cap(self._h, int(cap)), "dtfill_set_band_cap")

    def debug_set_skip(self, mask: int):
        """Tuning only: stages whose bit is set (0 K1, 1 K1b, 2 K2, 3 k3_sky) are not launched by the next runs."""
        _check(self._L.dtfill_debug_set_skip(self._h, int(mask)), "dtfill_debug_set_skip")

    def set_sky_min(self, rows: int):
        """Least number of source-free top rows handed to the closed-form kernel k3_sky; 0: never; -1 (default): 8."""
        _check(self._L.dtfill_set_sky_min(self._h, int(rows)), "dtfill_set_sky_min")

    def set_stage_threads(self, threads: int):
        """Host threads per direction that stage pageable numpy buffers through pinned mirrors (-1 auto, 0 never)."""
        _check(self._L.dtfill_set_stage_threads(self._h, int(threads)), "dtfill_set_stage_threads")

    def set_metrics_exact(self, enabled: bool):
        """metrics(): numpy's pairwise summation order, bit for bit (default), or one-pass fixed-order float64 sums."""
        _check(self._L.dtfill_set_metrics_exact(self._h, int(bool(enabled))), "dtfill_set_metrics_exact")

    def set_sparse_upload(self, enabled: bool):
        """Pageable float32 host inputs are compacted to (index, value) pairs on the host instead of mirrored (default on)."""
        _check(self._L.dtfill_set_sparse_upload(self._h, int(bool(enabled))), "dtfill_set_sparse_upload")

    def transfer_bytes(self):
        """(host-to-device, device-to-host) bytes the last synchronous call with host buffers moved over the link."""
        a, b = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        _check(self._L.dtfill_transfer_bytes(self._h, ctypes.byref(a), ctypes.byref(b)), "dtfill_transfer_bytes")
        return int(a.value), int(b.value)

    def set_pipeline_depth(self, depth: int):
        """2: consecutive run_device_async calls may overlap (outputs final after flush()/status()); 1: strict."""
        _check(self._L.dtfill_set_pipeline_depth(self._h, int(depth)), "dtfill_set_pipeline_depth")

    def flush(self):
        """Pipelined mode: make the handle's stream wait for every call still in flight."""
        _check(self._L.dtfill_flush(self._h), "dtfill_flush")

    def set_subbatches(self, n: int):
        """Number of sub-batches run on forked streams (<= 0: automatic)."""
        _check(self._L.dtfill_set_subbatches(self._h, int(n)), "dtfill_set_subbatches")

    TASK_FIELDS = ("frame", "lo", "hi", "r0", "r1", "kind", "scratch_off", "fstart", "clo", "c0", "c1", "sky")

    def debug_tasks(self, max_tasks: int = 1 << 16) -> np.ndarray:
        """Tiles the planner produced for the last run: int32 [n, 12] (TASK_FIELDS), unused slots removed."""
        buf = np.zeros((max_tasks, 12), np.int32)
        n = self._L.dtfill_debug_get_tasks(self._h, _ptr(buf), max_tasks)
        if n < 0:
            _check(n, "dtfill_debug_get_tasks")
        t = buf[:n]
        return t[t[:, 5] != 3]

    def set_profiling(self, enabled: bool):
        _check(self._L.dtfill_set_profiling(self._h, int(bool(enabled))), "dtfill_set_profiling")

    def kernel_times(self) -> dict:
        """Milliseconds of each kernel of the last run (CUDA events on the handle's stream); profiling must be on."""
        ms = (ctypes.c_float * len(self.KERNEL_NAMES))()
        _check(self._L.dtfill_kernel_times(self._h, ms), "dtfill_kernel_times")
        return dict(zip(self.KERNEL_NAMES, (float(v) for v in ms)))

    def dt_pool(self, data, mask, B: int, H: int, W: int, table_size: int, scale_num: int, on_device: bool = False,
                out_ptr=None, want_masks: bool = False, masks_ptr=None):
        """DT pooling levels 2..scale_num (net.py:83-123).  Host arrays -> numpy [scale_num-1,B,H,W] (with
        want_masks: a pair, the second the uint8 level masks ``level > 0.001``)."""
        if scale_num <= 1:
            e = np.empty((0, B, H, W), np.float32)
            return (e, np.empty((0, B, H, W), np.uint8)) if want_masks else e
        if not on_device:
            out = np.empty((scale_num - 1, B, H, W), np.float32)
            masks = np.empty((scale_num - 1, B, H, W), np.uint8) if want_masks else None
            _check(self._L.dtfill_dt_pool_ex(self._h, _ptr(data), _ptr(mask), 0, B, H, W, table_size, scale_num,
                                             _ptr(out), _ptr(masks), 0), "dtfill_dt_pool")
            return (out, masks) if want_masks else out
        _check(self._L.dtfill_dt_pool_ex(self._h, _ptr(data), _ptr(mask), 1, B, H, W, table_size, scale_num,
                                         _ptr(out_ptr), _ptr(masks_ptr), 1), "dtfill_dt_pool")
        return None

    def dt_pool_demo(self, data: np.ndarray, B: int, H: int, W: int, table_size: int, scale_num: int) -> np.ndarray:
        """demo.py:65-149 pooling levels 2..scale_num (before the division by scale_range): float32 [scale_num-1,B,H,W]."""
        out = np.empty((max(scale_num - 1, 0), B, H, W), np.float32)
        _check(self._L.dtfill_dt_pool_demo(self._h, _ptr(data), 0, B, H, W, int(table_size), int(scale_num), _ptr(out), 0),
               "dtfill_dt_pool_demo")
        return out

    def edt(self, frames: np.ndarray, src_thr: float, want_idx: bool = True):
        """Exact Euclidean feature transform (extension): frames float32 [B,H,W] -> (d2 int32, idx int32 or None)."""
        B, H, W = frames.shape
        d2 = np.empty((B, H, W), np.int32)
        idx = np.empty((B, H, W), np.int32) if want_idx else None
        _check(self._L.dtfill_edt(self._h, _ptr(frames), 0, B, H, W, float(src_thr), _ptr(d2), _ptr(idx), 0), "dtfill_edt")
        return d2, idx

    def outlier_removal(self, frames: np.ndarray) -> np.ndarray:
        """frames float32 [B,H,W] -> filtered float32 [B,H,W] (data_read.py:103-128)."""
        B, H, W = frames.shape
        out = np.empty((B, H, W), np.float32)
        _check(self._L.dtfill_outlier_removal(self._h, _ptr(frames), 0, B, H, W, _ptr(out), 0), "dtfill_outlier_removal")
        return out

    def metrics(self, pred, gt, B: int, H: int, W: int, mode: int, gt_is_f64: bool, on_device: bool = False,
                per_frame_ptr=None, sums_ptr=None, accumulate: bool = False):
        """Host arrays (on_device False) -> (per_frame [B,9], sums [10]) numpy; device pointers otherwise
        (accumulate: add this batch's totals to the device vector at sums_ptr instead of overwriting it)."""
        if accumulate:
            _check(self._L.dtfill_metrics_ex(self._h, _ptr(pred), _ptr(gt), int(gt_is_f64), 1, B, H, W, mode,
                                             _ptr(per_frame_ptr), _ptr(sums_ptr), 1, 1), "dtfill_metrics_ex")
            return None
        if not on_device:
            per_frame = np.empty((B, METRIC_COLS), np.float64)
            sums = np.empty(METRIC_COLS + 1, np.float64)
            _check(self._L.dtfill_metrics(self._h, _ptr(pred), _ptr(gt), int(gt_is_f64), 0, B, H, W, mode,
                                          _ptr(per_frame), _ptr(sums), 0), "dtfill_metrics")
            return per_frame, sums
        _check(self._L.dtfill_metrics(self._h, _ptr(pred), _ptr(gt), int(gt_is_f64), 1, B, H, W, mode,
                                      _ptr(per_frame_ptr), _ptr(sums_ptr), 1), "dtfill_metrics")
        return None


    # ---- the one collective of the path (include/dtfill.h: dtfill_allreduce_sums) --------------------------
    def comm_create(self, unique_id: bytes, nranks: int, rank: int) -> int:
        """ncclCommInitRank on this handle's device; returns the ncclComm_t as an int."""
        assert len(unique_id) == NCCL_ID_BYTES
        buf = ctypes.create_string_buffer(unique_id, NCCL_ID_BYTES)
        comm = ctypes.c_void_p()
        _check(self._L.dtfill_comm_create(self._h, buf, int(nranks), int(rank), ctypes.byref(comm)), "dtfill_comm_create")
        return comm.value

    def allreduce_sums(self, comm: int, sums_ptr: int, n: int):
        """In-place NCCL sum all-reduce of n float64 at the device pointer, enqueued on the handle's stream."""
        _check(self._L.dtfill_allreduce_sums(self._h, ctypes.c_void_p(comm), _ptr(sums_ptr), int(n)), "dtfill_allreduce_sums")


NCCL_ID_BYTES = 128

PNG_STATUS = ("ok", "bad signature", "unsupported IHDR", "size differs from the batch's",
              "broken or truncated chunk structure, or no IDAT", "bad zlib header", "invalid DEFLATE data",
              "decompressed size differs from H*(1+2W)", "filter type > 4", "Adler-32 mismatch")


def _png_args(data, offsets):
    data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64).reshape(-1)
    if offsets.size < 2:
        raise ValueError("PNG decode: offsets must hold B + 1 >= 2 entries")
    if offsets[0] < 0 or offsets[-1] > data.size or np.any(np.diff(offsets) < 0):
        raise ValueError("PNG decode: offsets must be non-decreasing and lie within the data")
    return data, offsets


def png_decode_host(png: bytes, H: int, W: int):
    """Test hook: the decode of one file run serially on the CPU (no GPU) -> (status, samples uint16 [H,W])."""
    png = bytes(png)
    buf = np.frombuffer(png or b"\0", np.uint8)
    out = np.empty((H, W), np.uint16)
    st = load().dtfill_debug_png_decode_host(_ptr(buf), len(png), int(H), int(W), _ptr(out))
    if st < 0:
        raise ValueError("dtfill_debug_png_decode_host: bad arguments")
    return st, out


def png_encode_bound(H: int, W: int) -> int:
    """Worst-case bytes of one encoded file of H x W samples (include/dtfill.h dtfill_png_encode_bound)."""
    n = load().dtfill_png_encode_bound(int(H), int(W))
    if n < 0:
        raise ValueError(f"PNG encode: unsupported size {H} x {W} (H * (1 + 2 W) < 2^28)")
    return n


def _split_files(buf: np.ndarray, offsets: np.ndarray) -> list:
    return [buf[offsets[b]:offsets[b + 1]].tobytes() for b in range(offsets.size - 1)]


def png_encode_host(samples) -> bytes:
    """Test hook: the encoder run serially on the CPU (no GPU): uint16 [H,W] -> the PNG file the device writes."""
    x = np.ascontiguousarray(samples)
    if x.dtype != np.uint16 or x.ndim != 2:
        raise TypeError(f"png_encode_host: uint16 [H,W] expected, got {x.dtype} {x.shape}")
    H, W = x.shape
    cap = png_encode_bound(H, W)
    out = np.empty(cap, np.uint8)
    n = load().dtfill_debug_png_encode_host(_ptr(x), H, W, _ptr(out), cap)
    if n < 0:
        raise ValueError("dtfill_debug_png_encode_host: bad arguments")
    return out[:n].tobytes()


def depth_samples_host(depth) -> np.ndarray:
    """Test hook: the depth -> sample rule of png_encode_depth run on the CPU: float32 array -> uint16 array."""
    x = np.ascontiguousarray(depth, dtype=np.float32)
    out = np.empty(x.shape, np.uint16)
    if load().dtfill_debug_depth_samples_host(_ptr(x), x.size, _ptr(out)) != 0:
        raise ValueError("dtfill_debug_depth_samples_host: bad arguments")
    return out

def nccl_unique_id() -> bytes:
    buf = ctypes.create_string_buffer(NCCL_ID_BYTES)
    _check(load().dtfill_nccl_unique_id(buf), "dtfill_nccl_unique_id")
    return buf.raw


def comm_destroy(comm: int):
    if comm:
        _check(load().dtfill_comm_destroy(ctypes.c_void_p(comm)), "dtfill_comm_destroy")


_handles: dict[int, Handle] = {}


def default_device() -> int:
    for k in ("DTFILL_DEVICE", "LOCAL_RANK"):
        if os.environ.get(k, "") != "":
            return int(os.environ[k])
    return 0


def get_handle(device: int | None = None) -> Handle:
    d = default_device() if device is None else int(device)
    with _lock:
        h = _handles.get(d)
    if h is None:
        h = Handle(d)
        with _lock:
            _handles[d] = h
    return h


class _PinnedBlock:
    """Owner of one page-locked host buffer; numpy arrays made from it keep it alive through ``.base``.  When the last
    array goes away the buffer returns to the pool (pooled blocks) or is freed."""

    def __init__(self, ptr: int, nbytes: int, shape, dtype, pooled: bool):
        self.ptr, self.nbytes, self.pooled = ptr, nbytes, pooled
        self.__array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": np.dtype(dtype).str,
                                    "data": (ptr, False), "version": 3}

    def __del__(self):
        try:
            _pinned_release(self.ptr, self.nbytes, self.pooled)
        except Exception:       # interpreter shutdown
            pass


_pin_lock = threading.Lock()
_pin_free: dict[int, list[int]] = {}      # size -> free pooled buffers
_pin_free_bytes = 0
# most page-locked memory kept for reuse by pinned_empty(pooled=True) (outputs handed to numpy callers)
PINNED_POOL_MAX = int(os.environ.get("DTFILL_PINNED_POOL_MAX", str(4 << 30)))
# largest single output that is handed out as page-locked memory at all (larger ones are ordinary numpy arrays)
PINNED_OUT_MAX = int(os.environ.get("DTFILL_PINNED_OUT_MAX", str(1 << 30)))


def _pinned_release(ptr: int, nbytes: int, pooled: bool):
    global _pin_free_bytes
    if pooled:
        with _pin_lock:
            if _pin_free_bytes + nbytes <= PINNED_POOL_MAX:
                _pin_free.setdefault(nbytes, []).append(ptr)
                _pin_free_bytes += nbytes
                return
    load().dtfill_host_free(ctypes.c_void_p(ptr))


def pinned_empty(shape, dtype=np.float32, pooled: bool = False) -> np.ndarray:
    """numpy array backed by page-locked host memory (dtfill_host_alloc): host<->device copies run at PCIe speed and
    need no staging.  The memory is released when the array (and every view of it) is gone; with ``pooled`` it goes
    back to a free list instead, so that a loop which receives a fresh output array per call does not pay for page
    locking (or for the page faults of a fresh pageable array) every time."""
    global _pin_free_bytes
    L = load()
    dtype = np.dtype(dtype)
    n = max(int(np.prod(shape)) * dtype.itemsize, 1)
    ptr = None
    if pooled:
        with _pin_lock:
            lst = _pin_free.get(n)
            if lst:
                ptr = lst.pop()
                _pin_free_bytes -= n
    if ptr is None:
        p = ctypes.c_void_p()
        _check(L.dtfill_host_alloc(ctypes.byref(p), n), "dtfill_host_alloc")
        ptr = p.value
    return np.asarray(_PinnedBlock(ptr, n, shape, dtype, pooled))


def output_empty(shape, dtype=np.float32) -> np.ndarray:
    """A fresh array for a result handed to a numpy caller (tools.py:13-35 returns a new array every call): page-locked
    and pooled up to PINNED_OUT_MAX bytes, so the device-to-host copy lands in it directly; ordinary memory above that."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    if 0 < n <= PINNED_OUT_MAX:
        try:
            return pinned_empty(shape, dtype, pooled=True)
        except (MemoryError, DTFillError):
            pass
    return np.empty(shape, dtype)
