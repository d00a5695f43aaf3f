"""CPU oracle for the DT + nearest-neighbour fill path -- TEST INFRASTRUCTURE ONLY.

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this module.  The product package never imports it (tests/test_host_logic.py::test_product_never_imports_the_oracle checks).

Three layers, each a restatement of reference lines (file:line relative to /root/reference):

* ``chamfer_l1_labels`` / ``nearest_point`` / ``dt_fill``  -- ctypes wrappers over ``dtfill_oracle.c`` (the C
  restatement of the third-party ``cv2.distanceTransformWithLabels(DIST_L1, 5, DIST_LABEL_PIXEL)`` scan called
  at solution_DeepNet/tools.py:9 and of the gather at tools.py:22-27 / eval_NYU.py:120-133).
* ``cv2_port_*`` -- the reference's own lines with the real ``cv2`` call (tools.py:7-35, eval_NYU.py:114-133),
  used as the "reference CPU path" timing arm when ``cv2`` is importable on the box.
* ``result_kitti`` / ``result_nyu`` -- numpy restatement of evaluation.py:82-123 and evaluation.py:196-239.

Parity pin: the reference ships no test vectors; the pin is the reference's own output on seeded inputs, stored under
tests/golden/ by tests/golden/make_golden.py (tests/test_oracle_golden.py, tests/test_oracle_vs_reference.py).
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libdtfill_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile dtfill_oracle.c with gcc (building the checker is not using it)."""
    src = os.path.join(_HERE, "dtfill_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc, "-O2", "-fPIC", "-std=c99", "-fno-fast-math", "-shared", "-o", _SO, src])
    return _SO


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_SO)
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int32)
        up = ctypes.POINTER(ctypes.c_uint8)
        L.oracle_chamfer_l1_labels.argtypes = [up, ctypes.c_int, ctypes.c_int, fp, ip]
        L.oracle_nearest_point_f32.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_float, fp, ip]
        L.oracle_dt_fill_f32.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                         fp, fp, ip, up]
        L.oracle_dt_fill_batch_f32.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                               ctypes.c_float, fp, fp, ip, up, ctypes.POINTER(ctypes.c_int)]
        for f in (L.oracle_chamfer_l1_labels, L.oracle_nearest_point_f32, L.oracle_dt_fill_f32,
                  L.oracle_dt_fill_batch_f32):
            f.restype = ctypes.c_int
        _lib = L
    return _lib


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def chamfer_l1_labels(mask: np.ndarray):
    """mask uint8 [H,W], 0 = source  ->  (dt float32 [H,W], lbl int32 [H,W]);  cv2 call at tools.py:9."""
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    H, W = mask.shape
    dt = np.empty((H, W), np.float32)
    lbl = np.empty((H, W), np.int32)
    rc = lib().oracle_chamfer_l1_labels(_p(mask, ctypes.c_uint8), H, W, _p(dt, ctypes.c_float),
                                        _p(lbl, ctypes.c_int32))
    if rc:
        raise RuntimeError(f"oracle_chamfer_l1_labels rc={rc}")
    return dt, lbl


def nearest_point(x: np.ndarray, thr: float = 0.1):
    """tools.py:7-10 (thr 0.1) / eval_NYU.py:114-117 (thr 0.001) for a float32 frame."""
    x = np.ascontiguousarray(np.squeeze(x), dtype=np.float32)
    H, W = x.shape
    dt = np.empty((H, W), np.float32)
    lbl = np.empty((H, W), np.int32)
    rc = lib().oracle_nearest_point_f32(_p(x, ctypes.c_float), H, W, np.float32(thr), _p(dt, ctypes.c_float),
                                        _p(lbl, ctypes.c_int32))
    if rc:
        raise RuntimeError(f"oracle_nearest_point_f32 rc={rc}")
    return dt, lbl


def dt_fill(x: np.ndarray, src_thr: float = 0.1, val_thr: float = 0.1):
    """One or many frames [H,W] / [B,H,W] float32 -> dict(depth, dt, lbl, mask); IndexError like numpy."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    single = x.ndim == 2
    xb = x[None] if single else x
    B, H, W = xb.shape
    depth = np.empty((B, H, W), np.float32)
    dt = np.empty((B, H, W), np.float32)
    lbl = np.empty((B, H, W), np.int32)
    mask = np.empty((B, H, W), np.uint8)
    bad = ctypes.c_int(-1)
    rc = lib().oracle_dt_fill_batch_f32(_p(xb, ctypes.c_float), B, H, W, np.float32(src_thr),
                                        np.float32(val_thr), _p(depth, ctypes.c_float), _p(dt, ctypes.c_float),
                                        _p(lbl, ctypes.c_int32), _p(mask, ctypes.c_uint8), ctypes.byref(bad))
    if rc in (-2, -3):
        raise IndexError(f"frame {bad.value}: label indexes outside the list of valid depths")
    if rc:
        raise RuntimeError(f"oracle_dt_fill_batch_f32 rc={rc}")
    out = dict(depth=depth, dt=dt, lbl=lbl, mask=mask)
    if single:
        out = {k: v[0] for k, v in out.items()}
    return out


# ---------------------------------------------------------------------------------------------------------
# The reference's own lines with the real cv2 call -- the "reference CPU path" used for timing.
# ---------------------------------------------------------------------------------------------------------
def have_cv2() -> bool:
    try:
        import cv2  # noqa: F401
        return True
    except Exception:
        return False


def cv2_port_nearest_point(refined_lidar, thr=0.1):
    """tools.py:7-10 / eval_NYU.py:114-117."""
    import cv2
    value_mask = np.asarray(1.0 - np.squeeze(refined_lidar) > thr).astype(np.uint8)
    dt, lbl = cv2.distanceTransformWithLabels(value_mask, cv2.DIST_L1, 5, labelType=cv2.DIST_LABEL_PIXEL)
    return dt, lbl


def cv2_port_fill_frame(frame2d, src_thr=0.1, val_thr=0.1, nyu_style=False):
    """tools.py:19-27 for one 2-D frame; ``nyu_style`` follows eval_NYU.py:120-133 instead, whose
    ``np.squeeze(lidar[with_value])`` (:126) turns a single valid depth into a 0-d array, so a frame with
    exactly one valid pixel raises IndexError there while tools.py:24 handles it.  The frame is taken as
    given (no squeeze) so that degenerate 1 x W / H x 1 test frames keep their shape."""
    import cv2
    lidar = np.asarray(frame2d)
    assert lidar.ndim == 2
    height, width = np.shape(lidar)
    with_value = lidar > val_thr
    value_mask = np.asarray(1.0 - lidar > src_thr).astype(np.uint8)
    dt, lbl = cv2.distanceTransformWithLabels(value_mask, cv2.DIST_L1, 5, labelType=cv2.DIST_LABEL_PIXEL)
    depth_list = np.squeeze(lidar[with_value]) if nyu_style else lidar[with_value]
    label_list = np.reshape(lbl, [1, height * width])
    depth_list_all = depth_list[label_list - 1]
    return np.reshape(depth_list_all, (height, width)), dt, with_value


def cv2_port_complete_batch(lidar_batch, src_thr=0.1, val_thr=0.1):
    """tools.py:13-35: per-frame loop, stack, expand_dims, astype(float32)."""
    new_batch = []
    for i in range(np.shape(lidar_batch)[0]):
        new_batch.append(cv2_port_fill_frame(lidar_batch[i, :, :, 0], src_thr, val_thr)[0])
    return np.expand_dims(np.asarray(new_batch), axis=-1).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------
# Metrics: numpy restatement of evaluation.py
# ---------------------------------------------------------------------------------------------------------
def result_kitti(output: np.ndarray, target: np.ndarray) -> dict:
    """evaluation.py:82-123 (Result.evaluate): metres -> mm and 1/km; dtype flow kept (H6)."""
    valid_mask = np.logical_and(output > 0.01, target > 0.01)          # :85-87
    output_mm = 1e3 * output[valid_mask]                               # :89  (float32 stays float32)
    target_mm = 1e3 * target[valid_mask]                               # :90
    abs_diff = np.abs(output_mm - target_mm)                           # :92
    with np.errstate(all="ignore"):
        mse = np.mean(np.power(abs_diff, 2))                           # :94
        rmse = math.sqrt(mse) if mse == mse else float("nan")          # :95
        mae = np.mean(abs_diff)                                        # :96
        inv_output_km = (1e-3 * output[valid_mask]) ** (-1)            # :116
        inv_target_km = (1e-3 * target[valid_mask]) ** (-1)            # :117
        abs_inv_diff = np.abs(inv_output_km - inv_target_km)           # :118
        irmse = np.sqrt(np.mean(np.power(abs_inv_diff, 2)))            # :119
        imae = np.mean(abs_inv_diff)                                   # :120
    return dict(mse=float(mse), rmse=float(rmse), mae=float(mae), irmse=float(irmse), imae=float(imae),
                count=int(valid_mask.sum()))


def result_nyu(output: np.ndarray, target: np.ndarray) -> dict:
    """evaluation.py:196-239 (Result_NYU.evaluate): no unit scaling; 'mae' is REL; delta1..3."""
    valid_mask = np.logical_and(output > 0.01, target > 0.01)          # :199-201
    o = output[valid_mask]                                             # :203
    t = target[valid_mask]                                             # :204
    abs_diff = np.abs(o - t)                                           # :206
    with np.errstate(all="ignore"):
        mse = np.mean(np.power(abs_diff, 2))                           # :208
        rmse = math.sqrt(mse) if mse == mse else float("nan")          # :209
        mae = np.mean(abs_diff / t)                                    # :210
        max_ratio = np.maximum(o / t, t / o)                           # :217
        d1 = np.mean(max_ratio < 1.25)                                 # :218
        d2 = np.mean(max_ratio < 1.25 ** 2)                            # :219
        d3 = np.mean(max_ratio < 1.25 ** 3)                            # :220
        inv_o = o ** (-1)                                              # :232
        inv_t = t ** (-1)                                              # :233
        abs_inv_diff = np.abs(inv_o - inv_t)                           # :234
        m2 = np.mean(np.power(abs_inv_diff, 2))
        irmse = math.sqrt(m2) if m2 == m2 else float("nan")            # :235
        imae = np.mean(abs_inv_diff)                                   # :236
    return dict(mse=float(mse), rmse=float(rmse), mae=float(mae), irmse=float(irmse), imae=float(imae),
                delta1=float(d1), delta2=float(d2), delta3=float(d3), count=int(valid_mask.sum()))


# ---------------------------------------------------------------------------------------------------------
# DT pooling of the CNN input stage (SURVEY.md section 8 f-1): numpy RESTATEMENT of net.py:71-123.
# TensorFlow is not installed in the build container.  The pin is the reference's own lines, AST-extracted and run on a
# numpy stand-in for the nine TensorFlow operations they call (tests/golden/tf_numpy_shim.py, make_golden.py): this
# restatement reproduces their outputs bit for bit (tests/test_oracle_golden.py, tests/test_oracle_vs_reference.py).
# TensorFlow's own kernels (the order of the <= T*T additions inside reduce_sum) stay unverified.
# ---------------------------------------------------------------------------------------------------------
def create_weight_matrix(table_size: int = 7) -> np.ndarray:
    """net.py:71-81: weight T - |i-mid| - |j-mid| of every window position, flattened, float32."""
    assert (table_size + 1) % 2 == 0
    middle = (table_size - 1) / 2
    w = np.zeros((table_size, table_size))
    for i in range(table_size):
        for j in range(table_size):
            w[i, j] = table_size - abs(i - middle) - abs(j - middle)
    return np.reshape(w, (table_size * table_size,)).astype(np.float32)


def _extract_patches_same(x: np.ndarray, t: int) -> np.ndarray:
    """tf.image.extract_patches(sizes=(1,t,t,1), strides 1, rates 1, padding='SAME') for x [B,H,W]:
    -> [B,H,W,t*t], window rows first, zero padded."""
    B, H, W = x.shape
    r = t // 2
    p = np.zeros((B, H + 2 * r, W + 2 * r), x.dtype)
    p[:, r:r + H, r:r + W] = x
    out = np.empty((B, H, W, t * t), x.dtype)
    k = 0
    for i in range(t):
        for j in range(t):
            out[..., k] = p[:, i:i + H, j:j + W]
            k += 1
    return out


def pool_level(lidar_data: np.ndarray, lidar_mask: np.ndarray, table_size: int = 7):
    """One level of generate_multi_channel (net.py:89-96): data, mask float32 [B,H,W] -> (pooled, new mask)."""
    w = create_weight_matrix(table_size)
    ein = _extract_patches_same(lidar_data.astype(np.float32), table_size)                       # :89
    emask = _extract_patches_same(lidar_mask.astype(np.float32), table_size)                     # :90
    mw = emask * w
    max_index = (mw == mw.max(axis=-1, keepdims=True)).astype(np.float32)                        # :91-92
    pooled = (ein * max_index).sum(axis=-1, dtype=np.float32) / (np.float32(0.000001) + max_index.sum(axis=-1, dtype=np.float32))   # :93
    return pooled.astype(np.float32), (pooled > 0.001).astype(np.float32)                        # :95-96


def generate_multi_channel(lidar_data: np.ndarray, lidar_mask: np.ndarray, table_size: int = 7, scale_num: int = 4):
    """net.py:83-123 for arrays [B,H,W] (the reference carries a trailing channel axis of 1)."""
    outs = [lidar_data.astype(np.float32)]
    d, m = lidar_data, lidar_mask
    for _ in range(scale_num - 1):
        d, m = pool_level(d, m, table_size)
        outs.append(d)
    while len(outs) < 4:
        outs.append(None)
    return tuple(outs[:4])


def demo_create_weight_matrix(size: int = 11) -> np.ndarray:
    """demo.py:65-76."""
    assert (size + 1) % 2 == 0
    middle = (size - 1) / 2
    w = np.zeros((size, size))
    for i in range(size):
        for j in range(size):
            w[i, j] = 10 ** (size - abs(i - middle) - abs(j - middle))
    return np.reshape(w, (size * size,)).astype(np.float32)


def demo_generate_multi_channel(lidar_data: np.ndarray, table_size: int = 11, scale_range: float = 90.0, scale_num: int = 4):
    """demo.py:107-149 for arrays [B,H,W] (numpy restatement of the TF lines; pinned like
    generate_multi_channel to the reference lines run on tests/golden/tf_numpy_shim.py)."""
    w = demo_create_weight_matrix(table_size)
    d = lidar_data.astype(np.float32)
    outs = [d / np.float32(scale_range)]
    for _ in range(scale_num - 1):
        ex = _extract_patches_same(d, table_size)                            # :119
        prod = ex * w
        mi = (prod == prod.max(axis=-1, keepdims=True)).astype(np.float32)   # :120
        sel = ex * mi
        d = (sel.sum(axis=-1) / (np.float32(0.000001) + np.count_nonzero(sel, axis=-1).astype(np.float32))).astype(np.float32)
        outs.append(d / np.float32(scale_range))
    while len(outs) < 4:
        outs.append(None)
    return tuple(outs[:4])



# ---------------------------------------------------------------------------------------------------------
# KITTI outlier filter (SURVEY.md section 8 f-2): data_read.py:103-128 with the real cv2.filter2D.
# ---------------------------------------------------------------------------------------------------------
def cv2_port_outlier_removal(lidar):
    """data_read.py:103-128 line by line (np.float, removed from numpy, is spelled float64 = what it aliased)."""
    import cv2
    DIAMOND_KERNEL_7 = np.asarray([[0, 0, 0, 1, 0, 0, 0], [0, 0, 1, 1, 1, 0, 0], [0, 1, 1, 1, 1, 1, 0],
                                   [1, 1, 1, 1, 1, 1, 1], [0, 1, 1, 1, 1, 1, 0], [0, 0, 1, 1, 1, 0, 0],
                                   [0, 0, 0, 1, 0, 0, 0]], dtype=np.uint8)                      # :104-113
    sparse_lidar = np.squeeze(lidar)                                                            # :115
    valid_pixels = (sparse_lidar > 0.1).astype(np.float64)                                      # :116
    lidar_sum = cv2.filter2D(sparse_lidar, -1, DIAMOND_KERNEL_7)                                # :119
    lidar_count = cv2.filter2D(valid_pixels, -1, DIAMOND_KERNEL_7)                              # :121
    lidar_aveg = lidar_sum / (lidar_count + 0.00001)                                            # :123
    potential_outliers = ((sparse_lidar - lidar_aveg) > 1.0).astype(np.float64)                 # :125
    return (sparse_lidar * (1 - potential_outliers)).astype(np.float32)                         # :128


# ------------------------------------------------------------------------------------------------------------
# Exact Euclidean feature transform (SURVEY.md 8 f-4, an extension without a reference function): the oracle is
# scipy.ndimage.distance_transform_edt on the source mask of tools.py:8; ``edt_bruteforce`` pins it on small frames.
# ------------------------------------------------------------------------------------------------------------
def source_mask(x: np.ndarray, thr: float = 0.1) -> np.ndarray:
    """tools.py:8 in float32: True where the pixel is a source (value_mask == 0)."""
    x = np.asarray(x, np.float32)
    with np.errstate(invalid="ignore"):
        return ~((np.float32(1.0) - x) > np.float32(thr))


def edt(x: np.ndarray, thr: float = 0.1):
    """(d2 int64 [H,W], idx int64 [H,W]) for one frame: squared Euclidean distance to the nearest source and the flat
    index y' * W + x' of the source scipy picked (-1 / 2^31 - 1 when the frame has no source)."""
    from scipy import ndimage
    src = source_mask(x, thr)
    H, W = src.shape
    if not src.any():
        return np.full((H, W), 2 ** 31 - 1, np.int64), np.full((H, W), -1, np.int64)
    dist, ind = ndimage.distance_transform_edt(~src, return_distances=True, return_indices=True)
    iy, ix = ind[0].astype(np.int64), ind[1].astype(np.int64)
    yy, xx = np.mgrid[0:H, 0:W]
    d2 = (yy - iy) ** 2 + (xx - ix) ** 2
    assert np.array_equal(np.rint(dist * dist).astype(np.int64), d2)
    return d2, iy * W + ix


def edt_bruteforce(x: np.ndarray, thr: float = 0.1) -> np.ndarray:
    """Squared distance to the nearest source by exhaustive search (small frames only)."""
    src = source_mask(x, thr)
    H, W = src.shape
    ys, xs = np.nonzero(src)
    if len(ys) == 0:
        return np.full((H, W), 2 ** 31 - 1, np.int64)
    yy, xx = np.mgrid[0:H, 0:W]
    d = (yy[..., None] - ys[None, None, :]) ** 2 + (xx[..., None] - xs[None, None, :]) ** 2
    return d.min(axis=-1).astype(np.int64)

