"""Drop-in for the two helper functions defined inside the reference's solution_DeepNet/eval_NYU.py:114-133, and the
script's evaluation loop on the GPU.

    nearest_point(refined_lidar)   -> (dt, lbl)          eval_NYU.py:114-117  (source threshold 0.001)
    Distance_Transform(lidar)      -> depth_map [H,W]    eval_NYU.py:120-133  (any size, dtype of the input)
    nyu_sample_coords(n)           -> (rows, cols)       data_read.py:360-364 (the random sample of one frame)
    evaluate_fill_sampled(gt, rows, cols) -> (per_frame [B,9], sums [10])   eval_NYU.py:138-254 from dense ground truth
    evaluate_fill_drawn(gt, n, rng)       -> (per_frame [B,9], sums [10])   the same loop with its draws, from rng's state
    evaluate_fill_drawn_many(gt, n, rngs) -> (per_frame [D,B,9], sums [D,10])   D such draws, each from its own generator
    evaluate_fill_kitti_png_files(lidar_files, gt) -> (per_frame [B,9], sums [10])   the script's KITTI branch, from files
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .tools import VALID_THR, _as_frames_f32, _gather_f64, _is_wide, _labels_f64
from .tools import nearest_point as _nearest_point

NYU_SRC_THR = 0.001     # eval_NYU.py:115
NYU_EVAL_CROP = (6, 234, 8, 312)      # eval_NYU.py:202-207: rows 6:234, columns 8:312 of the 240 x 320 frames are scored
KITTI_CROP_TOP = 96     # eval_NYU.py:151-165: the KITTI branch drops the first 96 rows of LiDAR and ground truth


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
    gt, is_tensor = _dense_gt(gt, device, "evaluate_fill_sampled")
    B, H, W = (int(v) for v in gt.shape)
    crop = _check_crop(crop, H, W)
    r, c, off = _sample_arrays(rows, cols, B, H, W)
    if is_tensor:
        gt = _aligned(gt)
        _torch_sync(gt)                 # the handle's stream reads gt
        h = _lib.get_handle(gt.device.index)
        return h.eval_sampled(gt.data_ptr(), B, H, W, r, c, off, crop, src_thr, VALID_THR, gt_is_device=True)
    return _lib.get_handle(device).eval_sampled(np.ascontiguousarray(gt), B, H, W, r, c, off, crop, src_thr, VALID_THR)


def _dense_gt(gt, device, who):
    """The dense float32 ground truth [B,H,W] of evaluate_fill_sampled / evaluate_fill_drawn: (a CUDA tensor or a numpy
    array, whether it is a tensor).  TypeError / ValueError before the device is touched."""
    is_tensor = type(gt).__module__.startswith("torch")
    if is_tensor:
        import torch
        if gt.dtype != torch.float32:
            raise TypeError(f"{who}: ground truth dtype {gt.dtype} not supported (float32 only)")
        if not gt.is_cuda:
            gt = gt.numpy()
            is_tensor = False
    if is_tensor and device is not None and int(device) != gt.device.index:
        raise ValueError(f"{who}: device={device} but the ground truth is on {gt.device}")
    if not is_tensor:
        gt = np.asarray(gt)
        if gt.dtype != np.float32:
            raise TypeError(f"{who}: ground truth dtype {gt.dtype} not supported (float32 only)")
    if gt.ndim != 3:
        raise ValueError(f"{who}: ground truth must be [B,H,W], got shape {tuple(gt.shape)}")
    if any(int(v) == 0 for v in gt.shape):
        raise ValueError(f"{who}: empty batch")
    return gt, is_tensor


def _torch_sync(t):
    import torch
    torch.cuda.current_stream(t.device).synchronize()


def evaluate_fill_drawn(gt, n: int, rng=np.random, crop=NYU_EVAL_CROP, src_thr: float = NYU_SRC_THR,
                        device: int | None = None, return_coords: bool = False):
    """evaluate_fill_sampled with the reference's draws made on the GPU from rng's state, that is this loop in one call:

        for b in range(B):
            rows = rng.randint(H - 12, size=n) + 6;  cols = rng.randint(W - 16, size=n) + 8   data_read.py:360-364
            Mask = np.zeros((H, W)); Mask[rows, cols] = 1
            pred = Distance_Transform(gt[b] * Mask)                                          eval_NYU.py:120-133
            result.evaluate(crop(pred), crop(gt[b]))                                          eval_NYU.py:202-207

    rng: a np.random.RandomState or the np.random module (its global state), MT19937 either way: only the generator's
    state goes up (2.5 KB), and the device reproduces randint's masked rejection on numpy's stream bit for bit.  rng
    ends where the loop leaves it, so after np.random.seed(s) this call draws the reference's masks, and the next host
    draw or the next call continues the same stream.  gt, crop, src_thr, device and the result are those of
    evaluate_fill_sampled; with return_coords the drawn (rows, cols) follow as int64 [B,n] arrays.

    Raises TypeError for an rng that is not MT19937-based (a np.random.Generator among them) and what
    evaluate_fill_sampled raises for gt and crop; ValueError with numpy's message for n < 0 ("negative dimensions are
    not allowed") and for frames too small to draw from (H <= 12 or W <= 16 with n > 0: "high <= 0") -- all before the
    device is touched and with rng untouched.  IndexError for the first frame Distance_Transform rejects (n = 0 and
    n = 1 at frame 0), with rng left after that frame's draws, as the loop leaves it."""
    gt, is_tensor = _dense_gt(gt, device, "evaluate_fill_drawn")
    if is_tensor:
        gt = _aligned(gt)
        _torch_sync(gt)                 # the handle's stream reads gt
        return _eval_drawn(lambda: _lib.get_handle(gt.device.index), gt.data_ptr(), True, gt.shape, n, rng, crop,
                           src_thr, return_coords)
    return _eval_drawn(lambda: _lib.get_handle(device), np.ascontiguousarray(gt), False, gt.shape, n, rng, crop, src_thr,
                       return_coords)


def _mt_state(rng, who="evaluate_fill_drawn"):
    get = getattr(rng, "get_state", None)
    st = get(legacy=False) if callable(get) else None
    if not isinstance(st, dict) or st.get("bit_generator") != "MT19937":
        raise TypeError(f"{who}: rng must be a np.random.RandomState or the np.random module (MT19937), got {rng!r}")
    return st


def _set_mt(rng, st, key, pos):
    """rng.set_state with the MT19937 key and pos, keeping the state's cached Gaussian."""
    rng.set_state({"bit_generator": "MT19937", "state": {"key": np.asarray(key, np.uint32), "pos": int(pos)},
                   "has_gauss": st["has_gauss"], "gauss": st["gauss"]})


def _eval_drawn(get_handle, gt, gt_is_device, shape, n, rng, crop, src_thr, return_coords):
    """The body of evaluate_fill_drawn and DTFillEngine.eval_drawn; get_handle() gives the Handle once the arguments
    are checked."""
    import operator
    from .tools import VALID_THR
    B, H, W = (int(v) for v in shape)
    crop = _check_crop(crop, H, W)
    st = _mt_state(rng)
    n = operator.index(n)
    if n < 0:
        raise ValueError("negative dimensions are not allowed")          # randint(size=n)
    if n > 0 and (H - 12 <= 0 or W - 16 <= 0):
        raise ValueError("high <= 0")
    if n == 0 and (H < 13 or W < 17):     # randint draws nothing; an empty mask leaves no valid depth in frame 0
        raise IndexError("frame 0: labels index outside the list of valid depths (numpy IndexError)")
    key, pos = np.asarray(st["state"]["key"], np.uint32), int(st["state"]["pos"])
    r = get_handle().eval_sampled_mt(gt, B, H, W, n, key, pos, crop, src_thr, VALID_THR, gt_is_device=gt_is_device,
                          want_coords=return_coords)
    if "index_error" in r:
        # the loop stops after frame first_bad's draws: replay the words every frame up to it consumed
        bg = np.random.MT19937()
        bg.state = {"bit_generator": "MT19937", "state": {"key": key, "pos": pos}}
        bg.random_raw(int(r["words"][:r["first_bad"] + 1].sum()))
        _set_mt(rng, st, bg.state["state"]["key"], bg.state["state"]["pos"])
        raise IndexError(r["index_error"])
    _set_mt(rng, st, r["key"], r["pos"])
    if return_coords:
        return r["per_frame"], r["sums"], r["rows"].astype(np.int64), r["cols"].astype(np.int64)
    return r["per_frame"], r["sums"]


def evaluate_fill_drawn_many(gt, n, rngs, crop=NYU_EVAL_CROP, src_thr: float = NYU_SRC_THR, device: int | None = None):
    """D calls of evaluate_fill_drawn over the same ground truth in one call on the GPU, that is this loop:

        for d in range(D):
            per_frame[d], sums[d] = evaluate_fill_drawn(gt, n[d], rngs[d], crop, src_thr)

    with its results bit for bit and every generator left where the loop leaves it (its cached Gaussian kept).  NYU
    numbers are reported per sample count and averaged over several random draws; a list n covers that whole grid in one
    call.  The generators are independent, so the device draws them side by side, one block each, and fills and scores
    the frames of several draws together.

    rngs: a sequence of D >= 1 MT19937 generators (np.random.RandomState, or the np.random module), no generator twice --
    the draws would then depend on each other; evaluate_fill_drawn already continues one stream over many calls.  n: one
    sample count for every draw, or a sequence of D counts.  gt, crop, src_thr, device: those of evaluate_fill_drawn.
    Returns (per_frame float64 [D,B,9], sums float64 [D,10]).

    Raises, before the device is touched and with every generator untouched: what evaluate_fill_drawn raises for any
    draw's arguments, TypeError for an n that is not an integer or a sequence, ValueError for a sequence n whose length
    is not D, for D = 0 and for a generator that appears twice.  IndexError ("draw d, frame b: ...") for the first frame
    Distance_Transform rejects, in loop order: the generators of draws before d end where their draws end, generator d
    after frame b's draws, and the generators after d stay untouched."""
    gt, is_tensor = _dense_gt(gt, device, "evaluate_fill_drawn_many")
    if is_tensor:
        gt = _aligned(gt)
        _torch_sync(gt)                 # the handle's stream reads gt
        return _eval_drawn_many(lambda: _lib.get_handle(gt.device.index), gt.data_ptr(), True, gt.shape, n, rngs, crop,
                                src_thr)
    return _eval_drawn_many(lambda: _lib.get_handle(device), np.ascontiguousarray(gt), False, gt.shape, n, rngs, crop,
                            src_thr)


def _bit_generator(rng):
    """What a generator draws from: the np.random module and the RandomState behind it are one stream, and so are
    RandomStates built on one bit generator."""
    if rng is np.random:
        rng = np.random.mtrand._rand
    return getattr(rng, "_bit_generator", rng)


def _eval_drawn_many(get_handle, gt, gt_is_device, shape, n, rngs, crop, src_thr):
    """The body of evaluate_fill_drawn_many and DTFillEngine.eval_drawn_many; get_handle() gives the Handle once the
    arguments are checked."""
    import operator
    from .tools import VALID_THR
    who = "evaluate_fill_drawn_many"
    B, H, W = (int(v) for v in shape)
    crop = _check_crop(crop, H, W)
    rngs = list(rngs)
    D = len(rngs)
    if D == 0:
        raise ValueError(f"{who}: no generators")
    states = [_mt_state(r, who) for r in rngs]
    seen = {}
    for d, r in enumerate(rngs):
        e = seen.setdefault(id(_bit_generator(r)), d)
        if e != d:
            raise ValueError(f"{who}: draws {e} and {d} share one generator; give each draw its own RandomState")
    if isinstance(n, (str, bytes)):
        raise TypeError(f"{who}: n must be an integer or a sequence of D integers, got {n!r}")
    try:
        ns = [operator.index(n)] * D
    except TypeError:
        try:
            ns = [operator.index(v) for v in n]
        except TypeError:
            raise TypeError(f"{who}: n must be an integer or a sequence of D integers, got {n!r}") from None
        if len(ns) != D:
            raise ValueError(f"{who}: {len(ns)} sample counts for {D} generators")
    for v in ns:                          # the checks of _eval_drawn, draw by draw
        if v < 0:
            raise ValueError("negative dimensions are not allowed")          # randint(size=n)
        if v > 0 and (H - 12 <= 0 or W - 16 <= 0):
            raise ValueError("high <= 0")
        if v == 0 and (H < 13 or W < 17):     # randint draws nothing; an empty mask leaves no valid depth in frame 0
            raise IndexError("draw 0, frame 0: labels index outside the list of valid depths (numpy IndexError)")
    keys = np.stack([np.asarray(st["state"]["key"], np.uint32) for st in states])
    pos = np.array([int(st["state"]["pos"]) for st in states], np.int32)
    r = get_handle().eval_sampled_mt_many(gt, B, H, W, np.array(ns, np.int32), keys, pos, crop, src_thr, VALID_THR,
                                          gt_is_device=gt_is_device)
    last = D
    if "index_error" in r:
        last = r["first_bad_draw"]
        # draw `last` stops after frame first_bad_frame's draws: replay the words every frame up to it consumed
        bg = np.random.MT19937()
        bg.state = {"bit_generator": "MT19937", "state": {"key": keys[last], "pos": int(pos[last])}}
        bg.random_raw(int(r["words"][last, :r["first_bad_frame"] + 1].sum()))
        _set_mt(rngs[last], states[last], bg.state["state"]["key"], bg.state["state"]["pos"])
    for d in range(last):
        _set_mt(rngs[d], states[d], r["keys"][d], r["pos"][d])
    if "index_error" in r:
        raise IndexError(r["index_error"])
    return r["per_frame"], r["sums"]


def _aligned(t):
    """A contiguous CUDA tensor whose data starts on a 16-byte boundary (the rows are read with 128-bit loads): t itself
    as a rule, else a copy."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def evaluate_fill_kitti_png_files(lidar_files, gt, crop_top: int = KITTI_CROP_TOP, src_thr: float = NYU_SRC_THR,
                                  device: int | None = None):
    """The KITTI branch of eval_NYU.py's evaluation loop, from the PNG files, in one call on the GPU.  The script is not
    part of this checkout; this follows SURVEY.md's record of it (section 3 B):

        for i in range(B):
            lidar = np.array(Image.open(lidar_files[i])).astype(np.float32) / 256    data_read.py:215
            gt = np.array(Image.open(gt_files[i])) / 256.                            data_read.py:223 (float64)
            lidar, gt = lidar[crop_top:], gt[crop_top:]                              eval_NYU.py:151-165
            pred = Distance_Transform(lidar, src_thr)                                eval_NYU.py:120-133 (0.001, :115)
            pred = relu(pred - 0.9) + 0.9                                            eval_NYU.py:202-206 (float32)
            result.evaluate(pred, gt)                                                evaluation.py:82-123

    lidar_files: paths or the files' bytes, 16-bit grayscale PNGs all of the size H_in x W of the first file.  gt: the
    ground truth as B such files, or as a uint16 CUDA tensor [B,H_in,W] of their samples (DTFillEngine.decode_png gives
    one), used in place on its own device: then only the LiDAR files go up, so a sweep over LiDAR densities against the
    same ground truth decodes it once.  Returns (per_frame float64 [B,9], sums float64 [10]) in the layout of
    evaluation.evaluate_batch: row b is [mse, rmse, mae, irmse, imae, 0, 0, 0, n_valid] of frame b, equal to
    Result.evaluate's bit for bit (a frame whose ground truth has no valid pixel gives numpy's mean of an empty array),
    and sums holds the column sums followed by B.  The division by the frame count (1000 in the reference) stays with
    the caller: sharding.finalize_means(sums).  device: the GPU that runs the call for ground-truth files; a tensor runs
    on its own device (a different device raises ValueError).

    Raises, before the device is touched: ValueError for empty or unequal lists, a first LiDAR file that is not a PNG,
    crop_top outside [0, H_in) and a tensor whose shape is not [B,H_in,W]; TypeError for a tensor that is not uint16 or
    not on a CUDA device.  Then ValueError for the first frame with a file that is not an intact 16-bit grayscale PNG of
    that size (naming the LiDAR or the ground-truth list and the frame; the LiDAR file wins at the same frame), and
    otherwise IndexError for the first frame Distance_Transform rejects in the cropped rows (no valid depth, exactly one
    valid depth, labels outside the list of valid depths)."""
    from .data_read import pack_png_files
    from .tools import VALID_THR
    who = "evaluate_fill_kitti_png_files"
    lidar_files = list(lidar_files)
    is_tensor = type(gt).__module__.startswith("torch")
    gt_files = None if is_tensor else list(gt)
    if not lidar_files or (gt_files is not None and not gt_files):
        raise ValueError(f"{who}: no files")
    B = len(lidar_files)
    if gt_files is not None and len(gt_files) != B:
        raise ValueError(f"{who}: {B} LiDAR files but {len(gt_files)} ground-truth files")
    try:       # the size comes from the first LiDAR file's IHDR
        data, offsets, H_in, W = pack_png_files(lidar_files + (gt_files or []))
    except ValueError:
        raise ValueError(f"{who}: LiDAR file 0 is not a PNG file") from None
    crop_top = int(crop_top)
    if not 0 <= crop_top < H_in:
        raise ValueError(f"{who}: crop_top {crop_top} outside [0, {H_in}) for frames of {H_in} rows")
    if gt_files is not None:
        return _lib.get_handle(device).eval_png_kitti(data, offsets[:B + 1], data, offsets[B:], None, H_in, W, crop_top,
                                                      src_thr, VALID_THR)
    import torch
    if gt.dtype != torch.uint16:
        raise TypeError(f"{who}: ground-truth tensor dtype {gt.dtype} not supported (uint16 PNG samples only)")
    if tuple(gt.shape) != (B, H_in, W):
        raise ValueError(f"{who}: ground-truth tensor of shape {tuple(gt.shape)}, the LiDAR files need {(B, H_in, W)}")
    if not gt.is_cuda:
        raise TypeError(f"{who}: the ground-truth tensor must be on a CUDA device, got {gt.device}")
    if device is not None and int(device) != gt.device.index:
        raise ValueError(f"{who}: device={device} but the ground truth is on {gt.device}")
    gt = gt.contiguous()
    torch.cuda.current_stream(gt.device).synchronize()      # the handle's stream reads gt
    return _lib.get_handle(gt.device.index).eval_png_kitti(data, offsets, None, None, gt.data_ptr(), H_in, W, crop_top,
                                                           src_thr, VALID_THR)
