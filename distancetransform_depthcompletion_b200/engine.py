"""Device-resident form of the path for callers that already hold their frames in HBM (torch tensors).

PyTorch is used here only for device memory and streams; every kernel is ours (libdtfill.so).
"""
from __future__ import annotations

from . import _lib


class DTFillEngine:
    """Runs DT + NN fill (+ metrics) on torch CUDA tensors, on torch's current stream, without host copies."""

    def __init__(self, device: int | None = None, pipeline_depth: int = 1):
        """pipeline_depth 2..4: consecutive fill() calls may overlap on the GPU (the HBM-bound first stage of one batch
        with the ALU-bound scan of the previous one); their outputs are final after flush() / status(), and a
        call's output tensors must not be handed to the next call.  Inputs and outputs of the calls in flight are
        kept alive by the engine until flush() / status() / eval_totals()."""
        import torch
        self.torch = torch
        self.device = _lib.default_device() if device is None else int(device)
        self.handle = _lib.Handle(self.device)
        self.pipeline_depth = max(1, int(pipeline_depth))
        if pipeline_depth != 1:
            self.handle.set_pipeline_depth(pipeline_depth)
        # pipelined mode: the kernels of a call run on library-internal streams that torch's caching allocator knows
        # nothing about, so the tensors of the calls in flight are kept alive here until they have been joined
        self._inflight = {}

    def _hold(self, *tensors):
        if self.pipeline_depth > 1:
            key = tuple(t.data_ptr() for t in tensors if t is not None)
            self._inflight[key] = tensors
            if len(self._inflight) > 8 * self.pipeline_depth:
                # a caller that allocates fresh tensors for every call: join the calls in flight (stream-level, no
                # host synchronisation) so that the older tensors can go back to the allocator
                self.handle.flush()
                self._inflight = {key: tensors}

    def close(self):
        """Wait for the work in flight and release the handle."""
        if getattr(self, "handle", None) is not None:
            try:
                self.handle.synchronize()
            finally:
                self._inflight = {}
                self.handle.close()
                self.handle = None

    def _bind_stream(self):
        # torch reports the legacy default stream as handle 0; CUDA's explicit handle for it is cudaStreamLegacy (0x1)
        self.handle.set_stream(self.torch.cuda.current_stream(self.device).cuda_stream or 0x1)

    def fill(self, frames, src_thr: float = 0.1, val_thr: float = 0.1, want_lbl: bool = False, out=None):
        """frames: float32 CUDA tensor [B,H,W] (contiguous).  Returns dict of CUDA tensors, enqueued only."""
        torch = self.torch
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.is_contiguous() and frames.dim() == 3
        B, H, W = frames.shape
        out = out or {}
        dev = frames.device
        depth = out.get("depth") if out.get("depth") is not None else torch.empty((B, H, W), dtype=torch.float32, device=dev)
        dt = out.get("dt") if out.get("dt") is not None else torch.empty((B, H, W), dtype=torch.float32, device=dev)
        mask = out.get("mask") if out.get("mask") is not None else torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        lbl = None
        if want_lbl:
            lbl = out.get("lbl") if out.get("lbl") is not None else torch.empty((B, H, W), dtype=torch.int32, device=dev)
        counts = out.get("counts") if out.get("counts") is not None else torch.empty((B, 2), dtype=torch.int32, device=dev)
        self._bind_stream()
        self.handle.run_device_async(frames.data_ptr(), B, H, W, src_thr, val_thr, depth.data_ptr(), dt.data_ptr(),
                                     lbl.data_ptr() if lbl is not None else None, mask.data_ptr(), counts.data_ptr())
        self._hold(frames, depth, dt, mask, lbl, counts)
        return dict(depth=depth, dt=dt, mask=mask, lbl=lbl, counts=counts)

    def fill_eval(self, frames, gt, mode: int = _lib.METRICS_KITTI, src_thr: float = 0.1, val_thr: float = 0.1, out=None):
        """One step of an evaluation sweep (eval.py:212-232): fill ``frames`` and add the per-frame metrics of the filled
        depth against ``gt`` (float32/float64 CUDA tensor [B,H,W]) to the engine's running totals; enqueued only,
        pipelined like fill().  Collect with eval_totals()."""
        torch = self.torch
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.is_contiguous() and frames.dim() == 3
        assert gt.is_cuda and gt.is_contiguous() and gt.shape == frames.shape and gt.dtype in (torch.float32, torch.float64)
        B, H, W = frames.shape
        out = out or {}
        dev = frames.device
        depth = out.get("depth") if out.get("depth") is not None else torch.empty((B, H, W), dtype=torch.float32, device=dev)
        dt = out.get("dt") if out.get("dt") is not None else torch.empty((B, H, W), dtype=torch.float32, device=dev)
        mask = out.get("mask") if out.get("mask") is not None else torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        counts = out.get("counts") if out.get("counts") is not None else torch.empty((B, 2), dtype=torch.int32, device=dev)
        self._bind_stream()
        self.handle.run_eval_async(frames.data_ptr(), gt.data_ptr(), gt.dtype == torch.float64, B, H, W, src_thr, val_thr,
                                   mode, depth.data_ptr(), dt.data_ptr(), None, mask.data_ptr(), counts.data_ptr())
        self._hold(frames, gt, depth, dt, mask, counts)
        return dict(depth=depth, dt=dt, mask=mask, lbl=None, counts=counts)

    def eval_totals(self, totals=None):
        """Running totals [mse, rmse, mae, irmse, imae, d1, d2, d3, valid px, frames] of the fill_eval() calls since the
        last collection, as a float64 CUDA tensor (added to ``totals`` if given); enqueued on torch's current stream."""
        torch = self.torch
        acc = totals is not None
        if totals is None:
            totals = torch.empty((_lib.METRIC_COLS + 1,), dtype=torch.float64, device=torch.device("cuda", self.device))
        self._bind_stream()
        self.handle.eval_totals(totals.data_ptr(), accumulate=acc)
        self._inflight = {}
        return totals

    def fill_png(self, png, crop_top: int = 96, src_thr: float = 0.1, val_thr: float = 0.1, want_lidar: bool = True,
                 want_lbl: bool = False):
        """png: uint16 CUDA tensor [B,H_in,W] of KITTI depth PNG samples (depth = sample / 256, data_read.py:215);
        rows [crop_top, H_in) are processed (train.py:211).  Decode and crop happen inside the first kernel.  Returns
        the dict of fill() plus ``lidar`` (the decoded float32 frames) when asked for; enqueued only."""
        torch = self.torch
        assert png.is_cuda and png.dtype == torch.uint16 and png.is_contiguous() and png.dim() == 3
        B, Hin, W = png.shape
        H = Hin - int(crop_top)
        assert 0 <= crop_top < Hin
        dev = png.device
        f32 = lambda: torch.empty((B, H, W), dtype=torch.float32, device=dev)       # noqa: E731
        lidar = f32() if want_lidar else None
        depth, dt = f32(), f32()
        mask = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        lbl = torch.empty((B, H, W), dtype=torch.int32, device=dev) if want_lbl else None
        counts = torch.empty((B, 2), dtype=torch.int32, device=dev)
        self._bind_stream()
        self.handle.run_device_u16_async(png.data_ptr(), B, Hin, W, int(crop_top), src_thr, val_thr, depth.data_ptr(),
                                         lidar.data_ptr() if lidar is not None else None, dt.data_ptr(),
                                         lbl.data_ptr() if lbl is not None else None, mask.data_ptr(), counts.data_ptr())
        self._hold(png, lidar, depth, dt, mask, lbl, counts)
        return dict(lidar=lidar, depth=depth, dt=dt, mask=mask, lbl=lbl, counts=counts)

    def decode_png(self, data_u8, offsets_i64, H: int, W: int):
        """16-bit grayscale PNG files on the device: data_u8 uint8 CUDA tensor of the files back to back, offsets_i64
        int64 CUDA tensor [B+1] (file b = data_u8[offsets[b]:offsets[b+1]]) -> (samples uint16 [B,H,W], status int32 [B]:
        0 ok, else the code of include/dtfill.h dtfill_png_decode, named by _lib.PNG_STATUS; a failed frame's samples are
        zero), enqueued on torch's current stream.  The samples are what fill_png() takes."""
        torch = self.torch
        assert data_u8.is_cuda and data_u8.dtype == torch.uint8 and data_u8.is_contiguous()
        assert offsets_i64.is_cuda and offsets_i64.dtype == torch.int64 and offsets_i64.is_contiguous()
        B = offsets_i64.numel() - 1
        assert B >= 1
        dev = data_u8.device
        samples = torch.empty((B, H, W), dtype=torch.uint16, device=dev)
        status = torch.empty((B,), dtype=torch.int32, device=dev)
        self._bind_stream()
        self.handle.png_decode_device_async(data_u8.data_ptr(), offsets_i64.data_ptr(), B, H, W, samples.data_ptr(),
                                            status.data_ptr())
        self._hold(data_u8, offsets_i64, samples, status)
        return samples, status

    def encode_png(self, t):
        """t: uint16 samples or float32 depth in metres, CUDA tensor [B,H,W] -> (data uint8 CUDA tensor [B * bound],
        offsets int64 CUDA tensor [B+1]): B 16-bit grayscale PNG files back to back, file b = data[offsets[b]:
        offsets[b+1]] (the layout decode_png takes), enqueued on torch's current stream.  Depth becomes
        sample = clip(nan_to_num(fl32(d * 256), nan=0, posinf=65535), 0, 65535) truncated toward zero.  In pipelined
        mode the fills in flight are joined into the stream first (no host synchronisation), so the output of fill() /
        fill_png() can be passed straight in."""
        torch = self.torch
        assert t.is_cuda and t.dtype in (torch.uint16, torch.float32) and t.is_contiguous() and t.dim() == 3
        B, H, W = t.shape
        bound = _lib.png_encode_bound(H, W)
        data = torch.empty((B * bound,), dtype=torch.uint8, device=t.device)
        offsets = torch.empty((B + 1,), dtype=torch.int64, device=t.device)
        self._bind_stream()
        if self.pipeline_depth > 1:
            self.handle.flush()
        self.handle.png_encode_device_async(t.data_ptr(), t.dtype == torch.float32, B, H, W, data.data_ptr(), B * bound,
                                            offsets.data_ptr())
        self._hold(t, data, offsets)
        return data, offsets

    def eval_sampled(self, gt, rows, cols, offsets=None, crop=None, src_thr: float | None = None, want_lidar: bool = False):
        """The NYU evaluation loop (eval_nyu.evaluate_fill_sampled) against the float32 CUDA tensor gt [B,H,W], used in
        place, on torch's current stream, so that repeated draws against the same resident ground truth move only their
        coordinates.  rows / cols: the host forms evaluate_fill_sampled takes, or int32 CUDA tensors of the concatenated
        coordinates with ``offsets`` an int64 CUDA tensor [B+1] (frame b: entries offsets[b]:offsets[b+1]; checked on the
        device, a coordinate outside the frame raises ValueError).  Synchronous: returns (per_frame [B,9], sums [10]) float64
        numpy arrays (and the sparse frames gt * Mask with want_lidar).  Fills still in flight are joined first."""
        from . import eval_nyu
        torch = self.torch
        assert gt.is_cuda and gt.dtype == torch.float32 and gt.dim() == 3
        gt = eval_nyu._aligned(gt)
        B, H, W = (int(v) for v in gt.shape)
        crop = eval_nyu._check_crop(eval_nyu.NYU_EVAL_CROP if crop is None else crop, H, W)
        src_thr = eval_nyu.NYU_SRC_THR if src_thr is None else src_thr
        on_device = isinstance(rows, torch.Tensor) and rows.is_cuda
        if on_device:
            assert cols.is_cuda and rows.dtype == cols.dtype == torch.int32 and rows.is_contiguous() and cols.is_contiguous()
            assert offsets is not None and offsets.is_cuda and offsets.dtype == torch.int64 and offsets.numel() == B + 1
            assert offsets.is_contiguous()
            if rows.numel() != cols.numel():
                raise ValueError(f"eval_sampled: {rows.numel()} rows but {cols.numel()} cols")
            # the kernel reads rows / cols between offsets[0] and offsets[B], so non-decreasing offsets whose ends lie within
            # the arrays keep every read inside them (a synchronous call: these checks cost two small copies)
            lo, hi = (int(v) for v in offsets[[0, B]].tolist())
            if lo < 0 or hi > rows.numel():
                raise ValueError(f"eval_sampled: offsets span [{lo}, {hi}) but there are {rows.numel()} coordinates")
            dec = torch.nonzero(offsets[1:] < offsets[:-1])
            if dec.numel():
                raise ValueError(f"eval_sampled: frame {int(dec[0, 0])} has a negative sample count")
            r, c, off = rows.data_ptr(), cols.data_ptr(), offsets.data_ptr()
        else:
            r, c, off = eval_nyu._sample_arrays(rows, cols, B, H, W)
        from .tools import VALID_THR
        self._bind_stream()
        res = self.handle.eval_sampled(gt.data_ptr(), B, H, W, r, c, off, crop, src_thr, VALID_THR, gt_is_device=True,
                                       coords_are_device=on_device, want_lidar=want_lidar)
        self._inflight = {}       # the call synchronised: every earlier call has finished
        return res

    def flush(self):
        """Pipelined mode: torch's current stream waits for every fill still in flight."""
        self._bind_stream()
        self.handle.flush()
        self._inflight = {}       # torch's current stream now follows every call: ordinary stream-ordered reuse is safe

    def status(self):
        """Synchronise; (first_bad_frame or -1, kernel launches of the last fill)."""
        r = self.handle.status()
        self._inflight = {}
        return r

    def metrics(self, pred, gt, mode: int = _lib.METRICS_KITTI, totals=None):
        """pred float32 [B,H,W], gt float32/float64 [B,H,W] CUDA tensors -> (per_frame [B,9], sums [10]) CUDA f64.
        totals: float64 CUDA tensor [10] of running totals; this batch's sums are ADDED to it on the device
        (eval.py:212-232) and it is returned in place of sums."""
        torch = self.torch
        assert pred.is_cuda and gt.is_cuda and pred.is_contiguous() and gt.is_contiguous() and pred.shape == gt.shape
        assert pred.dtype == torch.float32 and gt.dtype in (torch.float32, torch.float64)
        B = pred.shape[0]
        n = pred[0].numel()
        per_frame = torch.empty((B, _lib.METRIC_COLS), dtype=torch.float64, device=pred.device)
        sums = totals if totals is not None else torch.empty((_lib.METRIC_COLS + 1,), dtype=torch.float64, device=pred.device)
        self._bind_stream()
        self.handle.metrics(pred.data_ptr(), gt.data_ptr(), B, 1, n, mode, gt.dtype == torch.float64, on_device=True,
                            per_frame_ptr=per_frame.data_ptr(), sums_ptr=sums.data_ptr(), accumulate=totals is not None)
        return per_frame, sums
