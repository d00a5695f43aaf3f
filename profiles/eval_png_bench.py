"""The KITTI ablation notebook's evaluation loop from the PNG files (dtfill_eval_png) against the ways to run it without.

    python profiles/eval_png_bench.py [--frames 32] [--reps 5] [--out results.json]

Workload, generated from seeds: LiDAR rint(synth.kitti_frame(s) * 256) as uint16 352 x 1216 with 64 and 16 beams,
ground truth rint(synth.kitti_gt(s) * 256), each encoded with tests/png_oracle.encode (libpng's filter choice, zlib level
6).  `--frames` distinct pairs per beam count are tiled to B = 256 and 1000 (the size of KITTI's val_selection_cropped).
Prints one JSON document:

  files             mean bytes of a LiDAR file (64 and 16 beams) and of a ground-truth file
  eval_png          per beam count and B: end-to-end frames/s of evaluation.evaluate_fill_png_files' call (file bytes
                    in host memory -> per-frame metrics and sums on the host; best and median of --reps after a warm-up),
                    the bytes it moved over the link in each direction, and the device time of one call split into
                    decode (k8_png_*), fill (k1*, k2*, k3*), metrics (k4x_*) and copies (torch.profiler, its own run)
  composed          baseline (a), the same loop from today's calls: read_depth_pngs x 2 -> float32 / float64 on the host
                    -> dt_fill_batch -> evaluate_batch, with the bytes those calls move (computed from the shapes and
                    from dtfill_transfer_bytes)
  host_pool         baseline (b), the reference's own way on every host core: PIL decode, the cv2 port of
                    Distance_Transform (eval_NYU.py:120-133), oracle.result_kitti (numpy), one process per core
  checked_frames    frames whose rows were compared: every frame of every timed batch against (a) with ==, and against
                    (b) (metrics and count); mismatched_frames counts the failures
  gpu               card name, power limit and max SM clock, read in the same run
"""
from __future__ import annotations

import argparse
import io
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import png_oracle as P  # noqa: E402
from distancetransform_depthcompletion_b200 import _lib, data_read, evaluation, synth, tools  # noqa: E402
from png_bench import gpu_info  # noqa: E402

H, W = synth.KITTI_H, synth.KITTI_W
NPX = H * W


def _pil(png: bytes) -> np.ndarray:
    from PIL import Image
    return np.array(Image.open(io.BytesIO(png)))


def _host_rows(pairs):
    """Baseline (b) for a chunk of (lidar file, gt file): the notebook's loop body on the CPU."""
    from oracle import oracle as O
    rows = []
    for lf, gf in pairs:
        lidar = _pil(lf).astype(np.float32) / 256                   # data_read.py:215
        gt = _pil(gf) / 256.                                         # data_read.py:223
        pred = O.cv2_port_fill_frame(lidar, 0.1, 0.1, nyu_style=True)[0]
        m = O.result_kitti(pred, gt)
        rows.append([m["mse"], m["rmse"], m["mae"], m["irmse"], m["imae"], 0, 0, 0, m["count"]])
    return rows


def _best(fn, reps, warm=True):
    if warm:
        fn()
    ts, r = [], None
    for _ in range(reps):
        t = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t)
    return min(ts), float(np.median(ts)), r


def _same_rows(a, b):
    return (np.asarray(a) == np.asarray(b)) | (np.isnan(a) & np.isnan(b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_png_bench: no CUDA device (the numbers here are GPU times)")
    torch.cuda.init()

    t0 = time.time()
    n = args.frames
    gts = [np.rint(synth.kitti_gt(10_000 + s) * 256).astype(np.uint16) for s in range(n)]
    gfiles = [P.encode(x) for x in gts]
    lfiles = {beams: [P.encode(np.rint(synth.kitti_frame(s, beam_step=64 // beams) * 256).astype(np.uint16))
                      for s in range(n)] for beams in (64, 16)}
    res = {"gpu": gpu_info(), "encode_s": round(time.time() - t0, 1),
           "files": {"lidar64_mean_bytes": round(float(np.mean([len(f) for f in lfiles[64]]))),
                     "lidar16_mean_bytes": round(float(np.mean([len(f) for f in lfiles[16]]))),
                     "gt_mean_bytes": round(float(np.mean([len(f) for f in gfiles])))},
           "eval_png": {}, "composed": {}, "host_pool": {}}
    h = _lib.get_handle()
    ncpu = len(os.sched_getaffinity(0))
    res["host_cores"] = ncpu
    checked, mismatched = 0, 0
    pool = ProcessPoolExecutor(ncpu)
    try:
        for beams in (64, 16):
            for B in (256, 1000):
                key = f"kitti{beams}_B{B}"
                lf = [lfiles[beams][b % n] for b in range(B)]
                gf = [gfiles[(b // n + 3 * b + 1) % n] for b in range(B)]
                # the call
                e_min, e_med, (pf, sums) = _best(lambda: evaluation.evaluate_fill_png_files(lf, gf), args.reps)
                h2d, d2h = h.transfer_bytes()
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    for _ in range(3):
                        evaluation.evaluate_fill_png_files(lf, gf)
                    torch.cuda.synchronize()
                split = {"decode": 0.0, "fill": 0.0, "metrics": 0.0, "copies": 0.0}
                for ev in prof.key_averages():
                    k = ev.key
                    part = ("decode" if "k8_png" in k else "metrics" if "k4x_" in k else
                            "copies" if ("Memcpy" in k or "Memset" in k) else "fill")
                    split[part] += ev.device_time_total / 1e3 / 3
                res["eval_png"][key] = {
                    "frames_per_s": round(B / e_min), "call_s_best": round(e_min, 4), "call_s_median": round(e_med, 4),
                    "h2d_bytes": h2d, "d2h_bytes": d2h,
                    "device_ms": {k: round(v, 3) for k, v in split.items()},
                }
                # baseline (a): today's calls
                def composed():
                    lid = data_read.read_depth_pngs(lf).astype(np.float32) / 256
                    gt = data_read.read_depth_pngs(gf) / 256.
                    r = tools.dt_fill_batch(lid)
                    fill_bytes = h.transfer_bytes()
                    return evaluation.evaluate_batch(r["depth"], gt, _lib.METRICS_KITTI), fill_bytes
                c_min, c_med, ((pf_a, sums_a), (fh2d, fd2h)) = _best(composed, max(args.reps // 2, 2))
                files_bytes = sum(len(f) for f in lf) + sum(len(f) for f in gf)
                res["composed"][key] = {
                    "frames_per_s": round(B / c_min), "call_s_best": round(c_min, 4), "call_s_median": round(c_med, 4),
                    "h2d_bytes": files_bytes + fh2d + B * NPX * (4 + 8),
                    "d2h_bytes": 2 * B * NPX * 2 + fd2h + B * 72 + 80,
                }
                ok = _same_rows(pf, pf_a).all(axis=1)
                mismatched += int((~ok).sum()) + int(not _same_rows(sums, sums_a).all())
                checked += B
                # baseline (b): PIL + cv2 port + numpy metrics on every host core
                chunks = [list(zip(lf[i::ncpu], gf[i::ncpu])) for i in range(ncpu)]

                def host():
                    parts = list(pool.map(_host_rows, chunks))
                    out = np.empty((B, 9))
                    for i in range(ncpu):
                        if parts[i]:
                            out[i::ncpu] = np.asarray(parts[i])
                    return out
                h_min, h_med, pf_b = _best(host, 1 if B > 256 else 2, warm=B <= 256)    # B = 256 warms the workers
                res["host_pool"][key] = {"frames_per_s": round(B / h_min, 1), "call_s_best": round(h_min, 3),
                                         "call_s_median": round(h_med, 3)}
                okb = _same_rows(pf, pf_b).all(axis=1)
                mismatched += int((~okb).sum())
                checked += B
                print(key, res["eval_png"][key], file=sys.stderr, flush=True)
    finally:
        pool.shutdown()
    res["checked_frames"] = checked
    res["mismatched_frames"] = mismatched
    res["note"] = ("end-to-end times are host wall clock around synchronous calls, best of the repetitions after a "
                   "warm-up; every call uploads its files afresh.  device_ms sums kernel and copy activity per call "
                   "(torch.profiler, a separate run of 3 calls)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0 if mismatched == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
