"""The NYU evaluation loop from dense ground truth (dtfill_eval_sampled) against the ways to run it without.

    python profiles/eval_sampled_bench.py [--draws 16] [--host-draws 2] [--out results.json]

Workload, generated from seeds: 654 frames (NYU's test split) of synth.nyu_frame(s, 240, 320, return_dense=True) ground
truth, float32; for every sample count n in {20, 50, 200, 500} (eval_NYU.py's line_num) `--draws` draws of the reference's
sampler (eval_nyu.nyu_sample_coords, one RandomState per draw) against that same ground truth.  Prints one JSON document:

  resident          (i) eval_nyu.evaluate_fill_sampled on a CUDA tensor of the ground truth: frames/s over all draws of
                    an n (host wall clock around the synchronous calls, after a warm-up draw), link bytes of one draw
  host_gt           (ii) the same call on the numpy ground truth (uploaded by every call)
  composed          (iii) today's calls: the sample in numpy (gt * Mask), tools.dt_fill_batch (source threshold 0.001),
                    the crop on the host, evaluation.evaluate_batch in NYU mode; link bytes from dtfill_transfer_bytes and
                    the shapes
  host_pool         (iv) the reference's own way on every host core: gt * Mask, the cv2 port of Distance_Transform
                    (eval_NYU.py:120-133), oracle.result_nyu, one process per core (`--host-draws` draws per n)
  device_ms         device time of one resident draw per kernel and for the copies (torch.profiler, its own run)
  checked_frames    rows compared with ==: (i), (ii) and (iii) on every draw of (iii), (iv) on its draws (metrics and
                    count); mismatched_frames counts the failures
  gpu               card name, power limit and max SM clock, read in the same run
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from distancetransform_depthcompletion_b200 import _lib, eval_nyu, evaluation, synth, tools  # noqa: E402
from png_bench import gpu_info  # noqa: E402

B, H, W = 654, 240, 320
NS = (20, 50, 200, 500)
R0, R1, C0, C1 = eval_nyu.NYU_EVAL_CROP


def _draw(n, d):
    rs = np.random.RandomState(100_000 * n + d)
    coords = [eval_nyu.nyu_sample_coords(n, H, W, rng=rs) for _ in range(B)]
    return [c[0] for c in coords], [c[1] for c in coords]


def _sparse(gt, rows, cols):
    mask = np.zeros(gt.shape, np.float32)
    for b in range(len(gt)):
        mask[b, rows[b], cols[b]] = 1
    return gt * mask


def _host_rows(args):
    """Baseline (iv) for a chunk of frames: the loop body of eval_NYU.py on the CPU."""
    from oracle import oracle as O
    gt, rows, cols = args
    out = []
    for b in range(len(gt)):
        lidar = _sparse(gt[b:b + 1], rows[b:b + 1], cols[b:b + 1])[0]
        pred = O.cv2_port_fill_frame(lidar, 0.001, 0.1, nyu_style=True)[0]
        m = O.result_nyu(pred[R0:R1, C0:C1], gt[b, R0:R1, C0:C1])
        out.append([m[k] for k in ("mse", "rmse", "mae", "irmse", "imae", "delta1", "delta2", "delta3", "count")])
    return out


def _same_rows(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return (a == b) | (np.isnan(a) & np.isnan(b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, default=16)
    ap.add_argument("--host-draws", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_sampled_bench: no CUDA device (the numbers here are GPU times)")
    torch.cuda.init()
    gt = np.ascontiguousarray(np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(B)]))
    gt_t = torch.from_numpy(gt).cuda()
    draws = {n: [_draw(n, d) for d in range(args.draws + 1)] for n in NS}        # draw 0 warms up
    h = _lib.get_handle()
    ncpu = len(os.sched_getaffinity(0))
    res = {"gpu": gpu_info(), "host_cores": ncpu, "frames": B, "size": [H, W], "crop": list(eval_nyu.NYU_EVAL_CROP),
           "draws_per_n": args.draws, "gt_bytes": int(gt.nbytes),
           "resident": {}, "host_gt": {}, "composed": {}, "host_pool": {}, "device_ms": {}}
    checked = mismatched = 0
    pool = ProcessPoolExecutor(ncpu)
    try:
        for n in NS:
            key = f"n{n}"
            rows_of = {}
            for name, g in (("resident", gt_t), ("host_gt", gt)):
                evaluate = eval_nyu.evaluate_fill_sampled
                evaluate(g, *draws[n][0])
                t = time.perf_counter()
                for d in range(1, args.draws + 1):
                    rows_of[(name, d)] = evaluate(g, *draws[n][d])[0]
                dt = time.perf_counter() - t
                h2d, d2h = h.transfer_bytes()
                res[name][key] = {"frames_per_s": round(args.draws * B / dt), "draw_s": round(dt / args.draws, 5),
                                  "h2d_bytes_per_draw": h2d, "d2h_bytes_per_draw": d2h}
            # (iii) today's calls
            t = time.perf_counter()
            comp_bytes = [0, 0]
            for d in range(1, args.draws + 1):
                rows, cols = draws[n][d]
                r = tools.dt_fill_batch(_sparse(gt, rows, cols), src_thr=eval_nyu.NYU_SRC_THR)
                fh2d, fd2h = h.transfer_bytes()
                pred_c = np.ascontiguousarray(r["depth"][:, R0:R1, C0:C1])
                gt_c = np.ascontiguousarray(gt[:, R0:R1, C0:C1])
                pf_c, _ = evaluation.evaluate_batch(pred_c, gt_c, _lib.METRICS_NYU)
                comp_bytes = [fh2d + pred_c.nbytes + gt_c.nbytes, fd2h + B * 72 + 80]
                for name in ("resident", "host_gt"):
                    ok = _same_rows(rows_of[(name, d)], pf_c).all(axis=1)
                    mismatched += int((~ok).sum())
                    checked += B
            dt = time.perf_counter() - t
            res["composed"][key] = {"frames_per_s": round(args.draws * B / dt), "draw_s": round(dt / args.draws, 4),
                                    "h2d_bytes_per_draw": comp_bytes[0], "d2h_bytes_per_draw": comp_bytes[1]}
            # (iv) the cv2 port + numpy metrics on every host core
            t = time.perf_counter()
            for d in range(1, args.host_draws + 1):
                rows, cols = draws[n][d]
                chunks = [(gt[i::ncpu], rows[i::ncpu], cols[i::ncpu]) for i in range(ncpu)]
                parts = list(pool.map(_host_rows, chunks))
                out = np.empty((B, 9))
                for i in range(ncpu):
                    if parts[i]:
                        out[i::ncpu] = np.asarray(parts[i])
                ok = _same_rows(rows_of[("resident", d)], out).all(axis=1)
                mismatched += int((~ok).sum())
                checked += B
            dt = time.perf_counter() - t
            res["host_pool"][key] = {"frames_per_s": round(args.host_draws * B / dt, 1),
                                     "draw_s": round(dt / args.host_draws, 3)}
            # device time of one resident draw, per kernel
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for d in range(1, 4):
                    eval_nyu.evaluate_fill_sampled(gt_t, *draws[n][d])
                torch.cuda.synchronize()
            split = {}
            for ev in prof.key_averages():
                k = ev.key
                if ev.device_time_total <= 0:
                    continue
                name = ("copies" if ("Memcpy" in k or "Memset" in k) else
                        next((s for s in ("k10_sample_bits", "k1_mask_rows_v16", "k1_mask_rows", "k1b_scan_compact",
                                          "k2_chamfer_wide", "k2_chamfer", "k3_sky", "k4x_compact", "k4x_reduce", "k4x_sums")
                              if s in k), k[:60]))
                split[name] = split.get(name, 0.0) + ev.device_time_total / 1e3 / 3
            split["total"] = sum(split.values())
            res["device_ms"][key] = {k: round(v, 4) for k, v in split.items()}
            print(key, res["resident"][key], res["host_gt"][key], res["composed"][key], res["host_pool"][key],
                  file=sys.stderr, flush=True)
    finally:
        pool.shutdown()
    res["checked_frames"] = checked
    res["mismatched_frames"] = mismatched
    res["note"] = ("frames/s are host wall clock around synchronous calls over all draws of an n after a warm-up draw; "
                   "the ground truth (200 MB) exceeds the 126 MB L2, so every draw reads it from HBM.  device_ms sums "
                   "kernel and copy activity per draw (torch.profiler, a separate run of 3 draws)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0 if mismatched == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
