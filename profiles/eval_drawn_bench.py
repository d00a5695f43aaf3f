"""The NYU evaluation loop with its draws made on the GPU (evaluate_fill_drawn, dtfill_eval_sampled_mt) against drawing
them on the host first, as a user of evaluate_fill_sampled does today.

    python profiles/eval_drawn_bench.py [--draws 16] [--out results.json]

Workload, generated from seeds (that of eval_sampled_bench.py): 654 frames of synth.nyu_frame(s, 240, 320,
return_dense=True) ground truth, float32, resident on the device; for every sample count n in {20, 50, 200, 500} `--draws`
draws, draw d from np.random.RandomState(100000 n + d) in both ways.  Host wall clock around whole draws, the drawing
included, after a warm-up draw.  Prints one JSON document:

  drawn             (i) evaluate_fill_drawn(gt_tensor, n, rng): frames/s, seconds per draw, link bytes of one draw
  host_drawn        (ii) 654 x nyu_sample_coords(n, rng) followed by evaluate_fill_sampled(gt_tensor, rows, cols)
  device_ms         device time per draw of (i), per kernel and for the copies, k11_mt_draw's share (torch.profiler, a run
                    of its own, 3 draws)
  checked_frames    rows of (i) and (ii) compared with == (NaN equal to NaN) on every draw; mismatched_frames counts the
                    failures, and `state_mismatches` the draws after which the two generators' states differ
  gpu               card name, power limit and max SM clock, read in the same run
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from distancetransform_depthcompletion_b200 import _lib, eval_nyu, synth  # noqa: E402
from png_bench import gpu_info  # noqa: E402

B, H, W = 654, 240, 320
NS = (20, 50, 200, 500)


def _rng(n, d):
    return np.random.RandomState(100_000 * n + d)


def _host_drawn(gt_t, n, rs):
    coords = [eval_nyu.nyu_sample_coords(n, H, W, rng=rs) for _ in range(B)]
    return eval_nyu.evaluate_fill_sampled(gt_t, [c[0] for c in coords], [c[1] for c in coords])


def _same_rows(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


def _same_state(a, b):
    sa, sb = a.get_state(legacy=False)["state"], b.get_state(legacy=False)["state"]
    return np.array_equal(sa["key"], sb["key"]) and sa["pos"] == sb["pos"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_drawn_bench: no CUDA device (the numbers here are GPU times)")
    torch.cuda.init()
    gt = np.ascontiguousarray(np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(B)]))
    gt_t = torch.from_numpy(gt).cuda()
    h = _lib.get_handle()
    res = {"gpu": gpu_info(), "frames": B, "size": [H, W], "crop": list(eval_nyu.NYU_EVAL_CROP), "draws_per_n": args.draws,
           "drawn": {}, "host_drawn": {}, "device_ms": {}}
    checked = mismatched = state_mismatches = 0
    for n in NS:
        key = f"n{n}"
        rows_of = {}
        rngs = {}
        for name in ("drawn", "host_drawn"):
            run = ((lambda rs: eval_nyu.evaluate_fill_drawn(gt_t, n, rng=rs)) if name == "drawn" else
                   (lambda rs: _host_drawn(gt_t, n, rs)))
            run(_rng(n, 0))                                   # warm-up
            rs = [_rng(n, d) for d in range(1, args.draws + 1)]
            t = time.perf_counter()
            for d in range(args.draws):
                rows_of[(name, d)] = run(rs[d])[0]
            dt = time.perf_counter() - t
            rngs[name] = rs
            h2d, d2h = h.transfer_bytes()
            res[name][key] = {"frames_per_s": round(args.draws * B / dt), "draw_ms": round(1e3 * dt / args.draws, 3),
                              "h2d_bytes_per_draw": h2d, "d2h_bytes_per_draw": d2h}
        for d in range(args.draws):
            ok = _same_rows(rows_of[("drawn", d)], rows_of[("host_drawn", d)]).all(axis=1)
            mismatched += int((~ok).sum())
            checked += B
            state_mismatches += int(not _same_state(rngs["drawn"][d], rngs["host_drawn"][d]))
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for d in range(1, 4):
                eval_nyu.evaluate_fill_drawn(gt_t, n, rng=_rng(n, d))
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            k = ev.key
            if ev.device_time_total <= 0:
                continue
            name = ("copies" if ("Memcpy" in k or "Memset" in k) else
                    next((s for s in ("k11_mt_draw", "k10_sample_bits", "k1_mask_rows_v16", "k1_mask_rows", "k1b_scan_compact",
                                      "k2_chamfer_wide", "k2_chamfer", "k3_sky", "k4x_compact", "k4x_reduce", "k4x_sums")
                          if s in k), k[:60]))
            split[name] = split.get(name, 0.0) + ev.device_time_total / 1e3 / 3
        split["total"] = sum(split.values())
        split["k11_share"] = split.get("k11_mt_draw", 0.0) / split["total"]
        res["device_ms"][key] = {k: round(v, 4) for k, v in split.items()}
        print(key, res["drawn"][key], res["host_drawn"][key], res["device_ms"][key], file=sys.stderr, flush=True)
    res["checked_frames"] = checked
    res["mismatched_frames"] = mismatched
    res["state_mismatches"] = state_mismatches
    res["note"] = ("frames/s are host wall clock around whole draws (the drawing included) over all draws of an n after a "
                   "warm-up draw, ground truth resident; device_ms sums kernel and copy activity per draw of (i) "
                   "(torch.profiler, a separate run of 3 draws)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0 if mismatched == 0 and state_mismatches == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
