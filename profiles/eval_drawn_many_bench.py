"""Many NYU draws in one call (evaluate_fill_drawn_many, dtfill_eval_sampled_mt_many) against one call per draw
(evaluate_fill_drawn).

    python profiles/eval_drawn_many_bench.py [--draws 16] [--reps 5] [--out results.json]

Workload, that of eval_drawn_bench.py: 654 frames of synth.nyu_frame(s, 240, 320, return_dense=True) ground truth, float32,
resident on the device; for every sample count n in {20, 50, 200, 500} `--draws` draws, draw d from
np.random.RandomState(100000 n + d).  The whole n x draw grid is run three ways, each timed with the host wall clock around
its synchronous calls after a warm-up of all three; the three alternate `--reps` times and the median is reported:

  grid              (i) one evaluate_fill_drawn_many call for the whole grid (n given per draw)
  per_n             (ii) one evaluate_fill_drawn_many call per n
  per_draw          (iii) one evaluate_fill_drawn call per draw
  link_bytes        host<->device bytes of (i), and of the four calls of (ii) together
  device_ms         device time per kernel and for the copies, summed over the grid, of (i) and of (iii) (torch.profiler,
                    a run of its own)
  checked_rows      rows of (i) and (ii) compared with (iii) using == (NaN equal to NaN) on every repetition;
                    mismatched_rows counts the failures, state_mismatches the generators whose final states differ
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
KERNELS = ("k11_mt_draw_many", "k11_mt_draw", "k10_sample_bits", "k1_mask_rows_v16", "k1_mask_rows", "k1b_scan_compact",
           "k2_chamfer_wide", "k2_chamfer", "k3_sky", "k4x_compact", "k4x_reduce", "k4x_sums")


def _grid(draws):
    """(n, seed) of every draw of the grid, n-major."""
    return [(n, 100_000 * n + d) for n in NS for d in range(draws)]


def _run_grid(gt_t, grid):
    rngs = [np.random.RandomState(s) for _, s in grid]
    pf, _ = eval_nyu.evaluate_fill_drawn_many(gt_t, [n for n, _ in grid], rngs)
    return pf, rngs


def _run_per_n(gt_t, grid):
    rngs = [np.random.RandomState(s) for _, s in grid]
    pf = []
    for n in NS:
        idx = [i for i, (m, _) in enumerate(grid) if m == n]
        pf.append(eval_nyu.evaluate_fill_drawn_many(gt_t, n, [rngs[i] for i in idx])[0])
    return np.concatenate(pf), rngs


def _run_per_draw(gt_t, grid):
    rngs = [np.random.RandomState(s) for _, s in grid]
    pf = [eval_nyu.evaluate_fill_drawn(gt_t, n, rng=r)[0] for (n, _), r in zip(grid, rngs)]
    return np.stack(pf), rngs


def _same_rows(a, b):
    return ((a == b) | (np.isnan(a) & np.isnan(b))).all(axis=-1)


def _same_state(a, b):
    sa, sb = a.get_state(legacy=False)["state"], b.get_state(legacy=False)["state"]
    return np.array_equal(sa["key"], sb["key"]) and sa["pos"] == sb["pos"]


def _device_ms(torch, fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        k = ev.key
        if ev.device_time_total <= 0:
            continue
        name = "copies" if ("Memcpy" in k or "Memset" in k) else next((s for s in KERNELS if s in k), k[:60])
        split[name] = split.get(name, 0.0) + ev.device_time_total / 1e3
    split["total"] = sum(split.values())
    return {k: round(v, 3) for k, v in split.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_drawn_many_bench: no CUDA device (the numbers here are GPU times)")
    torch.cuda.init()
    gt = np.ascontiguousarray(np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(B)]))
    gt_t = torch.from_numpy(gt).cuda()
    h = _lib.get_handle()
    grid = _grid(args.draws)
    D = len(grid)
    runs = {"grid": _run_grid, "per_n": _run_per_n, "per_draw": _run_per_draw}
    for fn in runs.values():                                  # warm-up
        fn(gt_t, grid)
    times = {k: [] for k in runs}
    checked = mismatched = state_mismatches = 0
    link = {}
    for _ in range(args.reps):
        out = {}
        for name, fn in runs.items():
            torch.cuda.synchronize()
            t = time.perf_counter()
            out[name] = fn(gt_t, grid)
            times[name].append(time.perf_counter() - t)
            if name == "grid":
                link["grid"] = h.transfer_bytes()
        ref_pf, ref_rngs = out["per_draw"]
        for name in ("grid", "per_n"):
            pf, rngs = out[name]
            ok = _same_rows(pf, ref_pf)
            checked += ok.size
            mismatched += int((~ok).sum())
            state_mismatches += sum(not _same_state(a, b) for a, b in zip(rngs, ref_rngs))
    # link bytes of (ii): the four calls together
    up = down = 0
    rngs = [np.random.RandomState(s) for _, s in grid]
    for n in NS:
        eval_nyu.evaluate_fill_drawn_many(gt_t, n, [r for (m, _), r in zip(grid, rngs) if m == n])
        a, b = h.transfer_bytes()
        up, down = up + a, down + b
    link["per_n"] = (up, down)
    res = {"gpu": gpu_info(), "frames": B, "size": [H, W], "crop": list(eval_nyu.NYU_EVAL_CROP), "ns": list(NS),
           "draws_per_n": args.draws, "draws": D, "reps": args.reps}
    for name in runs:
        t = float(np.median(times[name]))
        res[name] = {"s": round(t, 4), "ms_per_draw": round(1e3 * t / D, 3), "frames_per_s": round(D * B / t),
                     "spread_s": [round(min(times[name]), 4), round(max(times[name]), 4)]}
    res["speedup_grid_vs_per_draw"] = round(res["per_draw"]["s"] / res["grid"]["s"], 3)
    res["speedup_per_n_vs_per_draw"] = round(res["per_draw"]["s"] / res["per_n"]["s"], 3)
    res["link_bytes"] = {k: {"h2d": int(v[0]), "d2h": int(v[1])} for k, v in link.items()}
    res["device_ms"] = {"grid": _device_ms(torch, lambda: _run_grid(gt_t, grid)),
                        "per_draw": _device_ms(torch, lambda: _run_per_draw(gt_t, grid))}
    res["checked_rows"] = checked
    res["mismatched_rows"] = mismatched
    res["state_mismatches"] = state_mismatches
    res["note"] = ("seconds are the median over reps of the host wall clock around the whole grid's synchronous calls "
                   "(drawing included, ground truth resident, the three ways alternating); device_ms sums kernel and "
                   "copy activity over the whole grid (torch.profiler, a separate run)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0 if mismatched == 0 and state_mismatches == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
