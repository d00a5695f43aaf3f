#!/usr/bin/env python
"""bench.py -- DT + NN-fill throughput on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]                 our CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] the reference's CPU path on host cores
    python bench.py --workload sweep [--gpus N]                         BASELINE.json configs[4] only
    python bench.py --dump-outputs DIR ...                              also save what the last timed step returned

A step = one pass of the hot path over one batch of synthetic KITTI-shaped frames (BASELINE.json configs[1]:
256 frames of 352x1216, 64-beam pattern, ~5 % density; outputs filled depth + distance channel + validity mask).
Weak scaling: every rank processes its own batch of 256 frames per step; `value` = total frames of all ranks /
max-over-ranks device time of exactly K timed steps between two CUDA events.  After the timed region 64 frames of
the timed run's own outputs are compared with the CPU oracle, bit for bit (`parity_checked`).  `e2e` is the drop-in
call `tools.DT_complete_batch(x)` with pageable numpy arrays in and out (tools.py:13-35); `e2e_pinned` is the C ABI
with pinned buffers and all three outputs.
The same line carries `sweep`: BASELINE.json configs[4] (8192 frames sharded over the ranks, fill + per-frame
metrics on the GPU, one NCCL sum all-reduce of the totals inside the timed region; strong scaling).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALG_BYTES_PER_PX = 13          # SURVEY.md 8(d): read input f32 4 + filled depth 4 + dt 4 + mask u8 1
H, W = 352, 1216
METRIC = "DT+NN-fill frames/s @1216x352 (64-beam KITTI-shaped frames, batch 256 per GPU)"
UNIT = "frames/s"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_BYTES = 60_000_000      # --dump-outputs stays below 64 MB


def dump_outputs(path: str, out: dict, B: int, H: int, W: int):
    """What one step returned to its caller (DTFillEngine.fill: depth, dt, mask, counts) as DIR/<name>.npy in float32 or
    float64: depth, dt and mask of a fixed, seeded sample of the batch's frames (11 of 256 KITTI frames fit the budget),
    counts [B,2] of every frame, and frame_index, the sampled frames' positions in the batch."""
    import torch
    n = min(B, DUMP_BYTES // (12 * H * W))
    sel = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    tsel = torch.from_numpy(sel).to(out["depth"].device)
    arrays = {"frame_index": sel.astype(np.float64),
              "depth": out["depth"][tsel].cpu().numpy(),
              "dt": out["dt"][tsel].cpu().numpy(),
              "mask": out["mask"][tsel].cpu().numpy().astype(np.float32),
              "counts": out["counts"].cpu().numpy().astype(np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread every ~2 ms
    (the timed region lasts ~10 ms), nvidia-smi -lms as fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.p = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.reasons, self.max_mhz = [], set(), None

    def _nvml_loop(self, pynvml, handle):
        bits = {}
        for name, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
            v = getattr(pynvml, attr, None) or getattr(pynvml, attr.replace("ClocksEventReason", "ClocksThrottleReason"), None)
            if v is not None:
                bits[name] = v
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop_flag:
            try:
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    r = int(get_reasons(handle))
                    for n, bit in bits.items():
                        if r & bit:
                            self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical GPUs; honour CUDA_VISIBLE_DEVICES when it is a list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.idx
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                phys = int(vis.split(",")[self.idx])
            handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(pynvml, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "how": "NVML polled every ~2 ms"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "how": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------------------
# reference CPU path: the reference's own tools.DT_complete_batch when a checkout is reachable, else the
# line-by-line port with the real cv2 call (oracle/oracle.py), else the C oracle
# ------------------------------------------------------------------------------------------------------------
_CPU_FRAMES = None      # frames shared with the forked workers (no pickling of pixel data)
_REF_TOOLS = None       # the reference's tools module (imported before the fork)


def load_reference_tools():
    """solution_DeepNet/tools.py of a reference checkout: $DTFILL_REFERENCE, baseline/_ref, /root/reference (the build
    container).  The module imports tensorflow without using it on this path and forgets to import cv2 (tools.py:1-9):
    a stub module and the real cv2 are supplied.  Returns (module, where) or (None, why)."""
    import importlib.util
    import types
    try:
        import cv2
    except Exception as e:          # noqa: BLE001
        return None, f"cv2 not importable ({e})"
    for root in (os.environ.get("DTFILL_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if not root:
            continue
        for rel in ("solution_DeepNet/tools.py", "tools.py"):
            p = os.path.join(root, rel)
            if os.path.isfile(p):
                try:
                    if "tensorflow" not in sys.modules:
                        sys.modules["tensorflow"] = types.ModuleType("tensorflow")
                    spec = importlib.util.spec_from_file_location("_reference_tools", p)
                    mod = importlib.util.module_from_spec(spec)
                    spec.loader.exec_module(mod)
                    mod.cv2 = cv2
                    return mod, p
                except Exception as e:      # noqa: BLE001
                    return None, f"{p}: {e}"
    return None, "no reference checkout on this box (it cannot travel: Python source outside the repo)"


def _cpu_worker(args):
    kind, lo, hi = args
    frames = _CPU_FRAMES[lo:hi]
    if kind == "reference":
        import cv2
        cv2.setNumThreads(1)
        out = _REF_TOOLS.DT_complete_batch(frames[:, :, :, None])          # tools.py:13-35, unmodified
        return float(out[0, 0, 0, 0])
    from oracle import oracle as O
    if kind == "cv2":
        import cv2
        cv2.setNumThreads(1)
        acc = 0.0
        for i in range(frames.shape[0]):
            # one cv2 call per frame yields the filled depth (tools.py:19-27), dt (tools.py:10) and the mask
            depth, dt, valid = O.cv2_port_fill_frame(frames[i], 0.1, 0.1)
            acc += float(depth[0, 0]) + float(dt[0, 0]) + float(valid[0, 0])
        return acc
    r = O.dt_fill(frames)
    return float(r["depth"][0, 0, 0])


class CpuReference:
    """The reference's per-frame work (tools.py:7-35: mask, cv2 DT with labels, compaction, gather), frames split evenly
    over a fork()ed process pool with one cv2 thread each (the reference itself loops over the frames on one core)."""

    def __init__(self, frames: np.ndarray):
        global _CPU_FRAMES, _REF_TOOLS
        from oracle import oracle as O
        O.build()
        mod, self.where = load_reference_tools()
        if mod is not None:
            _REF_TOOLS, self.kind = mod, "reference"
        else:
            self.kind = "cv2" if O.have_cv2() else "c_oracle"
        self.cores = os.cpu_count() or 1
        try:
            self.cores = len(os.sched_getaffinity(0))
        except Exception:
            pass
        _CPU_FRAMES = frames
        import multiprocessing as mp
        self.pool = mp.get_context("fork").Pool(self.cores)

    def run(self, n: int) -> float:
        """Process the first n frames; returns seconds."""
        edges = np.linspace(0, n, self.cores + 1).astype(int)
        jobs = [(self.kind, int(a), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a]
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker, jobs)
        return time.perf_counter() - t0

    def close(self):
        self.pool.terminate()

    def describe(self):
        if self.kind == "reference":
            return ("reference", f"the reference's own tools.DT_complete_batch ({self.where}) with cv2 "
                                 f"{__import__('cv2').__version__}, frames split over one process per core")
        if self.kind == "cv2":
            return ("port", "reference lines tools.py:7-35 restated with the real cv2.distanceTransformWithLabels "
                            f"(oracle/oracle.py cv2_port_fill_frame; {self.where}), one process per core")
        return ("port", "C restatement oracle/dtfill_oracle.c (cv2 not importable here), one process per core")


WORKLOADS = {   # name -> (beam_step or None for NYU, H, W, source threshold, default batch)
    "kitti64": (1, 352, 1216, 0.1, 256), "kitti32": (2, 352, 1216, 0.1, 256), "kitti16": (4, 352, 1216, 0.1, 256),
    "kitti8": (8, 352, 1216, 0.1, 256), "nyu": (None, 480, 640, 0.001, 1024),
}


def make_frames(n: int, seed0: int, workload: str = "kitti64") -> np.ndarray:
    from distancetransform_depthcompletion_b200 import synth
    distinct = min(n, 64)
    step = WORKLOADS[workload][0]
    if step is None:
        base = np.stack([synth.nyu_frame(seed0 + i) for i in range(distinct)])
    else:
        base = np.stack([synth.kitti_frame(seed0 + i, beam_step=step) for i in range(distinct)])
    if distinct == n:
        return base
    reps = -(-n // distinct)
    out = np.concatenate([base] * reps)[:n].copy()
    # make repeated frames differ (shift columns) so no two frames of the batch are identical
    for i in range(distinct, n):
        out[i] = np.roll(out[i], (i // distinct) * 7, axis=1)
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    batch = args.batch or 256
    ref = CpuReference(make_frames(batch, 0))
    for _ in range(args.warmup):
        ref.run(min(batch, max(ref.cores, 8)))
    t = 0.0
    for _ in range(args.steps):
        t += ref.run(batch)
    ref.close()
    fps = batch * args.steps / t
    kind, how = ref.describe()
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 keys (integer chamfer) + f32 copy", "data": "synthetic",
        "config": {"workload": f"kitti64: batch of {batch} synthetic KITTI 64-beam frames 352x1216 (~5% density) "
                               "(BASELINE.json configs[1]), the whole batch per step",
                   "outputs": "filled depth (tools.DT_complete_batch); the cv2 call also yields the distance channel",
                   "host_cores": ref.cores},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": ref.cores, "kind": kind,
                         "sample": f"{batch} frames x {args.steps} steps; {how}"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def pin_to_gpu_numa(local_rank: int):
    """Bind this process (and the threads it creates later: the pinned-staging pools) to the CPUs next to its GPU, before
    any pinned host memory is allocated, so that eight ranks do not share one socket's memory.  Returns a description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        phys = local_rank
        if vis and all(t.strip().isdigit() for t in vis.split(",")):
            phys = int(vis.split(",")[local_rank])
        hnd = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = sorted(cpus & allowed)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": f"{cpus[0]}-{cpus[-1]}", "n": len(cpus)}
    except Exception as e:      # noqa: BLE001
        return {"error": str(e)[:80]}
    return {"cpus": "unchanged"}


def run_sweep(args, eng, dev, rank, world, dist, comm, barrier, min_seconds):
    """BASELINE.json configs[4]: 8192 synthetic KITTI frames sharded contiguously over the ranks (sharding.shard_range),
    per batch fill -> per-frame Result.evaluate on the GPU -> running totals, no host synchronisation; one NCCL sum
    all-reduce of the 10 totals (dtfill_allreduce_sums) INSIDE the timed region (eval.py:212-232, evaluation.py:82-123)."""
    import torch
    from distancetransform_depthcompletion_b200 import sharding, synth
    from oracle import oracle as O
    Hs, Ws = 352, 1216
    frames, batch, pool = args.sweep_frames, args.sweep_batch, 32
    begin, end = sharding.shard_range(frames, rank, world)
    xp = torch.from_numpy(np.stack([synth.kitti_frame(i) for i in range(pool)])).to(dev)
    gp = torch.from_numpy(np.stack([synth.kitti_gt(i) for i in range(pool)])).to(dev)

    def make(first, n):      # global frames first..first+n: pool frame (i % pool) rolled by 8 * (i // pool) columns
        idx = torch.arange(first, first + n, device=dev)
        shifts = ((idx // pool) * 8) % Ws
        cols = ((torch.arange(Ws, device=dev)[None, :] - shifts[:, None]) % Ws)[:, None, :].expand(n, Hs, Ws)
        return torch.gather(xp[idx % pool], 2, cols).contiguous(), torch.gather(gp[idx % pool], 2, cols).contiguous()

    batches = []             # this rank's whole shard, resident in HBM before the clock starts
    for f in range(begin, end, batch):
        batches.append(make(f, min(batch, end - f)))
    depth = args.pipeline
    eng.handle.set_pipeline_depth(depth)
    outs = [None] * max(1, depth)
    totals = torch.zeros(10, dtype=torch.float64, device=dev)

    def one_sweep():
        for i, (xb, gb) in enumerate(batches):
            outs[i % len(outs)] = eng.fill_eval(xb, gb, out=outs[i % len(outs)] if outs[i % len(outs)] is not None and
                                                outs[i % len(outs)]["depth"].shape == xb.shape else None)
        eng.eval_totals(totals)                       # joins the calls in flight, writes the rank's totals
        if comm is not None:
            comm.allreduce(eng, totals)               # ncclAllReduce(sum, f64) on the same stream

    for _ in range(2):
        totals.zero_()
        one_sweep()
    bad, _ = eng.status()
    assert bad == -1
    times = []
    total_ms = 0.0
    while total_ms < min_seconds * 1e3 and len(times) < 400:
        totals.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        one_sweep()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        times.append(ms)
        total_ms += ms
    bad, _ = eng.status()
    assert bad == -1, f"sweep: unexpected bad frame {bad}"
    eng.handle.set_pipeline_depth(1)
    means = sharding.finalize_means(totals)
    # spot check on rank 0: the first frames of its shard against the oracle (fill) and evaluation.py's numbers
    checked = 0
    if rank == 0:
        xb, gb = batches[0]
        o = eng.fill(xb[:4])
        pf, _ = eng.metrics(o["depth"], gb[:4])
        ref = O.dt_fill(xb[:4].cpu().numpy())
        assert np.array_equal(o["depth"].cpu().numpy(), ref["depth"]), "sweep: filled depth differs from the oracle"
        for i in range(4):
            m = O.result_kitti(ref["depth"][i], gb[i].cpu().numpy())
            got = pf[i].cpu().numpy()
            for k, name in enumerate(("mse", "rmse", "mae", "irmse", "imae")):
                assert abs(got[k] - m[name]) <= 1e-9 * abs(m[name]), (i, name, got[k], m[name])
        checked = 4
    med = statistics.median(times)
    return {"workload": f"configs[4]: {frames} synthetic KITTI 64-beam frames 352x1216 sharded over {world} GPU(s) "
                        f"(contiguous ranges), batches of {batch}, {depth} batches in flight, fill + Result.evaluate per "
                        "frame on the GPU, one NCCL sum all-reduce of the 10 totals inside the timed region",
            "value": frames / (med * 1e-3), "unit": UNIT, "scaling": "strong", "ms_per_sweep": med, "sweeps_timed": len(times),
            "timed_region_s": total_ms * 1e-3, "frames": means["frames"], "mean_rmse_mm": means["rmse"],
            "mean_mae_mm": means["mae"], "mean_irmse_1_per_km": means["irmse"], "mean_imae_1_per_km": means["imae"],
            "valid_pixels": means["valid_pixels"], "collective": "ncclAllReduce(sum, float64 x 10) via dtfill_allreduce_sums"
            if comm is not None else "none (1 rank)", "metrics_checked": checked}


def run_ours(args, rank, world, local_rank):
    numa = pin_to_gpu_numa(local_rank)
    import torch
    from distancetransform_depthcompletion_b200 import _lib, sharding, tools
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    from oracle import oracle as O

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    os.environ.setdefault("DTFILL_DEVICE", str(local_rank))
    sweep_only = args.workload == "sweep"
    workload = "kitti64" if sweep_only else args.workload
    global H, W
    _, H, W, src_thr, default_batch = WORKLOADS[workload]
    B = args.batch or default_batch
    eng = DTFillEngine(local_rank)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    comm = sharding.MetricsComm(eng.handle, rank, world) if world > 1 else None
    if sweep_only:
        sw = run_sweep(args, eng, dev, rank, world, dist, comm, barrier, args.min_seconds)
        if rank == 0:
            emit({"metric": "DT+NN-fill+metrics frames/s, 8192-frame sweep (BASELINE.json configs[4])",
                              "value": sw["value"], "unit": UNIT, "n_gpus": world, "higher_is_better": True,
                  "scaling": "strong", "data": "synthetic", "config": {"workload": sw["workload"]},
                  "sweep": sw})
        if comm is not None:
            comm.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    frames_np = make_frames(B, 1000 * rank, workload)
    x = torch.from_numpy(frames_np).to(dev)
    if args.band_cap is not None:
        eng.handle.set_band_cap(args.band_cap)
    if args.subbatches is not None:
        eng.handle.set_subbatches(args.subbatches)

    def new_outs(with_lbl=False):
        o = dict(depth=torch.empty((B, H, W), dtype=torch.float32, device=dev),
                 dt=torch.empty((B, H, W), dtype=torch.float32, device=dev),
                 mask=torch.empty((B, H, W), dtype=torch.uint8, device=dev),
                 counts=torch.empty((B, 2), dtype=torch.int32, device=dev))
        if with_lbl:
            o["lbl"] = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        return o

    # one output set per batch in flight: consecutive steps of a pipelined run must not share outputs
    outs = [new_outs() for _ in range(max(2, args.pipeline))]
    no = len(outs)
    K = args.steps

    def timed_steps(depth):
        """Exactly K steps between two events on the launching stream (max over ranks); clocks are sampled over them."""
        eng.handle.set_pipeline_depth(depth)
        for i in range(args.warmup):
            eng.fill(x, src_thr=src_thr, out=outs[i % no])
        bad_, launches_ = eng.status()
        assert bad_ == -1, f"unexpected bad frame {bad_}"
        sampler_ = ClockSampler(local_rank)
        barrier()
        sampler_.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            eng.fill(x, src_thr=src_thr, out=outs[i % no])
        eng.flush()                                   # every step's outputs are complete at e1
        e1.record()
        barrier()
        ms_ = e0.elapsed_time(e1)
        if dist is not None:
            t_ = torch.tensor([ms_], dtype=torch.float64, device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            ms_ = float(t_.item())
        clocks_ = sampler_.stop()
        bad_, _ = eng.status()
        assert bad_ == -1, f"unexpected bad frame {bad_}"
        return ms_, launches_, clocks_

    ms_strict, launches_per_step, clocks_strict = timed_steps(1)
    if args.pipeline > 1:
        ms, launches_per_step, clocks = timed_steps(args.pipeline)
    else:
        ms, clocks = ms_strict, clocks_strict
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs[(K - 1) % no], B, H, W)     # the last timed step wrote this output set
    ms_per_step = ms / K
    value = world * B * K / (ms * 1e-3)
    strict = {"value": world * B * K / (ms_strict * 1e-3), "ms_per_step": ms_strict / K,
              "what": "same K steps with strict stream order between steps (pipeline depth 1, the API default)"}

    # ---- parity at the benchmarked configuration: 64 frames of the timed run's own outputs against the oracle ----
    # (the last timed step wrote output set (K-1) % no; every step has the same input)
    sel = np.unique(np.linspace(0, B - 1, min(B, args.parity_frames)).astype(int))
    want = O.dt_fill(frames_np[sel], src_thr=src_thr)
    last = outs[(K - 1) % no]
    tsel = torch.from_numpy(sel).to(dev)
    ok = all(np.array_equal(last[k][tsel].cpu().numpy(), want[k]) for k in ("depth", "dt", "mask"))
    eng.handle.set_pipeline_depth(args.pipeline)           # second pass, same mode, with the label map
    ol = [new_outs(with_lbl=True) for _ in range(2)]
    for i in range(2):
        r_l = eng.fill(x, src_thr=src_thr, want_lbl=True, out=ol[i])
    eng.flush(); eng.status()
    ok = ok and all(np.array_equal(r_l[k][tsel].cpu().numpy(), want[k]) for k in ("depth", "dt", "mask", "lbl"))
    del ol, r_l
    if dist is not None:
        t_ = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MIN)
        ok = bool(t_.item() > 0.5)
    assert ok, "parity: the timed run's outputs differ from the oracle"
    eng.handle.set_pipeline_depth(1)
    assert torch.equal(outs[0]["depth"], outs[1]["depth"]) and torch.equal(outs[0]["dt"], outs[1]["dt"])

    # ---- per-kernel shares (CUDA events between the launches, same stream), separate untimed steps ----
    # (the kernels of the timed configuration: with batches in flight the rows above the first source row go to
    # k3_sky, so the profiled steps ask for that explicitly -- profiling itself runs in strict order)
    eng.handle.set_profiling(True)
    if args.pipeline > 1:
        eng.handle.set_sky_min(8)
    kt = {}
    reps = 5
    for _ in range(reps):
        eng.fill(x, src_thr=src_thr, out=outs[0])
        for k, v in eng.handle.kernel_times().items():
            kt[k] = kt.get(k, 0.0) + v / reps
    eng.handle.set_profiling(False)
    eng.handle.set_sky_min(-1)
    tasks = eng.handle.debug_tasks(1 << 17)           # pixels the scan kernel wrote (the rest are k3_sky's)
    k2_px = int(((tasks[:, 4] - tasks[:, 3]).astype(np.int64) * (tasks[:, 10] - tasks[:, 9])).sum())
    ktot = sum(kt.values())

    # ---- the dominant kernel in the regime of the timed step: ONLY k2_chamfer launched (dtfill_debug_set_skip), the same
    # number of batches in flight, on the workspace complete runs left behind (bit rows, tasks, depth lists).  A launch
    # timed alone in strict order (kernel_ms above) leaves two thirds of the warp slots empty; this is the kernel's
    # throughput when the slots are full, which is how it runs inside the timed region.
    k2_sat_ms = None
    if args.pipeline > 1:
        eng.handle.set_pipeline_depth(args.pipeline)
        for i in range(2 * args.pipeline):
            outs[i % len(outs)] = eng.fill(x, src_thr=src_thr, out=outs[i % len(outs)])
        eng.flush(); eng.status()
        eng.handle.debug_set_skip(1 | 2 | 8)              # K1, K1b and k3_sky are not launched
        for i in range(args.pipeline):
            outs[i % len(outs)] = eng.fill(x, src_thr=src_thr, out=outs[i % len(outs)])
        eng.flush(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nsat = max(K, 20)
        e0.record()
        for i in range(nsat):
            outs[i % len(outs)] = eng.fill(x, src_thr=src_thr, out=outs[i % len(outs)])
        eng.flush(); e1.record(); torch.cuda.synchronize()
        k2_sat_ms = e0.elapsed_time(e1) / nsat
        eng.handle.debug_set_skip(0)
        eng.status()
        eng.handle.set_pipeline_depth(1)

    # ---- end to end, the drop-in call: tools.DT_complete_batch(pageable numpy) -> fresh pageable numpy (tools.py:13-35)
    e2e = e2e_pinned = None
    if workload.startswith("kitti"):
        x4 = frames_np[:, :, :, None]                 # [B,352,1216,1], ordinary (pageable) memory
        # staging threads: the CPUs this rank may use, shared with the other ranks bound to the same NUMA node
        avail, total = len(os.sched_getaffinity(0)), os.cpu_count() or 1
        sharing = max(1, round(world * avail / total))
        stage_threads = max(1, min(12, (3 * avail // 4) // sharing))
        _lib.get_handle(local_rank).set_stage_threads(stage_threads)
        for _ in range(3):                            # warm-up: staging mirrors, the pool of output buffers
            r4 = tools.DT_complete_batch(x4, device=local_rank)
        e2e_steps = max(3, min(K, 8))
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r4 = tools.DT_complete_batch(x4, device=local_rank)
        t_e2e = time.perf_counter() - t0
        t_own = t_e2e
        if dist is not None:
            t = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_e2e = float(t.item())
        assert np.array_equal(r4[sel, :, :, 0], want["depth"]), "drop-in call differs from the oracle"
        nbytes = int(B * H * W * 4)
        h2d_link, d2h_link = _lib.get_handle(local_rank).transfer_bytes()    # what the last call moved over the link
        per_rank = [nbytes * e2e_steps / t_own / 1e9]
        if dist is not None:
            g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
            dist.all_gather(g, torch.tensor([per_rank[0]], dtype=torch.float64, device=dev))
            per_rank = [float(v.item()) for v in g]
        e2e = {"value": world * B * e2e_steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d_link),
               "d2h_bytes_per_step": int(d2h_link), "host_input_bytes_per_step": nbytes, "steps": e2e_steps,
               "what": "tools.DT_complete_batch(x): pageable numpy [B,352,1216,1] in, a new numpy array out every call, "
                       "synchronous (the reference's contract, tools.py:13-35); host threads read the input once and "
                       "compact it to (pixel, value) pairs of the source / valid pixels (sparse upload, include/dtfill.h: "
                       "h2d_bytes_per_step is what crossed the link, host_input_bytes_per_step the array handed in), the "
                       "device rebuilds the dense frames; the output array's memory comes from a pool of page-locked buffers",
               "per_rank_gbs_of_host_arrays_each_direction": [round(v, 2) for v in per_rank], "numa": numa,
               "stage_threads_per_rank": stage_threads}
        del r4
    # ---- the C ABI with pinned host buffers and all three outputs (what round 1 reported as e2e) ----
    h = _lib.Handle(local_rank)
    pin_in = _lib.pinned_empty((B, H, W), np.float32)
    pin_in[...] = frames_np
    pin_out = dict(depth=_lib.pinned_empty((B, H, W), np.float32), dt=_lib.pinned_empty((B, H, W), np.float32),
                   mask=_lib.pinned_empty((B, H, W), np.uint8))
    h.run_host(pin_in, src_thr, 0.1, want_dt=True, want_mask=True, out=pin_out)
    pin_steps = max(3, min(K, 8))
    barrier()
    t0 = time.perf_counter()
    for _ in range(pin_steps):
        r = h.run_host(pin_in, src_thr, 0.1, want_dt=True, want_mask=True, out=pin_out)
    t_pin = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([t_pin], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_pin = float(t.item())
    assert np.array_equal(r["depth"][sel], want["depth"]) and np.array_equal(r["dt"][sel], want["dt"])
    e2e_pinned = {"value": world * B * pin_steps / t_pin, "unit": UNIT, "h2d_bytes_per_step": int(B * H * W * 4),
                  "d2h_bytes_per_step": int(B * H * W * 9), "steps": pin_steps,
                  "what": "dtfill_run (C ABI) with pinned host numpy buffers in and out, depth + dt + mask, synchronous"}
    if e2e is None:
        e2e = e2e_pinned
    h.close()

    # ---- BASELINE.json configs[4] on the same clock ----
    sweep = None
    if workload == "kitti64" and not args.no_sweep:
        del outs
        torch.cuda.empty_cache()
        sweep = run_sweep(args, eng, dev, rank, world, dist, comm, barrier, min(args.min_seconds, 0.5))

    if rank != 0:
        if comm is not None:
            comm.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    px_step = B * H * W
    achieved = ALG_BYTES_PER_PX * px_step / (ms_per_step * 1e-3) / 1e9 * 1.0      # per GPU (rank-0 clock = max)
    traffic = traffic_k2 = None          # DRAM bytes from the committed ncu --set full capture (batch 256 only)
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and B == 256 and workload == "kitti64":
        try:
            tj = json.load(open(tp))
            traffic, traffic_k2 = tj.get("dram_bytes_per_step"), tj.get("dram_bytes_per_launch")
        except Exception:
            traffic = traffic_k2 = None
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_what": "dram__bytes_read+write of all kernels of one step (profiles/traffic.json); "
                                              "algorithmic bytes per step = 13 B/px x px",
        "algorithmic_bytes": ALG_BYTES_PER_PX * px_step, "peak_source": peak_src,
        "strict_frac": ALG_BYTES_PER_PX * px_step / (ms_strict / K * 1e-3) / 1e9 / peak,
        "what": "whole fused path of one step (k1_mask_rows + k1b_scan_compact + k2_chamfer + k3_sky [+ k2_chamfer_wide "
                f"no-op]): {ALG_BYTES_PER_PX} B/px x {px_step} px per step / step time (K timed steps); dominant "
                "kernel k2_chamfer; kernel_ms = CUDA events between the launches of separate, strictly ordered steps",
        "kernel_ms": kt, "kernel_share": {k: (v / ktot if ktot else None) for k, v in kt.items()},
        "dominant_kernel": {"name": "k2_chamfer", "ms": kt.get("k2_chamfer"),
                            "alg_bytes": 8 * k2_px, "traffic": traffic_k2,
                            "alg_bytes_what": "8 B (depth + dt) x the pixels this kernel writes; the rows above the "
                                              "first source row are written by k3_sky",
                            "achieved_gbs": (8 * k2_px / (kt["k2_chamfer"] * 1e-3) / 1e9) if kt.get("k2_chamfer") else None,
                            "saturated": None if not k2_sat_ms else {
                                "ms": k2_sat_ms, "achieved_gbs": 8 * k2_px / (k2_sat_ms * 1e-3) / 1e9,
                                "frac": 8 * k2_px / (k2_sat_ms * 1e-3) / 1e9 / peak,
                                "traffic_gbs": (traffic_k2 / (k2_sat_ms * 1e-3) / 1e9) if traffic_k2 else None,
                                "what": f"only k2_chamfer launched, {args.pipeline} batches in flight, CUDA events around "
                                        "the run (profiles/stage_probe.py does the same for every stage): the kernel with "
                                        "its warp slots full, as inside the timed step"}},
    }

    # ---- CPU baseline on this box's host cores (bounded sample of the same workload) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(frames_np)        # (the port uses the KITTI thresholds; NYU frames have depths >= 1 m)
        sample = B if workload.startswith("kitti") else min(B, 256)
        ref.run(min(sample, max(ref.cores, 8)))
        reps_cpu, t_cpu = 0, 0.0
        while t_cpu < 10.0 and reps_cpu < 100:
            t_cpu += ref.run(sample)
            reps_cpu += 1
        ref.close()
        kind, how = ref.describe()
        cpu = {"value": sample * reps_cpu / t_cpu, "unit": UNIT, "cores": ref.cores, "kind": kind,
               "sample": f"{sample} frames x {reps_cpu} repeats ({t_cpu:.1f} s); {how}"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 keys (integer chamfer) + f32 copy", "data": "synthetic",
        "config": {"workload": (f"kitti64: batch of {B} synthetic KITTI 64-beam frames 352x1216 (~5% density) per GPU "
                                "(BASELINE.json configs[1])") if workload == "kitti64" else
                               f"{workload}: batch of {B} synthetic frames {H}x{W} per GPU",
                   "outputs": "filled depth f32 + distance channel f32 + validity mask u8 (13 B/px algorithmic)",
                   "l2": f"inputs+outputs per step {ALG_BYTES_PER_PX * px_step / 1e6:.0f} MB > 126 MB L2 (no flush needed)",
                   "frames_per_step_per_gpu": B,
                   "pipeline": (f"{args.pipeline} batches in flight (dtfill_set_pipeline_depth): K1/K1b of step n+1 "
                                f"overlap K2 of step n; {no} output sets rotate; all outputs complete at the end "
                                "of the timed steps") if args.pipeline > 1 else "strict stream order between steps",
                   "timing": f"{K} steps between two CUDA events (max over ranks)"},
        "timed_region_s": ms * 1e-3,
        "strict": strict, "parity_checked": int(len(sel)),
        "parity_what": f"{len(sel)} frames of the timed run's own outputs (depth, dt, mask; lbl in a second pass in the "
                       "same mode) bit-identical to oracle/dtfill_oracle.c, on every rank",
        "roofline": roofline, "cpu_baseline": cpu,
        "e2e": e2e, "e2e_pinned": e2e_pinned, "sweep": sweep,
        "gpu_launches": launches_per_step * K, "gpu_launches_per_step": launches_per_step,
        "clocks": clocks, "clocks_strict": clocks_strict,
    }
    emit(line)
    if comm is not None:
        comm.close()
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line, alone on the real stdout (see main: everything else printed to fd 1 goes to stderr)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    # libraries (NCCL prints its version banner at communicator creation) write to fd 1: keep the real stdout for the
    # JSON line and send everything else to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps (one batch per GPU each)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU and step (default: the workload's)")
    ap.add_argument("--workload", default="kitti64", choices=sorted(WORKLOADS) + ["sweep"],
                    help="kitti64 is the BASELINE.json metric (its line also carries the sweep); sweep runs configs[4] alone")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--pipeline", type=int, default=4, choices=[1, 2, 3, 4],
                    help="batches in flight in the device-resident timing (1 = strict stream order)")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="least duration of the timed sweep region")
    ap.add_argument("--parity-frames", type=int, default=64)
    ap.add_argument("--sweep-frames", type=int, default=8192)
    ap.add_argument("--sweep-batch", type=int, default=256)
    ap.add_argument("--band-cap", type=int, default=None, help="override the band planner target (row steps)")
    ap.add_argument("--subbatches", type=int, default=None, help="override the number of sub-batch streams")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (a seeded sample of frames, rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
