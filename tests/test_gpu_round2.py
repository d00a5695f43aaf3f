"""GPU tests added in round 2: parity at the benchmarked batch sizes and pipeline depth, the per-call status ring, the
fused evaluation step and its totals, the NCCL all-reduce behind the C ABI, the label-width boundary of the packed
keys, synchronous calls while batches are in flight, pooled output buffers, threads sharing a handle.
Run on the B200 box:  python -m pytest tests -m gpu"""
import os
import socket
import threading

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib, sharding, synth, tools
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle(dtfill_lib):
    return _lib.get_handle()


@pytest.fixture(scope="module")
def torch_mod():
    return pytest.importorskip("torch")


def _bench_frames(workload, n):
    import bench
    return bench.make_frames(n, 0, workload), bench.WORKLOADS[workload][3]


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["kitti16", "kitti64"])
def test_every_frame_of_pipelined_batches(handle, torch_mod, workload):
    """Every frame of every output set of a pipelined run against the oracle, not a sample: a bulk copy that overtook
    the stores of the last forward rows (missing async-proxy fence in k2_chamfer) corrupted the bottom rows of about one
    frame in a thousand, only with four batches in flight -- the 64-frame samples above never met one."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    frames, src_thr = _bench_frames(workload, 256)
    want = O.dt_fill(frames, src_thr=src_thr)
    x = torch.from_numpy(frames).cuda()
    eng = DTFillEngine(0, pipeline_depth=4)
    outs = [None] * 4
    for rounds in range(3):
        for i in range(8):
            outs[i % 4] = eng.fill(x, src_thr=src_thr, out=outs[i % 4])
        eng.flush()
        bad, _ = eng.status()
        assert bad == -1
        for j, o in enumerate(outs):
            for k in ("depth", "dt", "mask"):
                got = o[k].cpu().numpy()
                assert np.array_equal(got, want[k]), (workload, rounds, j, k, np.unique(np.nonzero(got != want[k])[0])[:8])


@pytest.mark.parametrize("workload,batch", [("kitti64", 256), ("kitti32", 256), ("kitti16", 256), ("kitti8", 256),
                                            ("nyu", 1024)])
def test_benchmarked_batches_pipelined_auto_cap(handle, torch_mod, workload, batch):
    """The configurations DESIGN.md section 5 and bench.py quote (BASELINE.json configs[1..3]: 256 KITTI frames of
    64/32/16/8 beams; configs[3]: 1024 NYU frames) through DTFillEngine(pipeline_depth=4) with the automatic band
    target, which depends on the batch size and the depth: 64 frames of every run against the oracle, bit for bit."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    frames, src_thr = _bench_frames(workload, batch)
    x = torch.from_numpy(frames).cuda()
    eng = DTFillEngine(0, pipeline_depth=4)
    outs = [None] * 4
    for i in range(6):                                   # several batches in flight, as in the timed region
        outs[i % 4] = eng.fill(x, src_thr=src_thr, want_lbl=True, out=outs[i % 4])
    eng.flush()
    bad, _ = eng.status()
    assert bad == -1
    sel = np.unique(np.linspace(0, batch - 1, 64).astype(int))
    want = O.dt_fill(frames[sel], src_thr=src_thr)
    tsel = torch.from_numpy(sel).cuda()
    for o in (outs[1], outs[0]):                         # the last call and the one three calls before it
        for k in ("depth", "dt", "mask", "lbl"):
            assert np.array_equal(o[k][tsel].cpu().numpy(), want[k]), (workload, k)
    assert len(eng.handle.debug_tasks(1 << 17)) > 0


def test_status_ring_keeps_every_calls_verdict(handle, torch_mod):
    """3 x depth calls between two status checks, a frame without a valid pixel (numpy IndexError, tools.py:26) in the
    FIRST call only: dtfill_status must still report it (one status slot per call)."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    depth = 3
    eng = DTFillEngine(0, pipeline_depth=depth)
    good = torch.from_numpy(np.stack([synth.kitti_frame(i)[100:180, :320] for i in range(4)])).cuda()
    badb = good.clone()
    badb[2].zero_()
    outs = [None] * depth
    outs[0] = eng.fill(badb, out=outs[0])
    for i in range(1, 3 * depth):
        outs[i % depth] = eng.fill(good, out=outs[i % depth])
    bad, _ = eng.status()
    assert bad == 2
    bad, _ = eng.status()                                # reported once
    assert bad == -1
    # more calls than the ring has slots: the verdict of a slot that is reused is folded, not dropped
    outs[0] = eng.fill(badb, out=outs[0])
    for i in range(1, 70):
        outs[i % depth] = eng.fill(good, out=outs[i % depth])
    bad, _ = eng.status()
    assert bad == 2


def test_sync_call_with_device_input_while_pipelined(handle, torch_mod):
    """dtfill_run with a device input and HOST outputs on a handle whose pipeline depth is 3 (ADVICE r1): the copies to
    the host must follow the kernels."""
    torch = torch_mod
    frames = np.stack([synth.kitti_frame(i)[90:250, :640] for i in range(6)])
    h = _lib.Handle(0)
    h.set_pipeline_depth(3)
    x = torch.from_numpy(frames).cuda()
    B, H, W = frames.shape
    depth = np.full((B, H, W), -1.0, np.float32)
    dt = np.full((B, H, W), -1.0, np.float32)
    bad = _lib.ctypes.c_int(-1)
    rc = h._L.dtfill_run(h._h, _lib._ptr(x.data_ptr()), 1, B, H, W, 0.1, 0.1, _lib._ptr(depth), _lib._ptr(dt), None, None,
                         None, 0, _lib.ctypes.byref(bad))
    assert rc == 0
    want = O.dt_fill(frames)
    assert np.array_equal(depth, want["depth"]) and np.array_equal(dt, want["dt"])
    h.close()


def test_fused_eval_step_and_totals(handle, torch_mod):
    """dtfill_run_eval_async + dtfill_eval_totals (one step of the sweep, eval.py:212-232) against per-frame
    Result.evaluate of the oracle: strict and pipelined, float64 and float32 ground truth."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    n = 10
    frames = np.stack([synth.kitti_frame(i) for i in range(n)])
    gt = np.stack([synth.kitti_gt(i) for i in range(n)])
    fill = O.dt_fill(frames)["depth"]
    per = [O.result_kitti(fill[i], gt[i]) for i in range(n)]
    want = np.array([sum(m[k] for m in per) for k in ("mse", "rmse", "mae", "irmse", "imae")])
    x, g = torch.from_numpy(frames).cuda(), torch.from_numpy(gt).cuda()
    for depth in (1, 3):
        eng = DTFillEngine(0, pipeline_depth=depth)
        for lo in range(0, n, 2):                        # five calls of two frames
            eng.fill_eval(x[lo:lo + 2], g[lo:lo + 2])
        tot = eng.eval_totals().cpu().numpy()
        assert eng.status()[0] == -1
        np.testing.assert_allclose(tot[:5], want, rtol=1e-9)
        assert tot[9] == n and tot[8] == sum(m["count"] for m in per)
        assert np.all(eng.eval_totals().cpu().numpy() == 0)          # collected totals are cleared
        run = torch.zeros(10, dtype=torch.float64, device="cuda")
        eng.fill_eval(x[:4], g[:4]); eng.eval_totals(run)
        eng.fill_eval(x[4:], g[4:]); eng.eval_totals(run)            # accumulate into the caller's vector
        np.testing.assert_allclose(run.cpu().numpy()[:5], want, rtol=1e-9)
    eng = DTFillEngine(0)
    g32 = g.float()
    eng.fill_eval(x, g32)
    tot = eng.eval_totals().cpu().numpy()
    per32 = [O.result_kitti(fill[i], gt[i].astype(np.float32)) for i in range(n)]
    np.testing.assert_allclose(tot[1], sum(m["rmse"] for m in per32), rtol=2e-5)


@pytest.mark.parametrize("nsrc", [(1 << 17) - 2, (1 << 17) - 1, 1 << 17, (1 << 17) + 1])
def test_label_width_boundary(handle, nsrc):
    """The packed key holds 17 label bits: frames with up to 2^17 - 1 sources take the fast kernels, from 2^17 on the
    64-bit-key path.  Both sides of the boundary against the oracle."""
    H, W = 352, 1216
    rng = np.random.default_rng(nsrc)
    x = np.zeros(H * W, np.float32)
    pos = rng.choice(H * W, size=nsrc, replace=False)
    x[pos] = rng.uniform(1.0, 60.0, nsrc).astype(np.float32)
    x = x.reshape(1, H, W)
    r = handle.run_host(x, 0.1, 0.1, want_dt=True, want_lbl=True, want_mask=True)
    assert "index_error" not in r
    o = O.dt_fill(x)
    assert int(r["counts"][0, 0]) == nsrc
    for k in ("depth", "dt", "lbl", "mask"):
        assert np.array_equal(r[k], o[k]), k
    assert int(o["lbl"].max()) == nsrc


def test_dt_complete_batch_returns_fresh_arrays(handle):
    """tools.py:27-33 returns a new array per call: results handed out earlier must not change when their pooled
    page-locked buffers are reused, and dropping a result must make its buffer reusable."""
    xa, xb = synth.kitti_batch([3]), synth.kitti_batch([4])
    ra = tools.DT_complete_batch(xa)
    keep = ra.copy()
    rb = tools.DT_complete_batch(xb)
    assert ra.ctypes.data != rb.ctypes.data
    assert np.array_equal(ra, keep)
    assert ra.flags.writeable and ra.dtype == np.float32 and ra.shape == (1, 352, 1216, 1)
    addr = rb.ctypes.data
    del rb
    rc = tools.DT_complete_batch(xb)
    assert rc.ctypes.data == addr                        # the buffer came back from the pool
    assert np.array_equal(ra, keep)
    assert np.array_equal(rc[..., 0], O.dt_fill(xb[..., 0])["depth"])
    view = rc[0, 100:110]
    del rc
    rd = tools.DT_complete_batch(xa)                     # a live view keeps its buffer out of the pool
    assert rd.ctypes.data != addr and view.base is not None


def test_threads_share_the_device_handle(handle):
    """Two Python threads calling the drop-ins at once go through the same cached handle (ADVICE r1): calls are
    serialised per handle, results stay correct."""
    xs = [synth.kitti_batch([10 + i]) for i in range(2)]
    want = [O.dt_fill(x[..., 0])["depth"] for x in xs]
    errs = []

    def work(i):
        try:
            for _ in range(4):
                got = tools.DT_complete_batch(xs[i])
                if not np.array_equal(got[..., 0], want[i]):
                    errs.append(f"thread {i}: wrong result")
        except Exception as e:          # noqa: BLE001
            errs.append(repr(e))

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs


def _nccl_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n = 6
    b, e = sharding.shard_range(n, rank, world)
    frames = np.stack([synth.kitti_frame(i) for i in range(b, e)])
    gt = np.stack([synth.kitti_gt(i) for i in range(b, e)])
    eng = DTFillEngine(rank, pipeline_depth=2)
    comm = sharding.MetricsComm(eng.handle, rank, world)
    x, g = torch.from_numpy(frames).cuda(), torch.from_numpy(gt).cuda()
    for lo in range(0, e - b):
        eng.fill_eval(x[lo:lo + 1], g[lo:lo + 1])
    tot = eng.eval_totals()
    comm.allreduce(eng, tot)                             # dtfill_allreduce_sums on the engine's stream
    torch.cuda.synchronize()
    if rank == 0:
        q.put(tot.cpu().numpy().copy())
    comm.close()
    dist.destroy_process_group()


def test_allreduce_sums_two_ranks_equal_one_rank(handle, torch_mod):
    """dtfill_allreduce_sums over 2 GPUs: the means of the sharded sweep equal the 1-rank means to 1e-12
    (eval.py:212-232, 252-259)."""
    torch = torch_mod
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    n = 6
    eng = DTFillEngine(0)
    x = torch.from_numpy(np.stack([synth.kitti_frame(i) for i in range(n)])).cuda()
    g = torch.from_numpy(np.stack([synth.kitti_gt(i) for i in range(n)])).cuda()
    for i in range(n):
        eng.fill_eval(x[i:i + 1], g[i:i + 1])
    one = eng.eval_totals().cpu().numpy()
    np.testing.assert_allclose(got, one, rtol=1e-12)
    m2, m1 = sharding.finalize_means(got), sharding.finalize_means(one)
    assert m2["frames"] == n and abs(m2["rmse"] - m1["rmse"]) <= 1e-12 * m1["rmse"]


@pytest.mark.gpu
def test_sparse_upload_matches_dense_upload(handle):
    """dtfill_run with a pageable float32 input compacts it on the host to (pixel, value) pairs (include/dtfill.h, sparse
    upload): same outputs as the dense copy and as the oracle, for sparse frames, for frames too dense for the pair
    buffer (fallback inside one call), for NaN / negative / denormal / signed-zero pixels and for the valid-but-not-source
    band of tools.py:8 vs :22; thresholds that make 0.0 a source switch it off."""
    rng = np.random.default_rng(11)
    H, W, B = 96, 256, 20
    x = np.zeros((B, H, W), np.float32)
    for b in range(B):
        dens = [0.01, 0.05, 0.2, 0.6][b % 4]                          # 0.6: more than the pair buffer holds
        m = rng.random((H, W)) < dens
        x[b][m] = (np.round(rng.uniform(0.05, 60.0, m.sum()) * 256) / 256).astype(np.float32)
    x[4, 5, 7] = np.nan; x[4, 9, 9] = -4.0; x[4, 10, 10] = -0.0; x[4, 11, 11] = 1e-41       # NaN: a source, not valid
    x[4, 20, 20] = 0.5; x[4, 21, 21] = 0.1; x[4, 22, 22] = 0.9; x[4, 23, 23] = np.float32(0.90000004)
    want = O.dt_fill(x)
    outs = {}
    for sparse in (True, False):
        handle.set_sparse_upload(sparse)
        try:
            r = handle.run_host(x, 0.1, 0.1, want_dt=True, want_lbl=True, want_mask=True)
            outs[sparse] = r, handle.transfer_bytes()
        finally:
            handle.set_sparse_upload(True)
        for k in ("depth", "dt", "lbl", "mask"):
            assert np.array_equal(r[k], want[k], equal_nan=True), (sparse, k)
    assert outs[False][1][0] == x.nbytes                                # dense: the whole array crossed the link
    assert outs[True][1][0] < x.nbytes                                  # sparse: pairs, plus the slices that fell back
    assert outs[True][1][1] == outs[False][1][1] == B * H * W * 13
    # a source threshold >= 1 makes 0.0 a source: the dense copy must be taken (every pixel valid, so no IndexError)
    xd = (np.round(rng.uniform(1.0, 50.0, (2, H, W)) * 256) / 256).astype(np.float32)
    r = handle.run_host(xd, 1.0, 0.1, want_dt=True)
    w2 = O.dt_fill(xd, src_thr=1.0)
    assert np.array_equal(r["dt"], w2["dt"]) and np.array_equal(r["depth"], w2["depth"])
    assert handle.transfer_bytes()[0] == xd.nbytes


@pytest.mark.gpu
def test_float64_and_integer_inputs_follow_the_reference(handle):
    """tools.py:8 / :22 evaluate their predicates in the input's dtype and eval_NYU.Distance_Transform returns it
    (:126-133): float64 (and integer) inputs go through the float64 route of the drop-ins -- predicates on the host in
    float64, labels from the kernels, depths gathered from the float64 values -- and equal the line-by-line cv2 port of
    the reference, including values that float32 would move across a threshold."""
    cv2 = pytest.importorskip("cv2")
    from distancetransform_depthcompletion_b200 import tools, eval_nyu
    rng = np.random.default_rng(21)
    x = np.zeros((2, 352, 1216, 1), np.float64)
    m = rng.random(x.shape) < 0.05
    x[m] = rng.uniform(1.0, 80.0, m.sum())
    x[0, 200, 300, 0] = 0.9                          # float64: 1 - 0.9 = 0.09999999999999998 -> a source; not one in float32
    x[0, 210, 310, 0] = 0.1 + 1e-12                  # valid in float64, equal to 0.1f after rounding
    x[0, 220, 320, 0] = 0.5                          # valid, not a source: later labels read a shifted entry
    want = O.cv2_port_complete_batch(x)
    got = tools.DT_complete_batch(x)
    assert got.dtype == np.float32 and got.shape == want.shape and np.array_equal(got, want)
    dt_w, lbl_w = O.cv2_port_nearest_point(x[0, :, :, 0])
    dt_g, lbl_g = tools.nearest_point(x[0, :, :, 0])
    assert np.array_equal(dt_g, dt_w) and np.array_equal(lbl_g, lbl_w)
    y = np.zeros((480, 640), np.float64)
    ys, xs = rng.integers(6, 468, 500), rng.integers(8, 624, 500)
    y[ys, xs] = rng.uniform(1.0, 10.0, 500)
    w, _, _ = O.cv2_port_fill_frame(y, 0.001, 0.1, nyu_style=True)
    g = eval_nyu.Distance_Transform(y)
    assert g.dtype == np.float64 and np.array_equal(g, w)
    yi = np.zeros((64, 96), np.int64); yi[10, 20] = 7; yi[40, 70] = 3
    gi = eval_nyu.Distance_Transform(yi)
    wi, _, _ = O.cv2_port_fill_frame(yi, 0.001, 0.1, nyu_style=True)
    assert gi.dtype == yi.dtype and np.array_equal(gi, wi)


@pytest.mark.parametrize("batch", [1, 7, 64, 66])
def test_strict_calls_on_both_sides_of_the_sky_split(handle, torch_mod, batch):
    """Strict order, full-size KITTI frames: up to 64 frames per call the cell row with k3_sky's base rows is a full-width
    task of its own and k3_sky runs beside the narrow tiles on the side stream; larger calls keep k3_sky behind the scan
    (csrc/dtfill.cu, fp.sky_split).  Every frame of both kinds of call against the oracle, labels on and off, and the
    task list shows which plan ran."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    frames = np.stack([synth.kitti_frame(100 + i, beam_step=(1, 2, 1, 4)[i % 4]) for i in range(batch)])
    want = O.dt_fill(frames)
    eng = DTFillEngine(0)
    x = torch.from_numpy(frames).cuda()
    for want_lbl in (False, True):
        out = eng.fill(x, want_lbl=want_lbl)
        bad, _ = eng.status()
        assert bad == -1
        for k in ("depth", "dt", "mask") + (("lbl",) if want_lbl else ()):
            assert np.array_equal(out[k].cpu().numpy(), want[k]), (batch, k)
    t = eng.handle.debug_tasks(1 << 16)
    kinds = t[:, 5]
    full_width = int((kinds == 0).sum())
    assert int((kinds == 4).sum()) > 0
    assert (full_width >= batch) if batch <= 64 else (full_width == 0), (batch, full_width)


def test_status_slots_are_rearmed_after_a_verdict(handle, torch_mod):
    """The device side of a status slot is armed once and re-armed only after it reported something: more calls than the
    ring has slots with a bad frame every 64th + 5th call, checked in groups -- a stale verdict would show up in a later
    group, a missing re-arm as a verdict that never goes away."""
    torch = torch_mod
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    eng = DTFillEngine(0)
    good = torch.from_numpy(np.stack([synth.kitti_frame(i)[100:180, :320] for i in range(3)])).cuda()
    badb = good.clone()
    badb[1].zero_()
    out = None
    for group in range(5):
        for i in range(40):
            out = eng.fill(badb if (group % 2 == 0 and i == 5) else good, out=out)
        bad, _ = eng.status()
        assert bad == (1 if group % 2 == 0 else -1), group
    for i in range(200):                                   # no status call in between: slots are reused three times
        out = eng.fill(badb if i == 3 else good, out=out)
    assert eng.status()[0] == 1
    for i in range(70):
        out = eng.fill(good, out=out)
    assert eng.status()[0] == -1
