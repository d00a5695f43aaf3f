"""evaluation.evaluate_fill_png_files (dtfill_eval_png): the KITTI ablation notebook's loop from the PNG files,

    lidar = png.astype(np.float32) / 256;  gt = png / 256.;  Result().evaluate(Distance_Transform(lidar, src_thr), gt)

per frame, against the same composition of the package's own calls, bit for bit (== with NaN where numpy gives NaN),
and a subset against the CPU oracle.  The CPU tests need no device: the export and the checks that run before the
device is touched.  Run the rest on the B200 box:  python -m pytest tests -m gpu"""
import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib, eval_nyu, evaluation, synth

STRATS = sorted(P.STRATEGIES)
K = 16          # distinct frame pairs per beam count; larger batches repeat them


# ---- expected values: the notebook's loop, one frame at a time -------------------------------------------------
def _samples(f):
    return P.decode(f) if isinstance(f, (bytes, bytearray)) else np.asarray(f, np.uint16)


def expected_row(lidar_file, gt_file, src_thr=0.1):
    """One frame of the loop: png_oracle.decode, eval_nyu.Distance_Transform, Result.evaluate -> the row of
    evaluate_fill_png_files (files as bytes, or their uint16 samples)."""
    lidar = _samples(lidar_file).astype(np.float32) / 256
    gt = _samples(gt_file) / 256.0
    pred = eval_nyu.Distance_Transform(lidar, src_thr)
    r = evaluation.Result()
    r.evaluate(pred, gt)
    n = int(np.logical_and(pred > 0.01, gt > 0.01).sum())
    return np.array([r.mse, r.rmse, r.mae, r.irmse, r.imae, 0, 0, 0, n], np.float64)


def expected_sums(rows):
    """The running sums the loop keeps (eval.py:212-232 `+=`, frame after frame), then the frame count."""
    s = np.zeros(10, np.float64)
    for r in rows:
        s[:9] += r
    s[9] = len(rows)
    return s


def oracle_row(lidar_file, gt_file, src_thr=0.1):
    """The same frame through the CPU oracle: oracle.dt_fill + oracle.result_kitti."""
    from oracle import oracle as O
    lidar = _samples(lidar_file).astype(np.float32) / 256
    gt = _samples(gt_file) / 256.0
    pred = O.dt_fill(lidar, src_thr, 0.1)["depth"]
    m = O.result_kitti(pred, gt)
    return np.array([m["mse"], m["rmse"], m["mae"], m["irmse"], m["imae"], 0, 0, 0, m["count"]], np.float64)


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def lidar16(seed, beams=64, H=synth.KITTI_H, W=synth.KITTI_W):
    return np.rint(synth.kitti_frame(seed, H, W, beam_step=64 // beams) * 256).astype(np.uint16)


def gt16(seed, H=synth.KITTI_H, W=synth.KITTI_W):
    return np.rint(synth.kitti_gt(seed, H, W) * 256).astype(np.uint16)


def _kinds(i, x):
    """The i-th kind of encoding: every filter, zlib level and strategy, IDAT splits, ancillary chunks."""
    filters = [0, 1, 2, 3, 4, "random", "msad"][i % 7]
    level = i % 10
    strategy = STRATS[(i // 10) % len(STRATS)]
    idat = ["one", 4096, "random", 7][(i // 3) % 4]
    return P.encode(x, filters=filters, level=level, strategy=strategy, idat=idat, ancillary=i % 5 == 0, seed=i)


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_symbol_is_exported(dtfill_lib):
    import ctypes
    assert hasattr(ctypes.CDLL(dtfill_lib), "dtfill_eval_png")
    assert _lib.load().dtfill_eval_png is not None
    assert callable(evaluation.evaluate_fill_png_files)


@pytest.fixture
def no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the device was touched")
    monkeypatch.setattr(_lib, "get_handle", refuse)
    monkeypatch.setattr(_lib, "Handle", refuse)


def test_list_checks_raise_before_the_device(no_device):
    f = P.encode(np.zeros((4, 5), np.uint16))
    with pytest.raises(ValueError, match="no files"):
        evaluation.evaluate_fill_png_files([], [])
    with pytest.raises(ValueError, match="no files"):
        evaluation.evaluate_fill_png_files([f], [])
    with pytest.raises(ValueError, match="2 LiDAR files but 3 ground-truth files"):
        evaluation.evaluate_fill_png_files([f, f], [f, f, f])
    with pytest.raises(ValueError, match="LiDAR file 0"):
        evaluation.evaluate_fill_png_files([b"not a png at all, but long enough"], [f])
    with pytest.raises(ValueError, match="LiDAR file 0"):
        evaluation.evaluate_fill_png_files([f[:20]], [f])


# ---- GPU ----------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def pool():
    """K distinct KITTI-size pairs per beam count, encoded at zlib level 6; expected rows cached per src_thr."""
    out = {}
    for beams in (64, 16):
        lid = [lidar16(s, beams) for s in range(K)]
        gt = [gt16(1000 + s) for s in range(K)]
        out[beams] = dict(lid=lid, gt=gt, lf=[P.encode(x) for x in lid], gf=[P.encode(x) for x in gt], rows={})
    return out


def _rows(p, idx, src_thr=0.1):
    rows = []
    for i, j in idx:
        key = (i, j, src_thr)
        if key not in p["rows"]:
            p["rows"][key] = expected_row(p["lid"][i], p["gt"][j], src_thr)
        rows.append(p["rows"][key])
    return np.stack(rows)


def _pairs(B):
    """(LiDAR, ground truth) of frame b: all K * K pairs before any repeats."""
    return [(b % K, (b // K + 5 * b + 3) % K) for b in range(B)]


@gpu
@pytest.mark.parametrize("beams", [64, 16])
@pytest.mark.parametrize("B", [1, 7, 256, 1000])
def test_rows_and_sums_bit_exact(dtfill_lib, pool, B, beams):
    p = pool[beams]
    idx = _pairs(B)
    pf, sums = evaluation.evaluate_fill_png_files([p["lf"][i] for i, _ in idx], [p["gf"][j] for _, j in idx])
    want = _rows(p, idx)
    assert pf.dtype == np.float64 and pf.shape == (B, 9) and sums.shape == (10,)
    for b in range(B):
        assert _same(pf[b], want[b]), (b, pf[b], want[b])
    assert _same(sums, expected_sums(want))


@gpu
def test_src_thr(dtfill_lib, pool):
    """The source threshold reaches the fill: a sample s is a source when 1 - s/256 <= src_thr, so samples 231..255
    are sources at 0.1 and not at 0.001 (and 1..25 are below the validity threshold at both)."""
    p = pool[64]
    rng = np.random.default_rng(11)
    lid, gt = [], []
    for b in range(8):
        x = p["lid"][b].copy()
        near = rng.random(x.shape) < 0.01
        x[near] = rng.integers(1, 256, int(near.sum()))
        lid.append(x)
        gt.append(p["gt"][(3 * b + 1) % K])
    lf, gf = [P.encode(x) for x in lid], [P.encode(x) for x in gt]
    rows = {}
    for src_thr in (0.1, 0.001):
        pf, sums = evaluation.evaluate_fill_png_files(lf, gf, src_thr)
        want = np.stack([expected_row(a, g, src_thr) for a, g in zip(lid, gt)])
        assert _same(pf, want) and _same(sums, expected_sums(want)), src_thr
        rows[src_thr] = pf
    assert all(not _same(rows[0.1][b], rows[0.001][b]) for b in range(8))


@gpu
def test_every_kind_of_file_and_the_projects_encoder(dtfill_lib, pool):
    p = pool[64]
    n = 40
    idx = _pairs(n)
    lf = [_kinds(b, p["lid"][i]) for b, (i, _) in enumerate(idx)]
    gf = [_kinds(b + 7, p["gt"][j]) for b, (_, j) in enumerate(idx)]
    for b in range(0, n, 8):       # the oracle reads what it wrote
        assert np.array_equal(P.decode(lf[b]), p["lid"][idx[b][0]]) and np.array_equal(P.decode(gf[b]), p["gt"][idx[b][1]])
    want = _rows(p, idx)
    pf, sums = evaluation.evaluate_fill_png_files(lf, gf)
    assert _same(pf, want) and _same(sums, expected_sums(want))
    # files written by the package's own GPU encoder (data_read.write_depth_pngs)
    from distancetransform_depthcompletion_b200 import data_read
    lf2 = data_read.write_depth_pngs(np.stack([p["lid"][i] for i, _ in idx]))
    gf2 = data_read.write_depth_pngs(np.stack([p["gt"][j] for _, j in idx]))
    pf2, sums2 = evaluation.evaluate_fill_png_files(lf2, gf2)
    assert _same(pf2, want) and _same(sums2, expected_sums(want))


@gpu
def test_non_kitti_size(dtfill_lib):
    H, W = 240, 320
    lid = [lidar16(s, 64, H, W) for s in range(9)]
    gt = [gt16(50 + s, H, W) for s in range(9)]
    pf, sums = evaluation.evaluate_fill_png_files([P.encode(x) for x in lid], [P.encode(x) for x in gt])
    want = np.stack([expected_row(a, b) for a, b in zip(lid, gt)])
    assert _same(pf, want) and _same(sums, expected_sums(want))
    assert (want[:, 8] > 0).all()


@gpu
def test_oracle_subset(dtfill_lib, pool):
    for beams in (64, 16):
        p = pool[beams]
        idx = _pairs(6)
        pf, _ = evaluation.evaluate_fill_png_files([p["lf"][i] for i, _ in idx], [p["gf"][j] for _, j in idx])
        for b, (i, j) in enumerate(idx):
            want = oracle_row(p["lf"][i], p["gf"][j])
            assert _same(pf[b], want), (beams, b, pf[b], want)
            assert _same(expected_row(p["lf"][i], p["gf"][j]), want)


@gpu
def test_edge_ground_truth(dtfill_lib, pool):
    """A ground truth with no valid pixel gives numpy's mean of an empty array (NaN metrics, count 0); samples 0 and 2
    are not valid (2/256 <= 0.01), 3 and 65535 are."""
    p = pool[64]
    rng = np.random.default_rng(7)
    lid = [p["lid"][i] for i in range(6)]
    gt = [p["gt"][i] for i in range(6)]
    gt[1] = np.zeros_like(gt[1])
    gt[2] = np.where(rng.random(gt[2].shape) < 0.3, np.uint16(2), np.uint16(0))           # nothing valid either
    gt[3] = rng.choice(np.array([0, 2, 3, 65535], np.uint16), gt[3].shape)
    gt[4] = np.where(gt[4] > 0, np.uint16(3), np.uint16(0))
    lf, gf = [P.encode(x) for x in lid], [P.encode(x) for x in gt]
    with np.errstate(all="ignore"):
        want = np.stack([expected_row(a, b) for a, b in zip(lid, gt)])
        pf, sums = evaluation.evaluate_fill_png_files(lf, gf)
        assert _same(pf, want) and _same(sums, expected_sums(want))
        for b in (1, 2):
            assert np.isnan(pf[b, :5]).all() and pf[b, 8] == 0
            assert _same(pf[b], oracle_row(lid[b], gt[b]))
        assert _same(pf[3], oracle_row(lid[3], gt[3])) and _same(pf[4], oracle_row(lid[4], gt[4]))
    assert np.isnan(sums[:5]).all() and sums[9] == 6


def _batch(p, n):
    return [p["lf"][i] for i in range(n)], [p["gf"][i] for i in range(n)]


def _check_recovers(p, h=None):
    """After an error the handle gives the right results again."""
    lf, gf = _batch(p, 5)
    want = _rows(p, [(i, i) for i in range(5)])
    if h is None:
        pf, sums = evaluation.evaluate_fill_png_files(lf, gf)
    else:
        data, off = _pack(lf + gf)
        pf, sums = h.eval_png(data, off[:6], data, off[5:], synth.KITTI_H, synth.KITTI_W, 0.1, 0.1)
    assert _same(pf, want) and _same(sums, expected_sums(want))


def _pack(files):
    off = np.zeros(len(files) + 1, np.int64)
    np.cumsum([len(f) for f in files], out=off[1:])
    return np.frombuffer(b"".join(files), np.uint8), off


@gpu
def test_lidar_frames_distance_transform_rejects(dtfill_lib, pool):
    p = pool[64]
    empty = P.encode(np.zeros_like(p["lid"][0]))
    one = np.zeros_like(p["lid"][0])
    one[200, 300] = 5000
    one = P.encode(one)
    for bad, first in (({2: empty}, 2), ({4: one}, 4), ({1: one, 3: empty}, 1), ({1: empty, 3: one}, 1)):
        lf, gf = _batch(p, 6)
        for b, f in bad.items():
            lf[b] = f
        with pytest.raises(IndexError, match=f"LiDAR file {first}:"):
            evaluation.evaluate_fill_png_files(lf, gf)
        with pytest.raises(IndexError):        # the frame the loop stops at
            eval_nyu.Distance_Transform(P.decode(lf[first]).astype(np.float32) / 256, 0.1)
        _check_recovers(p)


@gpu
def test_broken_files(dtfill_lib, pool):
    p = pool[64]
    other = P.encode(gt16(3, 240, 320))
    empty = P.encode(np.zeros_like(p["lid"][0]))
    cases = [
        (dict(lid={3: "cut"}), "LiDAR file 3:"),
        (dict(gt={2: "cut"}), "ground-truth file 2:"),
        (dict(gt={4: other}), "ground-truth file 4: image size differs"),
        (dict(lid={2: "cut"}, gt={2: "cut"}), "LiDAR file 2:"),
        (dict(lid={3: "cut"}, gt={1: "junk"}), "ground-truth file 1:"),
        (dict(lid={0: empty}, gt={3: "cut"}), "ground-truth file 3:"),        # a decode failure wins over IndexError
    ]
    for spec, msg in cases:
        lf, gf = _batch(p, 6)
        for key, files in (("lid", lf), ("gt", gf)):
            for b, how in spec.get(key, {}).items():
                files[b] = files[b][:len(files[b]) // 2] if how == "cut" else (b"\0" * 64 if how == "junk" else how)
        with pytest.raises(ValueError, match=msg):
            evaluation.evaluate_fill_png_files(lf, gf)
        _check_recovers(p)


@gpu
def test_handle_at_pipeline_depth_4_and_link_traffic(dtfill_lib, pool):
    p = pool[16]
    h = _lib.Handle(0)
    try:
        h.set_pipeline_depth(4)
        idx = _pairs(48)
        lf, gf = [p["lf"][i] for i, _ in idx], [p["gf"][j] for _, j in idx]
        data, off = _pack(lf + gf)
        want = _rows(p, idx)
        for _ in range(2):
            pf, sums = h.eval_png(data, off[:49], data, off[48:], synth.KITTI_H, synth.KITTI_W, 0.1, 0.1)
            assert _same(pf, want) and _same(sums, expected_sums(want))
        h2d, d2h = h.transfer_bytes()
        assert data.size <= h2d <= data.size + 16 + 8 * 97
        assert d2h == 48 * (8 + 8 + 72) + 80          # status, counts, rows, sums: no per-pixel data
        _check_recovers(p, h)
    finally:
        h.close()
