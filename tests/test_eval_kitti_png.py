"""eval_nyu.evaluate_fill_kitti_png_files (dtfill_eval_png_kitti): the KITTI branch of eval_NYU.py's loop from the PNG
files,

    lidar = png.astype(np.float32) / 256;  gt = png / 256.;  lidar, gt = lidar[96:], gt[96:]
    pred = relu(Distance_Transform(lidar, 0.001) - 0.9) + 0.9;  Result().evaluate(pred, gt)

per frame, against the same composition of the package's own calls, bit for bit (== with NaN where numpy gives NaN),
and a subset against the CPU oracle; the ground truth as files and as a resident uint16 tensor.  The CPU tests need no
device: the export, the checks that run before the device is touched and the floor's float32 identity.  Run the rest on
the B200 box:  python -m pytest tests -m gpu"""
import numpy as np
import pytest

import png_oracle as P
from distancetransform_depthcompletion_b200 import _lib, eval_nyu, evaluation, synth

CROP = eval_nyu.KITTI_CROP_TOP
BEAMS = (64, 32, 16)
K = 12          # distinct LiDAR frames per beam count and distinct ground-truth frames; larger batches repeat them


# ---- expected values: the script's loop, one frame at a time --------------------------------------------------
def relu(x):
    return np.maximum(x, 0)


def _samples(f):
    return P.decode(f) if isinstance(f, (bytes, bytearray)) else np.asarray(f, np.uint16)


def fill(lidar_file, crop=CROP):
    """png_oracle.decode, the crop and eval_nyu.Distance_Transform at the script's source threshold 0.001."""
    lidar = _samples(lidar_file).astype(np.float32) / 256
    return eval_nyu.Distance_Transform(lidar[crop:], 0.001)


def floored(pred):
    """eval_NYU.py:202-206 as written, in float32."""
    out = relu(pred - 0.9) + 0.9
    assert out.dtype == np.float32
    return out


def score(pred, gt_file, crop=CROP):
    gt = _samples(gt_file)[crop:] / 256.
    r = evaluation.Result()
    r.evaluate(pred, gt)
    n = int(np.logical_and(pred > 0.01, gt > 0.01).sum())
    return np.array([r.mse, r.rmse, r.mae, r.irmse, r.imae, 0, 0, 0, n], np.float64)


def expected_row(lidar_file, gt_file, crop=CROP, floor=True):
    pred = fill(lidar_file, crop)
    return score(floored(pred) if floor else pred, gt_file, crop)


def expected_sums(rows):
    """The running sums the loop keeps (eval_NYU.py:233-254 `+=`, frame after frame), then the frame count."""
    s = np.zeros(10, np.float64)
    for r in rows:
        s[:9] += r
    s[9] = len(rows)
    return s


def oracle_row(lidar_file, gt_file, crop=CROP):
    """The same frame through the CPU oracle: oracle.dt_fill + oracle.result_kitti."""
    from oracle import oracle as O
    lidar = _samples(lidar_file).astype(np.float32)[crop:] / 256
    gt = _samples(gt_file)[crop:] / 256.
    pred = floored(O.dt_fill(lidar, 0.001, 0.1)["depth"])
    m = O.result_kitti(pred, gt)
    return np.array([m["mse"], m["rmse"], m["mae"], m["irmse"], m["imae"], 0, 0, 0, m["count"]], np.float64)


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def lidar16(seed, beams=64, H=synth.KITTI_H, W=synth.KITTI_W):
    return np.rint(synth.kitti_frame(seed, H, W, beam_step=64 // beams) * 256).astype(np.uint16)


def gt16(seed, H=synth.KITTI_H, W=synth.KITTI_W):
    return np.rint(synth.kitti_gt(seed, H, W) * 256).astype(np.uint16)


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_symbol_is_exported(dtfill_lib):
    import ctypes
    assert hasattr(ctypes.CDLL(dtfill_lib), "dtfill_eval_png_kitti")
    assert _lib.load().dtfill_eval_png_kitti is not None
    assert _lib.load().dtfill_abi_version() == _lib.ABI_VERSION
    assert callable(eval_nyu.evaluate_fill_kitti_png_files)


def test_library_without_the_symbol_asks_for_a_rebuild(dtfill_lib, monkeypatch):
    """A build of the same ABI version from before the entry existed fails to load with the rebuild message."""
    import ctypes
    real = ctypes.CDLL(dtfill_lib)

    class Older:
        def __getattr__(self, name):
            if name == "dtfill_eval_png_kitti":
                raise AttributeError(name)
            return getattr(real, name)
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib.ctypes, "CDLL", lambda path: Older())
    with pytest.raises(_lib.DTFillError, match="rebuild it"):
        _lib.load()


def test_floor_is_fmax_on_every_png_sample():
    """relu(pred - 0.9) + 0.9 in float32 equals max(pred, 0.9f) bit for bit on every value the fill can give from PNG
    samples (s / 256, s in 0..65535), so the kernel floors with fmaxf."""
    x = np.arange(65536, dtype=np.uint32).astype(np.float32) / 256
    assert x.dtype == np.float32
    a = floored(x)
    b = np.maximum(x, np.float32(0.9))
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert (a > 0.01).all()


@pytest.fixture
def no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the device was touched")
    monkeypatch.setattr(_lib, "get_handle", refuse)
    monkeypatch.setattr(_lib, "Handle", refuse)


def test_argument_checks_raise_before_the_device(no_device):
    import torch
    f = P.encode(np.zeros((10, 5), np.uint16))
    run = eval_nyu.evaluate_fill_kitti_png_files
    with pytest.raises(ValueError, match="no files"):
        run([], [])
    with pytest.raises(ValueError, match="no files"):
        run([f], [])
    with pytest.raises(ValueError, match="no files"):
        run([], torch.zeros((0, 10, 5), dtype=torch.uint16))
    with pytest.raises(ValueError, match="2 LiDAR files but 3 ground-truth files"):
        run([f, f], [f, f, f])
    with pytest.raises(ValueError, match="LiDAR file 0"):
        run([b"not a png at all, but long enough"], [f])
    with pytest.raises(ValueError, match="LiDAR file 0"):
        run([f[:20]], [f])
    for crop in (-1, 10, 11):
        with pytest.raises(ValueError, match="crop_top"):
            run([f], [f], crop_top=crop)
        with pytest.raises(ValueError, match="crop_top"):
            run([f], torch.zeros((1, 10, 5), dtype=torch.uint16), crop_top=crop)
    for shape in ((2, 10, 5), (1, 10, 6), (1, 9, 5), (10, 5), (1, 1, 10, 5)):
        with pytest.raises(ValueError, match="shape"):
            run([f], torch.zeros(shape, dtype=torch.uint16), crop_top=2)
    for dtype in (torch.int16, torch.int32, torch.float32):
        with pytest.raises(TypeError, match="uint16"):
            run([f], torch.zeros((1, 10, 5), dtype=dtype), crop_top=2)
    with pytest.raises(TypeError, match="CUDA"):
        run([f], torch.zeros((1, 10, 5), dtype=torch.uint16), crop_top=2)


# ---- GPU ----------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def pool():
    """K LiDAR frames per beam count (index beam_index * K + i) and K ground-truth frames of KITTI size, encoded at zlib
    level 6; the filled LiDAR frames and the expected rows cached."""
    lid = [lidar16(s, beams) for beams in BEAMS for s in range(K)]
    gt = [gt16(1000 + s) for s in range(K)]
    return dict(lid=lid, gt=gt, lf=[P.encode(x) for x in lid], gf=[P.encode(x) for x in gt], pred={}, rows={})


def _rows(p, idx):
    rows = []
    for i, j in idx:
        if (i, j) not in p["rows"]:
            if i not in p["pred"]:
                p["pred"][i] = floored(fill(p["lid"][i]))
            p["rows"][(i, j)] = score(p["pred"][i], p["gt"][j])
        rows.append(p["rows"][(i, j)])
    return np.stack(rows)


def _pairs(B):
    """(LiDAR, ground truth) of frame b: the batch mixes 64, 32 and 16 beams."""
    n = len(BEAMS) * K
    return [(b % n, (b // n + 5 * b + 3) % K) for b in range(B)]


def _files(p, idx):
    return [p["lf"][i] for i, _ in idx], [p["gf"][j] for _, j in idx]


@gpu
@pytest.mark.parametrize("B", [1, 5, 256, 1000])
def test_rows_and_sums_bit_exact(dtfill_lib, pool, B):
    idx = _pairs(B)
    pf, sums = eval_nyu.evaluate_fill_kitti_png_files(*_files(pool, idx))
    want = _rows(pool, idx)
    assert pf.dtype == np.float64 and pf.shape == (B, 9) and sums.shape == (10,)
    for b in range(B):
        assert _same(pf[b], want[b]), (b, pf[b], want[b])
    assert _same(sums, expected_sums(want))
    assert (want[:, 8] > 0).all()


@gpu
def test_oracle_subset(dtfill_lib, pool):
    idx = [(BEAMS.index(beams) * K + i, (i + 2) % K) for beams in BEAMS for i in range(2)]
    pf, _ = eval_nyu.evaluate_fill_kitti_png_files(*_files(pool, idx))
    for b, (i, j) in enumerate(idx):
        want = oracle_row(pool["lid"][i], pool["gt"][j])
        assert _same(pf[b], want), (b, pf[b], want)
        assert _same(_rows(pool, [(i, j)])[0], want)


@gpu
@pytest.mark.parametrize("crop", [CROP, 0])
def test_odd_width(dtfill_lib, crop):
    H, W = synth.KITTI_H, 621
    lid = [lidar16(s, BEAMS[s % 3], H, W) for s in range(6)]
    gt = [gt16(70 + s, H, W) for s in range(6)]
    pf, sums = eval_nyu.evaluate_fill_kitti_png_files([P.encode(x) for x in lid], [P.encode(x) for x in gt], crop)
    want = np.stack([expected_row(a, g, crop) for a, g in zip(lid, gt)])
    assert _same(pf, want) and _same(sums, expected_sums(want))


@gpu
def test_shifted_labels_and_the_floor(dtfill_lib, pool):
    """Samples 26..255 are valid but not sources at 0.001 (a source needs s >= 256), so Distance_Transform's labels shift
    (SURVEY.md Appendix B) and the fill copies depths below 0.9 m, which the floor raises.  A frame whose valid samples
    are all below 256 has no source and is filled with its last valid depth."""
    rng = np.random.default_rng(5)
    lid, gt = [], []
    for b in range(6):
        x = pool["lid"][b].copy()
        near = rng.random(x.shape) < 0.02
        x[near] = rng.integers(1, 256, int(near.sum()))
        lid.append(x)
        gt.append(pool["gt"][(2 * b + 1) % K])
    below = np.where(pool["lid"][7] > 0, rng.integers(26, 231, pool["lid"][7].shape), 0).astype(np.uint16)
    lid.append(below)
    gt.append(pool["gt"][3])
    pf, sums = eval_nyu.evaluate_fill_kitti_png_files([P.encode(x) for x in lid], [P.encode(x) for x in gt])
    want = np.stack([expected_row(a, g) for a, g in zip(lid, gt)])
    assert _same(pf, want) and _same(sums, expected_sums(want))
    pred = fill(below)
    assert (pred < 0.9).all() and np.unique(pred).size == 1           # the last valid depth, below the floor
    unfloored = np.stack([expected_row(a, g, floor=False) for a, g in zip(lid, gt)])
    assert not _same(unfloored[-1], want[-1])
    assert sum(not _same(unfloored[b], want[b]) for b in range(6)) > 0
    assert _same(pf[-1], oracle_row(lid[-1], gt[-1]))


@gpu
def test_ground_truth_without_valid_samples(dtfill_lib, pool):
    """Ground truth all <= 2 (2/256 <= 0.01) in the cropped rows: numpy's mean of an empty array (NaN, count 0); valid
    samples above the crop do not count."""
    lf, _ = _files(pool, _pairs(4))
    gt = [pool["gt"][i].copy() for i in range(4)]
    gt[1][CROP:] = np.minimum(gt[1][CROP:], 2)
    gt[2][CROP:] = 0
    gt[2][:CROP] = 5000
    with np.errstate(all="ignore"):
        want = np.stack([expected_row(a, g) for a, g in zip(lf, gt)])
        pf, sums = eval_nyu.evaluate_fill_kitti_png_files(lf, [P.encode(x) for x in gt])
        assert _same(pf, want) and _same(sums, expected_sums(want))
        for b in (1, 2):
            assert np.isnan(pf[b, :5]).all() and pf[b, 8] == 0
            assert _same(pf[b], oracle_row(lf[b], gt[b]))
    assert np.isnan(sums[:5]).all() and sums[9] == 4


def _check_recovers(p):
    idx = _pairs(5)
    pf, sums = eval_nyu.evaluate_fill_kitti_png_files(*_files(p, idx))
    want = _rows(p, idx)
    assert _same(pf, want) and _same(sums, expected_sums(want))


@gpu
def test_lidar_frames_distance_transform_rejects(dtfill_lib, pool):
    """No valid sample, or exactly one, in the cropped rows: IndexError at that frame, also when the frame's other points
    lie in the rows the crop drops."""
    x = pool["lid"][0]
    empty = P.encode(np.zeros_like(x))
    above = np.zeros_like(x)
    above[8:CROP:8, ::4] = 3000             # points only in the rows the crop drops
    one = above.copy()
    one[200, 300] = 5000
    above, one = P.encode(above), P.encode(one)
    for bad, first in (({2: empty}, 2), ({3: above}, 3), ({4: one}, 4), ({1: one, 3: empty}, 1), ({1: above, 3: one}, 1)):
        lf, gf = _files(pool, _pairs(6))
        for b, f in bad.items():
            lf[b] = f
        with pytest.raises(IndexError, match=f"LiDAR file {first}:"):
            eval_nyu.evaluate_fill_kitti_png_files(lf, gf)
        with pytest.raises(IndexError):        # the frame the loop stops at
            fill(lf[first])
        _check_recovers(pool)


@gpu
def test_broken_files(dtfill_lib, pool):
    other = P.encode(gt16(3, 240, 320))
    empty = P.encode(np.zeros_like(pool["lid"][0]))
    cases = [
        (dict(lid={3: "cut"}), "LiDAR file 3:"),
        (dict(gt={2: "cut"}), "ground-truth file 2:"),
        (dict(gt={4: other}), "ground-truth file 4: image size differs"),
        (dict(lid={2: "cut"}, gt={2: "cut"}), "LiDAR file 2:"),
        (dict(lid={1: "junk"}, gt={1: "junk"}), "LiDAR file 1:"),
        (dict(lid={3: "cut"}, gt={1: "junk"}), "ground-truth file 1:"),
        (dict(lid={0: empty}, gt={3: "cut"}), "ground-truth file 3:"),        # a decode failure wins over IndexError
    ]
    for spec, msg in cases:
        lf, gf = _files(pool, _pairs(6))
        for key, files in (("lid", lf), ("gt", gf)):
            for b, how in spec.get(key, {}).items():
                files[b] = files[b][:len(files[b]) // 2] if how == "cut" else (b"\0" * 64 if how == "junk" else how)
        with pytest.raises(ValueError, match=msg):
            eval_nyu.evaluate_fill_kitti_png_files(lf, gf)
        _check_recovers(pool)


def _decoded_on_device(files):
    """The ground-truth files decoded once into a resident uint16 tensor by DTFillEngine.decode_png."""
    import torch
    from distancetransform_depthcompletion_b200.data_read import pack_png_files
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    data, off, H, W = pack_png_files(files)
    eng = DTFillEngine(0)
    samples, status = eng.decode_png(torch.from_numpy(data.copy()).cuda(), torch.from_numpy(off).cuda(), H, W)
    assert (status.cpu().numpy() == 0).all()
    return samples


@gpu
def test_resident_ground_truth_for_three_densities(dtfill_lib, pool):
    """One decoded ground-truth tensor scored against the 64-, 32- and 16-beam LiDAR sets equals the files form row for
    row, and each call moves only the LiDAR files and their offsets up and the metrics down."""
    B = 40
    gj = [(b // K + 5 * b + 3) % K for b in range(B)]
    gf = [pool["gf"][j] for j in gj]
    gt_t = _decoded_on_device(gf)
    assert np.array_equal(gt_t.cpu().numpy(), np.stack([pool["gt"][j] for j in gj]))
    h = _lib.get_handle(0)
    for beams in BEAMS:
        idx = [(BEAMS.index(beams) * K + b % K, j) for b, j in enumerate(gj)]
        lf = [pool["lf"][i] for i, _ in idx]
        pf_f, sums_f = eval_nyu.evaluate_fill_kitti_png_files(lf, gf)
        up_files = h.transfer_bytes()[0]
        pf_r, sums_r = eval_nyu.evaluate_fill_kitti_png_files(lf, gt_t, device=0)
        h2d, d2h = h.transfer_bytes()
        want = _rows(pool, idx)
        assert _same(pf_r, pf_f) and _same(sums_r, sums_f) and _same(pf_r, want)
        nbytes = sum(len(f) for f in lf)
        assert h2d == ((nbytes + 15) & ~15) + 8 * (B + 1)
        assert up_files == ((nbytes + sum(len(f) for f in gf) + 15) & ~15) + 8 * (2 * B + 1)
        assert d2h == B * (4 + 8 + 72) + 80          # status, counts, rows, sums: no per-pixel data
    # the tensor is read in place, not consumed
    assert np.array_equal(gt_t.cpu().numpy(), np.stack([pool["gt"][j] for j in gj]))


@gpu
def test_resident_ground_truth_errors(dtfill_lib, pool):
    idx = _pairs(6)
    lf, gf = _files(pool, idx)
    gt_t = _decoded_on_device(gf)
    with pytest.raises(ValueError, match="device=1"):
        eval_nyu.evaluate_fill_kitti_png_files(lf, gt_t, device=1)
    bad = list(lf)
    bad[2] = bad[2][:len(bad[2]) // 2]
    with pytest.raises(ValueError, match="LiDAR file 2:"):
        eval_nyu.evaluate_fill_kitti_png_files(bad, gt_t)
    bad = list(lf)
    bad[4] = P.encode(np.zeros_like(pool["lid"][0]))
    with pytest.raises(IndexError, match="LiDAR file 4:"):
        eval_nyu.evaluate_fill_kitti_png_files(bad, gt_t)
    pf, sums = eval_nyu.evaluate_fill_kitti_png_files(lf, gt_t)        # and recovers
    want = _rows(pool, idx)
    assert _same(pf, want) and _same(sums, expected_sums(want))
