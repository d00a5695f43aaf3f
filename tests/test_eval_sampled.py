"""eval_nyu.evaluate_fill_sampled (dtfill_eval_sampled): the NYU script's loop from dense ground truth,

    Mask = zeros(H, W); Mask[rows, cols] = 1; pred = Distance_Transform(gt * Mask); Result_NYU().evaluate(crop(pred), crop(gt))

per frame, against the same composition of the package's own calls, bit for bit (== with NaN where numpy gives NaN),
and a subset against the CPU oracle.  The CPU tests need no device: the export, the sampling expression and the checks
that run before the device is touched.  Run the rest on the B200 box:  python -m pytest tests -m gpu"""
import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib, eval_nyu, evaluation, synth
from distancetransform_depthcompletion_b200.eval_nyu import NYU_EVAL_CROP, evaluate_fill_sampled, nyu_sample_coords

H, W = 240, 320
NS = [2, 20, 50, 200, 500, 5000]


# ---- expected values: the reference's loop, one frame at a time ---------------------------------------------------
def sparse(gt, rows, cols):
    mask = np.zeros(gt.shape, np.float32)          # data_read.py:360-364; its dtype does not change the product
    mask[rows, cols] = 1
    return gt * mask


def expected_row(gt, rows, cols, crop=NYU_EVAL_CROP, src_thr=eval_nyu.NYU_SRC_THR):
    """One frame of the loop: gt * Mask, eval_nyu.Distance_Transform, crop, Result_NYU.evaluate -> the row of
    evaluate_fill_sampled.  Raises IndexError where Distance_Transform does."""
    pred = eval_nyu.Distance_Transform(sparse(gt, rows, cols), src_thr)
    r0, r1, c0, c1 = crop
    p, t = pred[r0:r1, c0:c1], gt[r0:r1, c0:c1]
    r = evaluation.Result_NYU()
    r.evaluate(p, t)
    n = int(np.logical_and(p > 0.01, t > 0.01).sum())
    return np.array([r.mse, r.rmse, r.mae, r.irmse, r.imae, r.delta1, r.delta2, r.delta3, n], np.float64)


def oracle_row(gt, rows, cols, crop=NYU_EVAL_CROP):
    """The same frame through the CPU oracle: the cv2 port of eval_NYU.py:120-133 + oracle.result_nyu."""
    from oracle import oracle as O
    pred = O.cv2_port_fill_frame(sparse(gt, rows, cols), 0.001, 0.1, nyu_style=True)[0]
    r0, r1, c0, c1 = crop
    m = O.result_nyu(pred[r0:r1, c0:c1], gt[r0:r1, c0:c1])
    return np.array([m[k] for k in ("mse", "rmse", "mae", "irmse", "imae", "delta1", "delta2", "delta3", "count")],
                    np.float64)


def expected_sums(rows):
    s = np.zeros(10, np.float64)
    for r in rows:
        s[:9] += r
    s[9] = len(rows)
    return s


def loop(gt, rows, cols, crop=NYU_EVAL_CROP):
    """The loop over a batch: (rows [B,9], sums), or ("IndexError", frame) where the loop stops."""
    out = []
    for b in range(len(gt)):
        try:
            with np.errstate(all="ignore"):
                out.append(expected_row(gt[b], rows[b], cols[b], crop))
        except IndexError:
            return "IndexError", b
    return np.stack(out), expected_sums(out)


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def _numpy_message(rows, cols, h=H, w=W):
    try:
        np.zeros((h, w), np.float32)[np.asarray(rows), np.asarray(cols)] = 1
    except IndexError as e:
        return str(e)
    raise AssertionError("numpy accepted the coordinates")


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_symbol_is_exported_and_abi_version(dtfill_lib):
    import ctypes
    assert hasattr(ctypes.CDLL(dtfill_lib), "dtfill_eval_sampled")
    assert _lib.ABI_VERSION == 9 and _lib.load().dtfill_abi_version() == 9
    assert callable(evaluate_fill_sampled)


@pytest.mark.parametrize("seed", [0, 1, 42, 2024])
@pytest.mark.parametrize("n", [0, 1, 20, 50, 200, 500])
def test_nyu_sample_coords_is_the_quoted_expression(seed, n):
    np.random.seed(seed)
    want = np.zeros((H, W))
    want[np.random.randint(H - 12, size=n) + 6, np.random.randint(W - 16, size=n) + 8] = 1      # SURVEY.md a-7
    after = np.random.randint(1 << 30)
    np.random.seed(seed)
    rows, cols = nyu_sample_coords(n)
    got = np.zeros((H, W))
    got[rows, cols] = 1
    assert np.array_equal(got, want) and np.random.randint(1 << 30) == after
    rs = np.random.RandomState(seed)
    r2, c2 = nyu_sample_coords(n, rng=rs)
    assert np.array_equal(r2, rows) and np.array_equal(c2, cols)
    assert ((rows >= 6) & (rows < H - 6)).all() and ((cols >= 8) & (cols < W - 8)).all()


@pytest.fixture
def no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the device was touched")
    monkeypatch.setattr(_lib, "get_handle", refuse)
    monkeypatch.setattr(_lib, "Handle", refuse)


def test_argument_checks_raise_before_the_device(no_device):
    gt = np.ones((3, H, W), np.float32)
    r = [np.array([10, 20]), np.array([30]), np.array([40, 50, 60])]
    c = [np.array([10, 20]), np.array([30]), np.array([40, 50, 60])]
    for bad in (gt.astype(np.float64), gt.astype(np.float16), gt.astype(np.int32)):
        with pytest.raises(TypeError):
            evaluate_fill_sampled(bad, r, c)
    with pytest.raises(ValueError, match="empty batch"):
        evaluate_fill_sampled(np.ones((0, H, W), np.float32), [], [])
    with pytest.raises(ValueError, match="3 frames but 2 rows"):
        evaluate_fill_sampled(gt, r[:2], c)
    with pytest.raises(ValueError, match="3 frames but 3 rows and 4 cols"):
        evaluate_fill_sampled(gt, r, c + [np.array([1])])
    with pytest.raises(ValueError, match="frame 1 has 1 rows but 2 cols"):
        evaluate_fill_sampled(gt, r, [c[0], np.array([1, 2]), c[2]])
    with pytest.raises(ValueError, match="must be \\[B,H,W\\]"):
        evaluate_fill_sampled(gt[0], r[0], c[0])
    for crop in ((6, 241, 8, 312), (-1, 234, 8, 312), (6, 234, 8, 321), (6, 6, 8, 312), (6, 234, 300, 8)):
        with pytest.raises(ValueError, match="not a non-empty window"):
            evaluate_fill_sampled(gt, r, c, crop=crop)
    with pytest.raises(IndexError, match="integer"):
        evaluate_fill_sampled(gt, [np.array([1.0, 2.0])] + r[1:], c)
    # an empty float array is refused as numpy refuses it (an empty list is an empty index, tested below)
    with pytest.raises(IndexError) as e:
        evaluate_fill_sampled(gt, [np.array([])] + r[1:], [np.array([])] + c[1:])
    assert str(e.value) == _numpy_message(np.array([]), np.array([]))
    # coordinates outside the frame: numpy's message, first frame first, rows before columns within a frame
    cases = [
        ([np.array([10, 240])] + r[1:], c, (np.array([10, 240]), c[0])),
        (r, [np.array([10, 320])] + c[1:], (r[0], np.array([10, 320]))),
        (r, [c[0], np.array([-321]), c[2]], (r[1], np.array([-321]))),
        ([r[0], np.array([-241]), r[2]], c, (np.array([-241]), c[1])),
        ([r[0], r[1], np.array([1, 2, 999])], [c[0], np.array([400]), c[2]], (r[1], np.array([400]))),
        ([r[0], np.array([300]), r[2]], [c[0], np.array([400]), c[2]], (np.array([300]), np.array([400]))),
    ]
    for rows, cols, (nr, nc) in cases:
        msg = _numpy_message(nr, nc)
        with pytest.raises(IndexError) as e:
            evaluate_fill_sampled(gt, rows, cols)
        assert str(e.value) == msg
    assert _numpy_message([240], [0]) == "index 240 is out of bounds for axis 0 with size 240"


def test_sample_arrays_wrap_and_layout():
    rows = [np.array([-1, 0, -240]), np.array([], np.int64), np.array([5])]
    cols = [np.array([-320, 319, 3]), np.array([], np.int64), np.array([-1])]
    r, c, off = eval_nyu._sample_arrays(rows, cols, 3, H, W)
    assert r.dtype == np.int32 and c.dtype == np.int32 and off.dtype == np.int64
    assert off.tolist() == [0, 3, 3, 4]
    assert r.tolist() == [239, 0, 0, 5] and c.tolist() == [0, 319, 3, 319]
    r, c, off = eval_nyu._sample_arrays([[], [7, -2]], [[], [1, 2]], 2, H, W)
    assert off.tolist() == [0, 0, 2] and r.tolist() == [7, 238] and c.tolist() == [1, 2]
    r, c, off = eval_nyu._sample_arrays(np.array([[1, 2], [3, 4]]), np.array([[5, 6], [7, 8]]), 2, H, W)
    assert off.tolist() == [0, 2, 4] and r.tolist() == [1, 2, 3, 4] and c.tolist() == [5, 6, 7, 8]


# ---- GPU ----------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
K = 16          # distinct ground-truth frames per size; larger batches repeat them with other draws
P = 64          # distinct (ground truth, draw) pairs; larger batches repeat them


def _draw(p, n, h=H, w=W):
    """Draw p of n samples: the reference's sampler; n = 2 redrawn until both samples differ (one valid depth is an
    IndexError, tested on its own)."""
    rs = np.random.RandomState(1000 + p)
    while True:
        rows, cols = nyu_sample_coords(n, h, w, rng=rs)
        if n != 2 or (rows[0], cols[0]) != (rows[1], cols[1]):
            return rows, cols


@pytest.fixture(scope="module")
def pool():
    gts = np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(K)])
    pairs = []
    for p in range(P):
        n = NS[p % len(NS)]
        rows, cols = _draw(p, n)
        pairs.append(dict(g=p % K, rows=rows, cols=cols, row=None))
    return dict(gt=gts, pairs=pairs)


def _batch(pool, B):
    idx = [b % P for b in range(B)]
    gt = np.ascontiguousarray(pool["gt"][[pool["pairs"][i]["g"] for i in idx]])
    rows = [pool["pairs"][i]["rows"] for i in idx]
    cols = [pool["pairs"][i]["cols"] for i in idx]
    want = []
    for i in idx:
        q = pool["pairs"][i]
        if q["row"] is None:
            q["row"] = expected_row(pool["gt"][q["g"]], q["rows"], q["cols"])
        want.append(q["row"])
    return gt, rows, cols, np.stack(want)


@gpu
@pytest.mark.parametrize("B", [1, 7, 654, 2048])
def test_rows_and_sums_bit_exact(dtfill_lib, pool, B):
    gt, rows, cols, want = _batch(pool, B)
    pf, sums = evaluate_fill_sampled(gt, rows, cols)
    assert pf.dtype == np.float64 and pf.shape == (B, 9) and sums.shape == (10,)
    for b in range(B):
        assert _same(pf[b], want[b]), (b, len(rows[b]), pf[b], want[b])
    assert _same(sums, expected_sums(want))
    assert (want[:, 8] > 0).all()


@gpu
@pytest.mark.parametrize("n", NS)
def test_equal_counts_as_one_array(dtfill_lib, pool, n):
    """[B,n] arrays (every frame n samples; n = 5000 draws many duplicates) give what per-frame lists give."""
    B = 9
    draws = [_draw(500 + b, n) for b in range(B)]
    rows, cols = np.stack([d[0] for d in draws]), np.stack([d[1] for d in draws])
    gt = pool["gt"][:B]
    if n == 5000:
        assert all(len(set(zip(r.tolist(), c.tolist()))) < n for r, c in draws)
    want, wsums = loop(gt, rows, cols)
    pf, sums = evaluate_fill_sampled(gt, rows, cols)
    assert _same(pf, want) and _same(sums, wsums)
    pf2, _ = evaluate_fill_sampled(gt, list(rows), list(cols))
    assert _same(pf2, pf)


@gpu
def test_oracle_subset(dtfill_lib, pool):
    gt, rows, cols, want = _batch(pool, 12)
    pf, _ = evaluate_fill_sampled(gt, rows, cols)
    for b in range(12):
        o = oracle_row(gt[b], rows[b], cols[b])
        assert _same(pf[b], o), (b, pf[b], o)
        assert _same(want[b], o)


@gpu
@pytest.mark.parametrize("crop", [NYU_EVAL_CROP, (0, 480, 0, 640), (100, 101, 0, 640), (0, 480, 639, 640)])
def test_480x640(dtfill_lib, crop):
    """BASELINE configs[3]'s frame size with the script's literal crop, the full frame and one-pixel-wide windows."""
    h, w = 480, 640
    B = 6
    gt = np.stack([synth.nyu_frame(30 + s, h, w, return_dense=True)[1] for s in range(B)])
    draws = [_draw(700 + b, NS[b % len(NS)], h, w) for b in range(B)]
    rows, cols = [d[0] for d in draws], [d[1] for d in draws]
    want, wsums = loop(gt, rows, cols, crop)
    pf, sums = evaluate_fill_sampled(gt, rows, cols, crop=crop)
    assert _same(pf, want) and _same(sums, wsums)


@gpu
def test_crop_edges_outside_the_crop_and_wrapping(dtfill_lib, pool):
    gt = pool["gt"][:6]
    edge_r = np.array([6, 233, 234, 5, 0, 239, 6, 233, 120, 120])
    edge_c = np.array([8, 311, 312, 7, 0, 319, 311, 8, 8, 311])
    rows = [edge_r, edge_r[2:6], np.array([-1, -240, -6, 100]), np.array([-234, 0, -1]), edge_r, np.array([0, 239])]
    cols = [edge_c, edge_c[2:6], np.array([-1, -320, -8, 100]), np.array([-312, -320, 7]), edge_c[::-1], np.array([0, 319])]
    want, wsums = loop(gt, rows, cols)
    pf, sums = evaluate_fill_sampled(gt, rows, cols)
    assert _same(pf, want) and _same(sums, wsums)
    # the wrapped coordinates are the same samples as their positive forms
    pos_r = [np.where(r < 0, r + H, r) for r in rows]
    pos_c = [np.where(c < 0, c + W, c) for c in cols]
    assert _same(evaluate_fill_sampled(gt, pos_r, pos_c)[0], pf)


EDGE_SAMPLED = np.array([-1.5, -0.0, 0.0, np.inf, -np.inf, 3e-39, -3e-39, 1e-45, 0.001, 0.0011, 0.05, 0.0099999, 0.01,
                         0.0100001, 0.1, 0.1000001, 0.5, 0.999, 1.0], np.float32)
EDGE_UNSAMPLED = np.array([-1.5, -1e30, -0.0, 0.0, 3e-39, -3e-39, -1e-45, 0.001, 0.0011, 0.05, 0.0099999, 0.01, 0.0100001,
                           0.1, 0.1000001, 0.5], np.float32)
NONFINITE = np.array([np.nan, np.inf, -np.inf], np.float32)


def _edge_frame(seed, n=500, nonfinite=0, h=H, w=W):
    """(gt, rows, cols): synthetic depths sampled by the reference's sampler, with every value of EDGE_SAMPLED at sampled
    pixels and every value of EDGE_UNSAMPLED at unsampled ones, spread over the whole frame (inside and outside the crop).
    With nonfinite > 0 that many unsampled pixels hold NaN / +inf / -inf (gt * Mask makes them NaN: sources that are no
    valid depth) and a few sampled ones hold NaN; as many extra samples of 0.5 (a valid depth that is no source) keep the
    labels within the list of valid depths, so the frame is filled and scored instead of raising IndexError."""
    rng = np.random.default_rng(seed)
    g = synth.nyu_frame(seed, h, w, return_dense=True)[1].copy()
    rows, cols = _draw(seed, n, h, w)
    taken = np.zeros((h, w), bool)
    taken[rows, cols] = True
    pick = rng.permutation(np.flatnonzero(~taken))
    ks, ku, kn = 5 * EDGE_SAMPLED.size, 8 * EDGE_UNSAMPLED.size, nonfinite
    nan_s = 3 if nonfinite else 0
    ps, pu, pn = pick[:ks], pick[ks:ks + ku], pick[ks + ku:ks + ku + kn]
    pnan = pick[ks + ku + kn:ks + ku + kn + nan_s]
    pv = pick[ks + ku + kn + nan_s:ks + ku + 2 * (kn + nan_s)]
    flat = g.reshape(-1)
    flat[ps] = np.resize(EDGE_SAMPLED, ks)
    flat[pu] = np.resize(EDGE_UNSAMPLED, ku)
    flat[pn] = np.resize(NONFINITE, kn)
    flat[pnan] = np.nan
    flat[pv] = 0.5
    extra = np.concatenate([ps, pnan, pv, ps[:7]])          # a few samples twice
    return g, np.concatenate([rows, extra // w]), np.concatenate([cols, extra % w])


def _same_bits(a, b):
    """Bit for bit, except that a NaN matches a NaN: NaN at the same pixels, every other value with its sign and bits.
    (The sign and payload of the NaN that g * 0 gives for g = +-inf belong to the hardware -- x86 returns 0xFFC00000,
    CUDA 0x7FFFFFFF -- and no reference line can observe them.)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def _check_filled_and_scored(frames, h=H, w=W, crop=NYU_EVAL_CROP):
    """The batch through Handle.eval_sampled with the sparse frames: every frame is filled and scored by the loop (no
    IndexError), out_lidar equals gt * Mask bit for bit (_same_bits), rows and sums equal the loop's."""
    gt = np.stack([f[0] for f in frames])
    rows, cols = [f[1] for f in frames], [f[2] for f in frames]
    want = loop(gt, rows, cols, crop)
    assert not isinstance(want[0], str), want           # the frames reach the comparisons below
    r, c, off = eval_nyu._sample_arrays(rows, cols, len(frames), h, w)
    pf, sums, lid = _lib.get_handle().eval_sampled(gt, len(frames), h, w, r, c, off, crop, 0.001, 0.1, want_lidar=True)
    for b in range(len(frames)):
        assert _same_bits(lid[b], sparse(gt[b], rows[b], cols[b])), b
        assert _same(pf[b], want[0][b]), (b, pf[b], want[0][b])
    assert _same(sums, want[1])
    return gt, lid, pf


@gpu
def test_edge_values_sparse_frame_and_rows(dtfill_lib):
    """out_lidar equals gt * Mask bit for bit: -0 for a negative g and for -0, +0 for +0, the value itself at sampled
    pixels (+-inf, denormals, (0.001, 0.1], around 0.01), NaN for NaN / +-inf at unsampled pixels; and each frame's row
    equals the loop's.  Every frame here is one the loop fills and scores."""
    frames = [_edge_frame(60 + s, n=[20, 200, 500, 5000, 50][s % 5], nonfinite=[0, 12][s % 2]) for s in range(10)]
    gt, lid, pf = _check_filled_and_scored(frames)
    for b, (g, rows, cols) in enumerate(frames):
        sampled = np.zeros((H, W), bool)
        sampled[rows, cols] = True
        neg = ~sampled & np.signbit(g) & np.isfinite(g)
        assert neg.sum() >= 5 * 8 and (lid[b][neg] == 0).all() and np.signbit(lid[b][neg]).all(), b
        pos0 = ~sampled & (g == 0) & ~np.signbit(g)
        assert pos0.any() and not np.signbit(lid[b][pos0]).any(), b
        nonfin = ~sampled & ~np.isfinite(g)
        assert nonfin.sum() == [0, 12][b % 2] and np.isnan(lid[b][nonfin]).all(), b
        spec = sampled & (~np.isfinite(g) | (g <= 0.1) | (g == 0.5))
        assert spec.sum() >= EDGE_SAMPLED.size * 3 and _same_bits(lid[b][spec], g[spec])
    assert (pf[:, 8] > 0).all()
    # the same batch through the public call
    rows, cols = [f[1] for f in frames], [f[2] for f in frames]
    pf2, _ = evaluate_fill_sampled(gt, rows, cols)
    assert _same(pf2, pf)


def _nan_gt(seed):
    """Dense ground truth with NaN, +-inf, negatives, +-0 and small values on 5 % of the pixels: hundreds of NaN sources
    in gt * Mask, more than the valid depths, so Distance_Transform rejects the frame."""
    rng = np.random.default_rng(seed)
    g = synth.nyu_frame(seed, H, W, return_dense=True)[1].copy()
    specials = np.array([np.nan, np.inf, -np.inf, -1.5, -0.0, 0.0, 0.001, 0.0011, 0.05, 0.1, 0.1000001, 0.0099999,
                         0.01, 0.0100001, 3e-39, -3e-39], np.float32)
    sel = rng.random((H, W)) < 0.05
    g[sel] = rng.choice(specials, int(sel.sum()))
    return g


@gpu
def test_nan_sources_give_the_loops_index_error(dtfill_lib):
    """NaN / +-inf at unsampled pixels become NaN sources (tools.py:8): with more of them than valid depths the loop
    raises IndexError, and so does the call, at the same frame; the handle stays usable."""
    good = [_edge_frame(80 + s, nonfinite=12) for s in range(2)]
    bad = []
    for s in range(4):
        g = _nan_gt(60 + s)
        rows, cols = _draw(900 + s, [20, 500][s % 2])
        assert loop(g[None], [rows], [cols]) == ("IndexError", 0)
        with pytest.raises(IndexError, match="frame 0:"):
            evaluate_fill_sampled(g[None], [rows], [cols])
        bad.append((g, rows, cols))
    frames = good + bad
    gt = np.stack([f[0] for f in frames])
    rows, cols = [f[1] for f in frames], [f[2] for f in frames]
    assert loop(gt, rows, cols) == ("IndexError", 2)
    with pytest.raises(IndexError, match="frame 2:"):
        evaluate_fill_sampled(gt, rows, cols)
    _check_filled_and_scored(good)


@gpu
@pytest.mark.parametrize("w", [324, 322])
def test_widths_of_the_other_k1_instances(dtfill_lib, w):
    """W = 324 (a multiple of 4, not of 16: k1_mask_rows_v16<SampledGt, false>) and W = 322 (the scalar k1_mask_rows)."""
    frames = [_edge_frame(120 + s, n=[50, 500, 2000][s % 3], nonfinite=[0, 12][s % 2], w=w) for s in range(5)]
    _check_filled_and_scored(frames, w=w)
    _check_filled_and_scored(frames, w=w, crop=(0, H, 0, w))


@gpu
def test_zero_and_one_sample(dtfill_lib, pool):
    gt, rows, cols, want = _batch(pool, 8)
    for spec, first in (({3: 1}, 3), ({5: 0}, 5), ({2: 0, 4: 1}, 2), ({6: 1, 1: 0}, 1)):
        r, c = list(rows), list(cols)
        for b, n in spec.items():
            r[b], c[b] = rows[b][:n], cols[b][:n]
        assert loop(gt, r, c) == ("IndexError", first)
        with pytest.raises(IndexError, match=f"frame {first}:"):
            evaluate_fill_sampled(gt, r, c)
        pf, sums = evaluate_fill_sampled(gt, rows, cols)          # the handle recovers
        assert _same(pf, want) and _same(sums, expected_sums(want))


@gpu
def test_resident_ground_truth_16_draws(dtfill_lib, pool):
    import torch
    B = 654
    gt = np.ascontiguousarray(np.stack([pool["gt"][b % K] for b in range(B)]))
    gt_t = torch.from_numpy(gt).cuda()
    h = _lib.get_handle(0)
    for n in (20, 500):
        for d in range(8):
            rs = np.random.RandomState(10 * n + d)
            draws = [nyu_sample_coords(n, rng=rs) for _ in range(B)]
            rows, cols = [x[0] for x in draws], [x[1] for x in draws]
            pf_d, sums_d = evaluate_fill_sampled(gt_t, rows, cols)
            h2d, d2h = h.transfer_bytes()
            pf_h, sums_h = evaluate_fill_sampled(gt, rows, cols)
            assert _same(pf_d, pf_h) and _same(sums_d, sums_h), (n, d)
            coords = ((8 * B * n + 15) // 16) * 16 + 8 * (B + 1)
            assert h2d == coords, (h2d, coords)                          # no ground truth went up
            assert d2h == B * (8 + 72) + 4 + 80
            assert h.transfer_bytes()[0] == coords + gt.nbytes          # the host call uploads it
    b = 5
    assert _same(pf_d[b], expected_row(gt[b], rows[b], cols[b]))
    with pytest.raises(ValueError, match="device=1 but the ground truth is on cuda:0"):
        evaluate_fill_sampled(gt_t, rows, cols, device=1)
    assert torch.equal(gt_t.cpu(), torch.from_numpy(gt))                 # used in place, untouched


@gpu
def test_engine_at_pipeline_depth_4(dtfill_lib, pool):
    import torch
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    gt, rows, cols, want = _batch(pool, 96)
    gt_t = torch.from_numpy(gt).cuda()
    eng = DTFillEngine(0, pipeline_depth=4)
    try:
        x = torch.from_numpy(synth.nyu_batch(range(64))).cuda()
        for _ in range(2):
            for _ in range(6):                                          # fills in flight on all four lanes
                eng.fill(x)
            pf, sums = eng.eval_sampled(gt_t, rows, cols)
            assert _same(pf, want) and _same(sums, expected_sums(want))
        # device-resident coordinates
        r, c, off = eval_nyu._sample_arrays(rows, cols, 96, H, W)
        r_t, c_t, off_t = (torch.from_numpy(a).cuda() for a in (r, c, off))
        for _ in range(4):
            eng.fill(x)
        pf, sums, lid = eng.eval_sampled(gt_t, r_t, c_t, off_t, want_lidar=True)
        assert _same(pf, want) and _same(sums, expected_sums(want))
        assert np.array_equal(lid[7].view(np.uint32), sparse(gt[7], rows[7], cols[7]).view(np.uint32))
        # a device coordinate outside the frame is found on the device
        r_bad = r.copy()
        r_bad[off[3] + 1] = H
        with pytest.raises(ValueError, match="frame 3: a sample outside the frame"):
            eng.eval_sampled(gt_t, torch.from_numpy(r_bad).cuda(), c_t, off_t)
        off_bad = off.copy()
        off_bad[5] = off_bad[4] - 1
        off_bad_t = torch.from_numpy(off_bad).cuda()
        with pytest.raises(ValueError, match="frame 4 has a negative sample count"):
            eng.eval_sampled(gt_t, r_t, c_t, off_bad_t)
        with pytest.raises(ValueError, match="frame 4: a sample outside the frame, or a negative sample count"):
            eng.handle.eval_sampled(gt_t.data_ptr(), 96, H, W, r_t.data_ptr(), c_t.data_ptr(), off_bad_t.data_ptr(),
                                    NYU_EVAL_CROP, 0.001, 0.1, gt_is_device=True, coords_are_device=True)
        with pytest.raises(ValueError, match="1 cols"):
            eng.eval_sampled(gt_t, r_t, c_t[:1], off_t)
        off_long = off.copy()
        off_long[-1] += 1
        with pytest.raises(ValueError, match="offsets span"):
            eng.eval_sampled(gt_t, r_t, c_t, torch.from_numpy(off_long).cuda())
        pf, sums = eng.eval_sampled(gt_t, r_t, c_t, off_t)
        assert _same(pf, want) and _same(sums, expected_sums(want))
        eng.status()
    finally:
        eng.close()
