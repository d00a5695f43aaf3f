"""eval_nyu.evaluate_fill_drawn (dtfill_eval_sampled_mt): the NYU script's loop with its draws made on the device from
numpy's MT19937 state,

    rows = rng.randint(H - 12, size=n) + 6; cols = rng.randint(W - 16, size=n) + 8; ... evaluate_fill_sampled's loop body

per frame.  The CPU tests run the draw through the host hook (the kernel's MT19937 helpers run serially) against numpy's
randint and get_state, and the checks that run before the device is touched.  The GPU tests compare the device's draws,
rows, sums and final state with the host loop, bit for bit.  Run them on the B200 box:  python -m pytest tests -m gpu"""
import ctypes

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib, eval_nyu, evaluation, synth
from distancetransform_depthcompletion_b200.eval_nyu import (NYU_EVAL_CROP, evaluate_fill_drawn, evaluate_fill_sampled,
                                                             nyu_sample_coords)

H, W = 240, 320


def _rs(seed, pos=None):
    """A RandomState seeded with seed, its pos moved to `pos` (the key stays)."""
    rs = np.random.RandomState(seed)
    if pos is not None:
        st = rs.get_state(legacy=False)
        st["state"]["pos"] = pos
        rs.set_state(st)
    return rs


def _state(rng):
    st = rng.get_state(legacy=False)
    return st["state"]["key"].copy(), int(st["state"]["pos"]), st["has_gauss"], st["gauss"]


def _same_state(a, b):
    return np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def host_draws(rng, B, n, h=H, w=W):
    """The reference's draws of B frames, and rng's state after each frame."""
    rows, cols, after = [], [], []
    for _ in range(B):
        r, c = nyu_sample_coords(n, h, w, rng=rng)
        rows.append(r)
        cols.append(c)
        after.append(_state(rng))
    return np.array(rows).reshape(B, n), np.array(cols).reshape(B, n), after


def _replay(key, pos, words):
    bg = np.random.MT19937()
    bg.state = {"bit_generator": "MT19937", "state": {"key": key, "pos": pos}}
    bg.random_raw(int(words))
    return bg.state["state"]["key"], int(bg.state["state"]["pos"])


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_symbol_is_exported_and_abi_version(dtfill_lib):
    lib = ctypes.CDLL(dtfill_lib)
    assert hasattr(lib, "dtfill_eval_sampled_mt") and hasattr(lib, "dtfill_debug_mt_draw_host")
    assert _lib.ABI_VERSION == 9 and _lib.load().dtfill_abi_version() == 9


SIZES = [(240, 320), (480, 640), (13, 17), (268, 320), (269, 273)]


@pytest.mark.parametrize("seed", [0, 1, 42, 2 ** 32 - 1])
@pytest.mark.parametrize("pos", [0, 1, 623, 624])
def test_host_hook_is_numpys_randint(dtfill_lib, seed, pos):
    """Coordinates, words per frame and the final state of the hook equal numpy's randint pair per frame and get_state:
    13 x 17 has ranges of 1 (no word consumed), 268 x 320 a row range of 256 (no rejection), 269 x 273 ranges of 257
    (about half the words rejected)."""
    for h, w in SIZES:
        for n in (0, 1, 20, 500, 5000):
            B = 3
            rs = _rs(seed, pos)
            key0, pos0 = _state(rs)[:2]
            rows, cols, k, p, words = _lib.mt_draw_host(key0, pos0, B, h, w, n)
            want_r, want_c, after = host_draws(rs, B, n, h, w)
            case = (h, w, n)
            assert np.array_equal(rows, want_r) and np.array_equal(cols, want_c), case
            assert np.array_equal(k, after[-1][0]) and p == after[-1][1], case
            for b in range(B):          # words[:b+1] replayed from the start is the state after frame b
                rk, rp = _replay(key0, pos0, words[:b + 1].sum())
                assert np.array_equal(rk, after[b][0]) and rp == after[b][1], (case, b)
            if (h, w) == (13, 17) or n == 0:
                assert (words == 0).all() and p == pos0 and np.array_equal(k, key0), case
            if (h, w) == (268, 320):
                assert (words >= n).all()
            if (h, w) == (269, 273) and n >= 500:
                assert (words > 3 * n).all()          # 257 of 512 values accepted in both ranges


@pytest.fixture
def no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the device was touched")
    monkeypatch.setattr(_lib, "get_handle", refuse)
    monkeypatch.setattr(_lib, "Handle", refuse)


def test_argument_checks_raise_before_the_device(no_device):
    gt = np.ones((3, H, W), np.float32)
    rs = _rs(7)
    rs.standard_normal()                       # a cached Gaussian that must survive
    before = _state(rs)
    glob = _state(np.random)

    def refused(exc, *args, match=None, **kw):
        with pytest.raises(exc, match=match):
            evaluate_fill_drawn(*args, **kw)
        assert _same_state(_state(rs), before) and _same_state(_state(np.random), glob)

    for bad_rng in (np.random.default_rng(0), np.random.RandomState(np.random.PCG64(0)), np.random.Generator(np.random.MT19937(0)),
                    object(), None):
        refused(TypeError, gt, 20, rng=bad_rng, match="RandomState")
    refused(TypeError, gt.astype(np.float64), 20, rng=rs)
    refused(TypeError, gt, 2.5, rng=rs)
    refused(ValueError, gt, -1, rng=rs, match="^negative dimensions are not allowed$")
    refused(ValueError, np.ones((2, 12, W), np.float32), 5, rng=rs, crop=(0, 12, 0, W), match="^high <= 0$")
    refused(ValueError, np.ones((2, H, 16), np.float32), 5, rng=rs, crop=(0, H, 0, 16), match="^high <= 0$")
    refused(IndexError, np.ones((2, H, 16), np.float32), 0, rng=rs, crop=(0, H, 0, 16), match="frame 0:")
    refused(ValueError, np.ones((0, H, W), np.float32), 5, rng=rs, match="empty batch")
    refused(ValueError, gt[0], 5, rng=rs, match="must be \\[B,H,W\\]")
    refused(ValueError, gt, 5, rng=rs, crop=(6, 241, 8, 312), match="not a non-empty window")
    refused(ValueError, gt, -1, match="negative dimensions")          # the global state, untouched
    # numpy raises the same messages
    with pytest.raises(ValueError, match="^high <= 0$"):
        np.random.RandomState(0).randint(0, size=5)
    with pytest.raises(ValueError, match="^negative dimensions are not allowed$"):
        np.random.RandomState(0).randint(5, size=-1)


# ---- GPU ----------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
K = 16          # distinct ground-truth frames; larger batches repeat them


@pytest.fixture(scope="module")
def gts():
    return np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(K)])


def _gt(gts, B):
    return np.ascontiguousarray(gts[[b % K for b in range(B)]])


def _outcome(fn):
    """(per_frame, sums) of a call, or ("IndexError", frame) parsed from the message."""
    try:
        return fn()
    except IndexError as e:
        return "IndexError", int(str(e).split("frame ")[1].split(":")[0])


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def _check_against_sampled(gt_arg, gt_np, n, seed, B):
    """evaluate_fill_drawn from RandomState(seed) equals the host loop: its draws, evaluate_fill_sampled on them, and the
    state the loop leaves."""
    rs_host = _rs(seed)
    rows, cols, after = host_draws(rs_host, B, n)
    want = _outcome(lambda: evaluate_fill_sampled(gt_np, rows, cols))
    rs = _rs(seed)
    got = _outcome(lambda: evaluate_fill_drawn(gt_arg, n, rng=rs, return_coords=True))
    if isinstance(want[0], str):
        assert got == want, (n, seed, got, want)
        assert _same_state(_state(rs), after[want[1]])
        return None
    pf, sums, r, c = got
    assert r.dtype == np.int64 and np.array_equal(r, rows) and np.array_equal(c, cols), (n, seed)
    assert _same(pf, want[0]) and _same(sums, want[1]), (n, seed)
    assert _same_state(_state(rs), after[-1])
    return pf, rows, cols


@gpu
@pytest.mark.parametrize("B", [1, 7, 654])
def test_coordinates_and_state_equal_the_host_loop(dtfill_lib, gts, B):
    gt = _gt(gts, B)
    for n, pos in ((20, None), (500, 0), (200, 624), (50, 1)):
        rs = _rs(B * 100 + n, pos)
        rows, cols, after = host_draws(_rs(B * 100 + n, pos), B, n)
        pf, sums, r, c = evaluate_fill_drawn(gt, n, rng=rs, return_coords=True)
        assert np.array_equal(r, rows) and np.array_equal(c, cols), (B, n)
        assert _same_state(_state(rs), after[-1]), (B, n)


@gpu
@pytest.mark.parametrize("n", [2, 20, 50, 200, 500, 5000])
def test_rows_and_sums_equal_evaluate_fill_sampled(dtfill_lib, gts, n):
    import torch
    B = 24
    gt = _gt(gts, B)
    gt_t = torch.from_numpy(gt).cuda()
    for seed in (n, n + 1):
        _check_against_sampled(gt, gt, n, seed, B)
        _check_against_sampled(gt_t, gt, n, seed + 10, B)


def _oracle_row(gt, rows, cols, crop=NYU_EVAL_CROP):
    """The cv2 port of eval_NYU.py:120-133 + oracle.result_nyu on one frame."""
    from oracle import oracle as O
    mask = np.zeros(gt.shape, np.float32)
    mask[rows, cols] = 1
    pred = O.cv2_port_fill_frame(gt * mask, 0.001, 0.1, nyu_style=True)[0]
    r0, r1, c0, c1 = crop
    m = O.result_nyu(pred[r0:r1, c0:c1], gt[r0:r1, c0:c1])
    return np.array([m[k] for k in ("mse", "rmse", "mae", "irmse", "imae", "delta1", "delta2", "delta3", "count")])


@gpu
def test_oracle_subset(dtfill_lib, gts):
    gt = _gt(gts, 6)
    pf, _, rows, cols = evaluate_fill_drawn(gt, 200, rng=_rs(5), return_coords=True)
    for b in range(6):
        assert _same(pf[b], _oracle_row(gt[b], rows[b], cols[b])), b


@gpu
def test_two_calls_continue_one_stream(dtfill_lib, gts):
    B, n = 40, 50
    gt = _gt(gts, B)
    rs_host = _rs(11)
    rows, cols, after = host_draws(rs_host, 2 * B, n)
    want, wsums = evaluate_fill_sampled(np.concatenate([gt, gt]), rows, cols)
    rs = _rs(11)
    pf1, s1, r1, c1 = evaluate_fill_drawn(gt, n, rng=rs, return_coords=True)
    pf2, s2, r2, c2 = evaluate_fill_drawn(gt, n, rng=rs, return_coords=True)
    assert np.array_equal(np.concatenate([r1, r2]), rows) and np.array_equal(np.concatenate([c1, c2]), cols)
    assert _same(np.concatenate([pf1, pf2]), want)
    assert _same_state(_state(rs), after[-1])
    assert rs.randint(1 << 30) == rs_host.randint(1 << 30)      # a host draw after the calls continues the stream


@gpu
def test_global_np_random(dtfill_lib, gts):
    B, n = 9, 20
    gt = _gt(gts, B)
    saved = np.random.get_state()
    try:
        np.random.seed(3)
        rows, cols, after = host_draws(np.random, B, n)
        tail = np.random.randint(1 << 30)
        np.random.seed(3)
        pf, sums, r, c = evaluate_fill_drawn(gt, n, return_coords=True)
        assert np.array_equal(r, rows) and np.array_equal(c, cols)
        assert _same_state(_state(np.random), after[-1])
        assert np.random.randint(1 << 30) == tail
        assert _same(pf, evaluate_fill_sampled(gt, rows, cols)[0])
    finally:
        np.random.set_state(saved)


@gpu
def test_index_error_leaves_rng_after_that_frame(dtfill_lib, gts):
    B = 8
    gt = _gt(gts, B)
    for n in (0, 1):
        rs = _rs(21)
        _, _, after = host_draws(_rs(21), B, n)
        with pytest.raises(IndexError, match="frame 0:"):
            evaluate_fill_drawn(gt, n, rng=rs)
        assert _same_state(_state(rs), after[0]), n
    bad = gt.copy()
    bad[5] = 0                                   # no valid depth in frame 5
    for n in (20, 500):
        rs = _rs(22 + n)
        _, _, after = host_draws(_rs(22 + n), B, n)
        with pytest.raises(IndexError, match="frame 5:"):
            evaluate_fill_drawn(bad, n, rng=rs)
        assert _same_state(_state(rs), after[5]), n
        assert not _same_state(after[5], after[-1])
    # the handle recovers
    _check_against_sampled(gt, gt, 20, 30, B)


@gpu
def test_transfer_bytes_and_engine(dtfill_lib, gts):
    import torch
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    B, n = 654, 20
    gt = _gt(gts, B)
    gt_t = torch.from_numpy(gt).cuda()
    rs = _rs(40)
    pf, sums = evaluate_fill_drawn(gt_t, n, rng=rs)
    h2d, d2h = _lib.get_handle(0).transfer_bytes()
    assert h2d == 624 * 4                                            # the key only: no coordinates, no ground truth
    assert d2h == 2512 + B * 8 + B * (8 + 72) + 4 + 80              # state and words, counts and flag, metrics
    rows, cols, after = host_draws(_rs(40), B, n)
    assert _same(pf, evaluate_fill_sampled(gt_t, rows, cols)[0]) and _same_state(_state(rs), after[-1])
    eng = DTFillEngine(0, pipeline_depth=2)
    try:
        x = torch.from_numpy(synth.nyu_batch(range(32))).cuda()
        eng.fill(x)
        rs2 = _rs(40)
        pf2, sums2 = eng.eval_drawn(gt_t, n, rng=rs2)
        assert _same(pf2, pf) and _same(sums2, sums) and _same_state(_state(rs2), after[-1])
        eng.status()
    finally:
        eng.close()
