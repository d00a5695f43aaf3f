"""eval_nyu.evaluate_fill_drawn_many (dtfill_eval_sampled_mt_many): D draws of evaluate_fill_drawn over one ground truth
in one call, each from its own MT19937 generator,

    for d in range(D): per_frame[d], sums[d] = evaluate_fill_drawn(gt, n[d], rngs[d], crop, src_thr)

The CPU tests check the symbol and the refusals that happen before the device is touched, with every generator left as
it was.  The GPU tests compare the call with that loop on copies of the generators, bit for bit, final states included.
Run them on the B200 box:  python -m pytest tests -m gpu"""
import copy
import ctypes

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib, synth
from distancetransform_depthcompletion_b200.eval_nyu import evaluate_fill_drawn, evaluate_fill_drawn_many

H, W = 240, 320
FILL_PX = 1 << 28        # dtfill.cu: at most this many pixels per fill of whole draws (at least one draw)


def _state(rng):
    st = rng.get_state(legacy=False)
    return st["state"]["key"].copy(), int(st["state"]["pos"]), st["has_gauss"], st["gauss"]


def _same_state(a, b):
    return np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def _rngs(seeds, gauss=False):
    out = [np.random.RandomState(s) for s in seeds]
    if gauss:
        for r in out:
            r.standard_normal()                # a cached Gaussian that must survive
    return out


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_symbol_is_exported(dtfill_lib):
    lib = ctypes.CDLL(dtfill_lib)
    assert hasattr(lib, "dtfill_eval_sampled_mt_many")
    assert _lib.load().dtfill_abi_version() == 9


@pytest.fixture
def no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the device was touched")
    monkeypatch.setattr(_lib, "get_handle", refuse)
    monkeypatch.setattr(_lib, "Handle", refuse)


def test_argument_checks_raise_before_the_device(no_device):
    gt = np.ones((3, H, W), np.float32)
    rngs = _rngs([1, 2, 3], gauss=True)
    before = [_state(r) for r in rngs]
    glob = _state(np.random)

    def refused(exc, *args, match=None, **kw):
        with pytest.raises(exc, match=match):
            evaluate_fill_drawn_many(*args, **kw)
        assert all(_same_state(_state(r), s) for r, s in zip(rngs, before))
        assert _same_state(_state(np.random), glob)

    for bad in (np.random.default_rng(0), np.random.RandomState(np.random.PCG64(0)), object(), None):
        for at in range(3):                    # a non-MT19937 generator in any position
            rs = list(rngs)
            rs[at] = bad
            refused(TypeError, gt, 20, rs, match="RandomState")
    refused(ValueError, gt, 20, [rngs[0], rngs[1], rngs[0]], match="share one generator")
    refused(ValueError, gt, 20, [np.random, rngs[1], np.random], match="share one generator")
    refused(ValueError, gt, 20, [np.random, np.random.mtrand._rand], match="share one generator")
    shared = np.random.MT19937(5)
    refused(ValueError, gt, 20, [np.random.RandomState(shared), np.random.RandomState(shared)], match="share one generator")
    refused(ValueError, gt, 20, [], match="no generators")
    refused(ValueError, gt, [20, 50], rngs, match="2 sample counts for 3 generators")
    refused(ValueError, gt, [20, 50, 200, 500], rngs, match="4 sample counts for 3 generators")
    refused(ValueError, gt, [20, -1, 50], rngs, match="^negative dimensions are not allowed$")
    refused(ValueError, gt, -1, rngs, match="^negative dimensions are not allowed$")
    refused(TypeError, gt, 2.5, rngs)
    refused(TypeError, gt, [20, 2.5, 50], rngs)
    refused(TypeError, gt, "20", rngs)
    refused(ValueError, gt, 20, rngs, crop=(6, 241, 8, 312), match="not a non-empty window")
    refused(ValueError, gt, 20, rngs, crop=(6, 6, 8, 312), match="not a non-empty window")
    refused(TypeError, gt.astype(np.float64), 20, rngs, match="float32")
    refused(TypeError, gt.astype(np.float16), 20, rngs, match="float32")
    refused(ValueError, np.ones((2, 12, W), np.float32), [5, 5, 5], rngs, crop=(0, 12, 0, W), match="^high <= 0$")
    refused(IndexError, np.ones((2, H, 16), np.float32), [0, 5, 5], rngs, crop=(0, H, 0, 16), match="draw 0, frame 0:")
    refused(ValueError, np.ones((0, H, W), np.float32), 5, rngs, match="empty batch")


# ---- GPU ----------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
K = 16          # distinct ground-truth frames; larger batches repeat them


@pytest.fixture(scope="module")
def gts():
    return np.stack([synth.nyu_frame(s, H, W, return_dense=True)[1] for s in range(K)])


def _gt(gts, B):
    return np.ascontiguousarray(gts[[b % K for b in range(B)]])


def _loop(gt, ns, rngs, **kw):
    """The reference of the call: evaluate_fill_drawn per draw on the generators given (copies of the call's)."""
    pf, sums = zip(*[evaluate_fill_drawn(gt, n, rng=r, **kw) for n, r in zip(ns, rngs)])
    return np.stack(pf), np.stack(sums)


def _check(gt_arg, gt_loop, ns, seeds, n_arg=None, **kw):
    rngs = _rngs(seeds, gauss=True)
    ref = copy.deepcopy(rngs)
    want_pf, want_sums = _loop(gt_loop, ns, ref, **kw)
    pf, sums = evaluate_fill_drawn_many(gt_arg, ns if n_arg is None else n_arg, rngs, **kw)
    assert pf.shape == (len(ns), gt_loop.shape[0], 9) and sums.shape == (len(ns), 10)
    assert pf.dtype == np.float64 and sums.dtype == np.float64
    assert _same(pf, want_pf) and _same(sums, want_sums), (ns, seeds)
    for d, (r, q) in enumerate(zip(rngs, ref)):
        assert _same_state(_state(r), _state(q)), d
    return pf, sums


@gpu
@pytest.mark.parametrize("D", [1, 3, 7])
def test_equals_the_loop_per_draw(dtfill_lib, gts, D):
    B = 9
    gt = _gt(gts, B)
    ns = [(20, 30, 50, 100, 200, 500, 5000)[(d + D) % 7] for d in range(D)]
    _check(gt, gt, ns, [1000 * D + d for d in range(D)])
    _check(gt, gt, [20] * D, [2000 * D + d for d in range(D)], n_arg=20)          # one n for every draw


@gpu
@pytest.mark.parametrize("D", [1, 3, 7])
def test_ranges_of_one_consume_no_words(dtfill_lib, D):
    """13 x 17 frames: randint(1) takes no word, so every sample is pixel (6, 8), frame 0 of draw 0 has one valid depth
    and Distance_Transform rejects it, as in the loop; every generator comes back unchanged."""
    B = 5
    rng = np.random.default_rng(7)
    gt = (rng.random((B, 13, 17), np.float32) * 9 + 0.5).astype(np.float32)
    crop = (0, 13, 0, 17)
    rngs = _rngs([11 + d for d in range(D)])
    before = [_state(r) for r in rngs]
    ref = copy.deepcopy(rngs)
    for n in (1, 4):
        want = [_outcome(lambda: evaluate_fill_drawn(gt, n, rng=r, crop=crop)) for r in ref]
        got = _outcome(lambda: evaluate_fill_drawn_many(gt, n, rngs, crop=crop))
        if isinstance(want[0][0], str):
            assert got == want[0] == ("IndexError", (0, 0))
        else:
            assert _same(got[0], np.stack([w[0] for w in want])) and _same(got[1], np.stack([w[1] for w in want]))
        assert all(_same_state(_state(r), s) for r, s in zip(rngs, before))


def _outcome(fn):
    """(per_frame, sums) of a call, or ("IndexError", (draw, frame)) parsed from the message."""
    try:
        return fn()
    except IndexError as e:
        msg = str(e)
        d = int(msg.split("draw ")[1].split(",")[0]) if "draw " in msg else 0
        return "IndexError", (d, int(msg.split("frame ")[1].split(":")[0]))


@gpu
def test_nyu_batch_across_fill_boundaries(dtfill_lib, gts):
    """654 frames of 240 x 320, 12 draws: 5 draws per fill, so three fills and two boundaries between them."""
    B, D = 654, 12
    assert FILL_PX // (B * H * W) == 5
    gt = _gt(gts, B)
    ns = [(20, 50, 200, 500)[d % 4] for d in range(D)]
    _check(gt, gt, ns, [100000 * n + d for d, n in enumerate(ns)])


@gpu
def test_tensor_and_numpy_ground_truth(dtfill_lib, gts):
    import torch
    B = 40
    gt = _gt(gts, B)
    gt_t = torch.from_numpy(gt).cuda()
    ns = [20, 200, 50, 500]
    pf, sums = _check(gt_t, gt, ns, [31, 32, 33, 34])
    pf2, sums2 = _check(gt, gt, ns, [31, 32, 33, 34])
    assert _same(pf, pf2) and _same(sums, sums2)


@gpu
def test_engine(dtfill_lib, gts):
    import torch
    from distancetransform_depthcompletion_b200.engine import DTFillEngine
    B = 32
    gt = _gt(gts, B)
    gt_t = torch.from_numpy(gt).cuda()
    ns = [50, 20, 200]
    rngs = _rngs([41, 42, 43])
    ref = copy.deepcopy(rngs)
    want_pf, want_sums = _loop(gt, ns, ref)
    eng = DTFillEngine(0, pipeline_depth=2)
    try:
        x = torch.from_numpy(synth.nyu_batch(range(32))).cuda()
        eng.fill(x)
        pf, sums = eng.eval_drawn_many(gt_t, ns, rngs)
        assert _same(pf, want_pf) and _same(sums, want_sums)
        assert all(_same_state(_state(r), _state(q)) for r, q in zip(rngs, ref))
        eng.status()
    finally:
        eng.close()


@gpu
def test_index_error_raised_by_a_middle_draw(dtfill_lib, gts):
    """n = 1 leaves one valid depth per frame: Distance_Transform rejects frame 0 of that draw.  With draws
    (20, 50, 1, 200), draw 2 fails: draws 0 and 1 end where their whole draws end, draw 2 after frame 0's draws, draw 3
    is untouched."""
    B = 8
    gt = _gt(gts, B)
    ns = [20, 50, 1, 200]
    rngs = _rngs([61, 62, 63, 64], gauss=True)
    before = [_state(r) for r in rngs]
    ref = copy.deepcopy(rngs)
    for d in range(2):
        evaluate_fill_drawn(gt, ns[d], rng=ref[d])
    with pytest.raises(IndexError, match="frame 0:") as e_loop:
        evaluate_fill_drawn(gt, ns[2], rng=ref[2])
    with pytest.raises(IndexError) as e:
        evaluate_fill_drawn_many(gt, ns, rngs)
    assert str(e.value).startswith("draw 2, frame 0: ")
    assert str(e.value).split(": ", 1)[1] == str(e_loop.value).split(": ", 1)[1]
    for d in range(3):
        assert _same_state(_state(rngs[d]), _state(ref[d])), d
    assert _same_state(_state(rngs[3]), before[3])
    # the handle recovers
    _check(gt, gt, [20, 50], [71, 72])


@gpu
@pytest.mark.parametrize("B,D", [(654, 12), (40, 3)])
def test_transfer_bytes(dtfill_lib, gts, B, D):
    import torch
    gt = _gt(gts, B)
    ns = [(20, 50, 200, 500)[d % 4] for d in range(D)]
    per_fill = max(1, FILL_PX // (B * H * W))
    fills = -(-D // per_fill)
    state_up = D * 624 * 4 + D * 8                                  # keys, {pos, n} per draw
    down = (D * B * 8 + D * 624 * 4 + D * 4                        # words, keys, pos
            + D * B * 8 + fills * 4                                  # fill counts, one flag word per fill
            + D * B * 72 + D * 80)                                   # rows, sums
    h = _lib.get_handle(0)
    evaluate_fill_drawn_many(torch.from_numpy(gt).cuda(), ns, _rngs(range(D)))
    assert h.transfer_bytes() == (state_up, down)
    evaluate_fill_drawn_many(gt, ns, _rngs(range(D)))
    assert h.transfer_bytes() == (state_up + B * H * W * 4, down)
