"""KITTI outlier filter (kernel k6_outlier_removal, data_read.py:103-128) at the edges the KITTI-grid frames of
test_outlier_removal.py do not reach, compared bit for bit (the sign of zero included) with oracle.outlier_removal_numpy:
batches whose warps straddle frames, both the vectorised and the scalar path, the verdict and count thresholds swept one
float32 step at a time, and NaN, +-inf, denormals, -0.0 and negative depths.  The restatement itself is pinned to the
reference's lines with the real cv2.filter2D here too (no GPU needed)."""
import ctypes

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import _lib
from oracle import oracle as O

f32 = np.float32
SPECIALS = (np.nan, np.inf, -np.inf, 1e-40, -1e-40, 1.4e-45, -0.0, 0.0, 3e38, -3e38)      # quiet NaN only


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same_bits(got, want, what):
    g, w = bits(got), bits(want)
    bad = np.argwhere(g != w)
    assert bad.size == 0, (f"{what}: {len(bad)} pixels differ; first at {tuple(bad[0])}: got {got[tuple(bad[0])]!r} "
                           f"({g[tuple(bad[0])]:#010x}), want {want[tuple(bad[0])]!r} ({w[tuple(bad[0])]:#010x})")


def negative_frame():
    """A 9 x 9 frame of -5 m with -1 m at the centre: no pixel counts as valid, every average is below its depth by far
    more than 1 m, so the reference drops all 81 and -5 * (1 - 1) in float64 gives -0.0 for each."""
    x = np.full((9, 9), f32(-5.0))
    x[4, 4] = f32(-1.0)
    return x


def edge_frames():
    """Frames away from the 1/256 grid: random depths of several scales, frames that are all border (the diamond
    reflects more than once), signed frames, and NaN, +-inf, denormals, +-0 and negative neighbourhoods."""
    rng = np.random.default_rng(11)
    frames = []
    for H, W, scale, dens in ((40, 64, 80.0, 0.3), (33, 47, 1.0, 0.8), (20, 24, 1e4, 0.5), (16, 16, 3.0, 1.0)):
        frames.append((rng.uniform(0, scale, (H, W)) * (rng.random((H, W)) < dens)).astype(f32))
    frames.append(rng.normal(0, 4, (24, 28)).astype(f32))
    for H, W in ((1, 1), (1, 9), (1, 12), (9, 1), (2, 2), (3, 3), (2, 3), (3, 2), (4, 5), (6, 6)):
        frames.append((rng.uniform(0.05, 6.0, (H, W)) * (rng.random((H, W)) < 0.7)).astype(f32))
        frames.append(-rng.uniform(0.05, 6.0, (H, W)).astype(f32))
    frames.append(negative_frame())
    for k, s in enumerate(SPECIALS):
        x = (rng.uniform(0.5, 3.0, (12, 16)) * (rng.random((12, 16)) < 0.6)).astype(f32)
        x[5, 7] = f32(s)
        x[rng.integers(0, 12), rng.integers(0, 16)] = f32(s)
        if k % 2:
            x[0:4, 0:4] = -rng.uniform(2, 9, (4, 4)).astype(f32)          # a negative corner
        frames.append(x)
    mix = rng.uniform(1, 50, (14, 20)).astype(f32)
    for i, s in enumerate(SPECIALS):
        mix[(3 * i) % 14, (7 * i) % 20] = f32(s)
    frames.append(mix)
    tiny = (rng.uniform(1, 2, (10, 11)) * 1e-39).astype(f32)                  # denormals only, one normal depth
    tiny[4, 4] = f32(0.5)
    frames.append(tiny)
    return frames


@pytest.mark.skipif(not O.have_cv2(), reason="cv2 absent")
def test_numpy_restatement_matches_cv2():
    dropped = 0
    for x in edge_frames():
        want = O.cv2_port_outlier_removal(x, squeeze=False)
        got = O.outlier_removal_numpy(x)
        assert got.dtype == np.float32 and got.shape == x.shape
        assert_same_bits(got, want, f"frame {x.shape}")
        dropped += int((bits(got) != bits(x)).sum())
    assert dropped > 200, dropped
    neg = negative_frame()
    assert (bits(O.outlier_removal_numpy(neg)) == 0x80000000).all()
    assert_same_bits(O.cv2_port_outlier_removal(neg[None, :, :, None]), O.outlier_removal_numpy(neg), "squeezed")
    xb = np.stack([edge_frames()[0]] * 3)
    xb[1] *= f32(7.5)
    for b in range(3):
        assert_same_bits(O.outlier_removal_numpy(xb)[b], O.outlier_removal_numpy(xb[b]), f"batch frame {b}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def handle(dtfill_lib):
    return _lib.get_handle()


def filter_device(handle, xb, offset, out_offset=None):
    """dtfill_outlier_removal on device pointers `offset` floats into fresh torch buffers (offset 1 defeats the 16-byte
    alignment the vectorised path needs); the floats around the output must stay as they were."""
    import torch
    xb = np.ascontiguousarray(xb, np.float32)
    B, H, W = xb.shape
    n = xb.size
    oo = offset if out_offset is None else out_offset
    src = torch.full((n + 8,), -7.0, dtype=torch.float32, device="cuda")
    dst = torch.full((n + 8,), 1234.5, dtype=torch.float32, device="cuda")
    src[offset:offset + n] = torch.from_numpy(xb.ravel()).cuda()
    torch.cuda.synchronize()
    rc = handle._L.dtfill_outlier_removal(handle._h, ctypes.c_void_p(src.data_ptr() + 4 * offset), 1, B, H, W,
                                          ctypes.c_void_p(dst.data_ptr() + 4 * oo), 1)
    _lib._check(rc, "dtfill_outlier_removal")
    handle.synchronize()
    d = dst.cpu().numpy()
    assert (d[:oo] == 1234.5).all() and (d[oo + n:] == 1234.5).all(), "wrote outside the output"
    return d[oo:oo + n].reshape(B, H, W)


def check_batch(handle, xb, what, per_frame=False):
    """Host call (vectorised when W % 4 == 0), device call through the scalar path, and the reference; with per_frame
    every frame must also equal a B = 1 call."""
    xb = np.ascontiguousarray(xb, np.float32)
    want = O.outlier_removal_numpy(xb)
    got = handle.outlier_removal(xb)
    assert got.shape == xb.shape and got.dtype == np.float32
    assert_same_bits(got, want, f"{what} host")
    assert_same_bits(filter_device(handle, xb, 1), want, f"{what} scalar path")
    if per_frame:
        for b in range(xb.shape[0]):
            assert_same_bits(handle.outlier_removal(xb[b:b + 1])[0], got[b], f"{what} frame {b} alone")
    return want


def scaled_batch(rng, B, H, W):
    """Frames of very different depth scales next to each other (a window read from the wrong frame flips verdicts),
    non-grid values, mostly sparse with planted far points, some signed."""
    scales = (1.0, 1000.0, 0.01, 30.0, 5e4, 0.3)
    xb = np.empty((B, H, W), np.float32)
    for b in range(B):
        s = scales[b % len(scales)]
        x = rng.uniform(0.2, 1.0, (H, W)) * s * (rng.random((H, W)) < (0.35, 0.8, 1.0)[b % 3])
        far = rng.random((H, W)) < 0.08
        x[far] *= 6.0
        if b % 7 == 3:
            x = -x
        xb[b] = x
    return xb


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(37, 9, 12), (7, 2, 8), (5, 1, 4), (33, 7, 20), (4, 3, 1216), (9, 5, 4),
                                   (5, 9, 13), (3, 352, 1215), (6, 1, 7), (2, 352, 1216)])
def test_batches_against_reference(handle, shape):
    """Warps that hold the end of one frame and the start of the next (H * W / 4 not a multiple of 32), widths that take
    the scalar path, and the full KITTI size."""
    B, H, W = shape
    rng = np.random.default_rng(B * 100003 + H * 101 + W)
    xb = scaled_batch(rng, B, H, W)
    want = check_batch(handle, xb, f"{shape}", per_frame=True)
    assert (bits(want) != bits(xb)).sum() > 0                 # the batch has verdicts to get wrong


def sweep(neigh, centre, count=100):
    """Frames 7 x 12 (21 four-pixel groups: warps straddle frames) with one diamond neighbourhood around (3, 5) and the
    centre stepped through the float32 values centre - count ulps .. centre + count - 1 ulps."""
    c = np.asarray(f32(centre)).view(np.int32) + np.arange(-count, count, dtype=np.int32)
    vals = c.view(np.float32)
    xb = np.zeros((vals.size, 7, 12), np.float32)
    k = 0
    for dy in range(-3, 4):
        for dx in range(-3, 4):
            if abs(dy) + abs(dx) <= 3 and (dy, dx) != (0, 0):
                xb[:, 3 + dy, 5 + dx] = neigh[k]
                k += 1
    xb[:, 3, 5] = vals
    return xb


def centre_flip(neigh, lo, hi):
    """The least float32 centre in [lo, hi] that the reference drops (bisection on the bit pattern; positive floats)."""
    a, b = int(np.asarray(f32(lo)).view(np.int32)), int(np.asarray(f32(hi)).view(np.int32))
    dropped = lambda i: O.outlier_removal_numpy(sweep(neigh, np.asarray(np.int32(i)).view(np.float32), 1)[1])[3, 5] == 0
    assert not dropped(a) and dropped(b)
    while b - a > 1:
        m = (a + b) // 2
        a, b = (a, m) if dropped(m) else (m, b)
    return np.asarray(np.int32(b)).view(np.float32)


@pytest.mark.gpu
def test_verdict_threshold_sweep(handle):
    """The strict `> 1.0` of the float64 average: the kernel must drop the centre from exactly the same float32 value on.
      - 24 neighbours of random depths, all counted;
      - 24 neighbours at exactly 0.1f, which are not counted (`> 0.1` in float32): the centre is the only valid pixel,
        its average is within 1e-5 of itself, and the verdict turns on the float64 division by 1.00001;
      - the same at nextafter(0.1f, 1), which are counted;
      - one neighbour at -1 and centre 1: the sum is 0 and x - average is exactly 1.0, which is not dropped."""
    rng = np.random.default_rng(21)
    p1 = np.nextafter(f32(0.1), f32(1))
    cases = [(rng.uniform(2.0, 3.0, 24).astype(f32), 1.0, 8.0),
             (np.full(24, f32(0.1)), 1e5, 1e6),
             (np.full(24, p1), 1.0, 2.0)]
    xbs = [sweep(n, centre_flip(n, lo, hi)) for n, lo, hi in cases]
    one = np.zeros(24, np.float32)
    one[5] = f32(-1.0)
    xbs.append(sweep(one, 1.0))
    xb = np.concatenate(xbs)
    want = check_batch(handle, xb, "threshold sweep")
    for i, first in enumerate((100, 100, 100, 101)):
        kept = want[200 * i:200 * (i + 1), 3, 5] != 0
        assert kept[:first].all() and not kept[first:].any(), i      # the reference flips at the swept point
    assert want[700, 3, 5] == 1.0 and want[701, 3, 5] == 0.0         # exactly 1.0 m above the average: kept
    # the count threshold on its own: a centre of 1.2 m is kept beside 0.1f and dropped beside nextafter(0.1f, 1)
    pair = np.concatenate([sweep(np.full(24, f32(0.1)), 1.2, 1), sweep(np.full(24, p1), 1.2, 1)])
    want = check_batch(handle, pair, "count threshold")
    assert want[1, 3, 5] == f32(1.2) and want[3, 3, 5] == 0


@pytest.mark.gpu
def test_special_values_and_signs(handle):
    """NaN, +-inf, denormals, +-0 at the centre and in the window, and negative depths beside more negative ones: a
    dropped negative depth is -0.0, as the reference's x * (1 - 1) in float64 gives."""
    frames = edge_frames()
    for x in frames:
        check_batch(handle, x[None], f"frame {x.shape}")
    same = np.stack([x for x in frames if x.shape == (12, 16)])
    check_batch(handle, same, "specials batch", per_frame=True)
    got = handle.outlier_removal(negative_frame()[None])
    assert (bits(got) == 0x80000000).all(), "dropped negative depths must keep their sign"
    rng = np.random.default_rng(31)
    neg = -rng.uniform(0.5, 9.0, (6, 10, 12)).astype(f32)
    neg[:, 4:6, 4:6] = f32(-0.2)                               # shallow pixels beside deeper ones: dropped
    want = check_batch(handle, neg, "negative batch", per_frame=True)
    assert (bits(want) == 0x80000000).sum() > 20


@pytest.mark.gpu
def test_device_pointers(handle):
    """Device-resident calls: 16-byte aligned buffers take the vectorised path and buffers one float off take the scalar
    one; both equal the host call.  An output that is the input is refused."""
    import torch
    rng = np.random.default_rng(41)
    xb = scaled_batch(rng, 11, 9, 12)
    xb[4] = np.pad(negative_frame(), ((0, 0), (0, 3)))
    want = O.outlier_removal_numpy(xb)
    assert_same_bits(handle.outlier_removal(xb), want, "host")
    for off, out_off in ((0, 0), (4, 8), (1, 1), (0, 1), (3, 0)):
        assert_same_bits(filter_device(handle, xb, off, out_off), want, f"offsets {off} {out_off}")
    t = torch.from_numpy(xb).cuda()
    torch.cuda.synchronize()
    p = ctypes.c_void_p(t.data_ptr())
    with pytest.raises(ValueError, match="alias"):
        _lib._check(handle._L.dtfill_outlier_removal(handle._h, p, 1, 11, 9, 12, p, 1), "dtfill_outlier_removal")
    assert_same_bits(filter_device(handle, xb, 1), want, "after the refusal")
