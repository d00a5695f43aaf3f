"""Pins the oracle against what the reference computed, stored under tests/golden/ by make_golden.py: the outputs of
cv2.distanceTransformWithLabels (the call at tools.py:9) on random masks, and checksums of the reference's own
tools.DT_complete_batch / tools.nearest_point / eval_NYU.Distance_Transform on seeded synthetic frames
(test_oracle_golden.py compares other seeds of the same files)."""
import hashlib
import os

import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import synth
from oracle import oracle as O


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def sums(golden_dir):
    return np.load(os.path.join(golden_dir, "checksums.npz"))


def test_random_masks_vs_cv2(golden_dir):
    z = np.load(os.path.join(golden_dir, "cv2_masks.npz"))
    assert len(z["shapes"]) == 300
    off = 0
    for t, (H, W) in enumerate(z["shapes"]):
        n = int(H) * int(W)
        m = z["mask"][off:off + n].reshape(H, W)
        d2, l2 = O.chamfer_l1_labels(m)
        dt = z["dt_u16"][off:off + n].reshape(H, W).astype(np.float32)
        lbl = z["lbl_i16"][off:off + n].reshape(H, W).astype(np.int32)
        assert np.array_equal(dt, d2) and np.array_equal(lbl, l2), (t, H, W)
        off += n
    assert off == len(z["mask"])


def test_tools_dt_complete_batch(sums):
    seeds = [1, 2]
    xb = synth.kitti_batch(seeds, beam_step=2)
    got = O.dt_fill(xb[..., 0])
    for i, seed in enumerate(seeds):
        assert [sha(got["depth"][i]), sha(got["dt"][i]), sha(got["lbl"][i])] == list(sums[f"kitti_b32_s{seed}"]), seed


def test_eval_nyu_distance_transform(sums):
    for seed in (0, 1, 3):
        r = O.dt_fill(synth.nyu_frame(seed), 0.001, 0.1)
        assert [sha(r["depth"]), sha(r["dt"]), sha(r["lbl"])] == list(sums[f"nyu_s{seed}"]), seed


@pytest.mark.skipif(not O.have_cv2(), reason="cv2 absent")
def test_cv2_port_matches_tools(sums):
    for step, seed in ((1, 1), (1, 2), (4, 0), (8, 1)):
        xb = synth.kitti_batch([seed], beam_step=step)
        got = O.cv2_port_complete_batch(xb)
        assert got.dtype == np.float32 and got.shape == (1, 352, 1216, 1)
        assert sha(got[0, :, :, 0]) == sums[f"kitti_b{64 // step}_s{seed}"][0], (step, seed)


def test_tf_stand_in_extract_patches():
    """The stand-in for TensorFlow that make_golden.py runs the reference's DT-pooling lines on (net.py:83-123,
    demo.py:107-149; their outputs are dt_pool.npz): its extract_patches against a plain loop over window offsets and
    pixels."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import tf_numpy_shim as tf
    rng = np.random.default_rng(5)
    img = rng.random((2, 6, 7, 1)).astype(np.float32)
    for t in (3, 5):
        got = tf.image.extract_patches(img, sizes=(1, t, t, 1), strides=(1, 1, 1, 1), rates=(1, 1, 1, 1), padding="SAME")
        assert got.shape == (2, 6, 7, t * t)
        for b in range(2):
            for y in range(6):
                for x in range(7):
                    for i in range(t):
                        for j in range(t):
                            yy, xx = y + i - t // 2, x + j - t // 2
                            want = img[b, yy, xx, 0] if 0 <= yy < 6 and 0 <= xx < 7 else 0.0
                            assert got[b, y, x, i * t + j] == want
