"""KITTI outlier filter (SURVEY.md section 8 f-2, data_read.py:103-128)."""
import numpy as np
import pytest

from distancetransform_depthcompletion_b200 import data_read, synth
from oracle import oracle as O


def _frames():
    rng = np.random.default_rng(3)
    x = synth.kitti_frame(2)
    # plant outliers: far points right next to near ones (the filter drops the far ones)
    ys, xs = np.nonzero(x > 0)
    pick = rng.choice(len(ys), 200, replace=False)
    x[ys[pick], xs[pick]] += np.float32(30.0)
    dense = (np.round(rng.uniform(1, 80, (40, 64)) * 256) / 256).astype(np.float32)      # every pixel is evaluated
    signed = x[150:200, 300:420].copy()
    signed[::7, ::5] = np.float32(-5.0)                                                   # negative neighbours
    return [x, synth.kitti_frame(3, beam_step=4), x[:9, :13].copy(), x[200:203, :].copy(), x[:, 600:602].copy(),
            dense, signed, x[:, 1:1216].copy()]


@pytest.mark.gpu
@pytest.mark.skipif(not O.have_cv2(), reason="cv2 absent")
def test_gpu_matches_cv2_port():
    for f in _frames():
        want = O.cv2_port_outlier_removal(f)
        got = data_read.outlier_removal(f[None, :, :, None])
        assert got.dtype == np.float32 and got.shape == f.shape
        assert np.array_equal(got, want)              # KITTI-grid depths: sums are exact in float32
    x = _frames()[0]
    assert (data_read.outlier_removal(x) != x).sum() > 100          # the planted outliers are removed
    with pytest.raises(TypeError):
        data_read.outlier_removal(x.astype(np.float64))
