"""Writes tests/golden/png_frames.npz: 16-bit grayscale PNG files encoded by libpng (through PIL and through cv2, at
several compression settings) with the samples they hold, so that the decoder is checked against a writer other than
the test oracle's.  Run from the repository root:  python tests/golden/make_png_golden.py"""
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import png_oracle as P  # noqa: E402


def main():
    import cv2
    from PIL import Image
    rng = np.random.default_rng(2024)
    frames = {
        "kitti64": P.kitti_png_samples(21),
        "kitti16_rows": P.kitti_png_samples(22, beams=16)[96:224],
        "noise_small": rng.integers(0, 65536, (37, 53)).astype(np.uint16),
    }
    out = {}
    for name, x in frames.items():
        for level in (0, 1, 6, 9):
            buf = io.BytesIO()
            Image.fromarray(x).save(buf, format="PNG", compress_level=level)
            out[f"pil_l{level}_{name}"] = (buf.getvalue(), x)
        for level in (1, 3, 9):
            ok, enc = cv2.imencode(".png", x, [cv2.IMWRITE_PNG_COMPRESSION, level])
            assert ok
            out[f"cv2_l{level}_{name}"] = (enc.tobytes(), x)
        ok, enc = cv2.imencode(".png", x, [cv2.IMWRITE_PNG_STRATEGY, cv2.IMWRITE_PNG_STRATEGY_RLE])
        out[f"cv2_rle_{name}"] = (enc.tobytes(), x)
    arrays = {}
    for k, (png, x) in out.items():
        assert np.array_equal(np.array(Image.open(io.BytesIO(png))).astype(np.uint16), x), k
        arrays[k + "/png"] = np.frombuffer(png, np.uint8)
        arrays[k + "/samples"] = x
    np.savez_compressed(os.path.join(HERE, "png_frames.npz"), **arrays)
    print(len(out), "files,", sum(len(p) for p, _ in out.values()), "bytes")


if __name__ == "__main__":
    main()
