"""Generates tests/golden/*.npz by running the REFERENCE itself (a checkout named by $DTFILL_REFERENCE).

The reference ships no tests or golden vectors, so the pin is its own output on
seeded synthetic inputs:  solution_DeepNet/tools.py (imported with a stub `tensorflow` module and the `cv2` it
forgot to import injected), the two functions of solution_DeepNet/eval_NYU.py:114-133 (AST-extracted, that
script builds a TF model at import), evaluation.py's Result / Result_NYU, live cv2 4.13.0, and the DT-pooling lines of net.py:71-123 / demo.py:65-149
(AST-extracted, run on tests/golden/tf_numpy_shim.py: TensorFlow itself is absent).
The vectors are committed so that the tests need no reference checkout.

    python tests/golden/make_golden.py [pool]   (from the repo root; needs a reference checkout and cv2)
    python tests/golden/make_golden.py cv2      (cv2_masks.npz alone; needs cv2 only)
"""
import ast
import hashlib
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = os.environ.get("DTFILL_REFERENCE", "/root/reference")
OUT = os.path.dirname(os.path.abspath(__file__))


def load_reference():
    import cv2
    sys.modules.setdefault("tensorflow", types.ModuleType("tensorflow"))
    sys.path.insert(0, os.path.join(REF, "solution_DeepNet"))
    sys.path.insert(0, REF)
    import tools
    import evaluation
    tools.cv2 = cv2                               # tools.py never imports cv2 (SURVEY.md section 0)
    ns = {"np": np, "cv2": cv2}
    tree = ast.parse(open(os.path.join(REF, "solution_DeepNet", "eval_NYU.py")).read())
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in ("nearest_point", "Distance_Transform"):
            exec(compile(ast.Module([node], []), "eval_NYU.py", "exec"), ns)
    return tools, evaluation, ns["nearest_point"], ns["Distance_Transform"], cv2


def load_pooling_reference():
    """The reference's own DT-pooling lines, AST-extracted and run on tf_numpy_shim (TensorFlow is absent here):
    net.py:71-123 (methods create_weight_matrix / generate_multi_channel of the first model class) and
    demo.py:65-76, :107-149.  Returns (net_pool(data, mask, table_size, scale_num), demo_pool(data, table_size,
    scale_range, scale_num)); inputs and outputs carry the reference's shapes ([B,H,W,1] in, [B,H,W] levels out)."""
    sys.path.insert(0, OUT)
    import tf_numpy_shim as tf
    ns = {"np": np, "tf": tf}
    tree = ast.parse(open(os.path.join(REF, "solution_DeepNet", "net.py")).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef)
               and any(isinstance(m, ast.FunctionDef) and m.name == "generate_multi_channel" for m in n.body))
    for m in cls.body:
        if isinstance(m, ast.FunctionDef) and m.name in ("create_weight_matrix", "generate_multi_channel"):
            m.name = "net_" + m.name
            exec(compile(ast.Module([m], []), "net.py", "exec"), ns)
    dns = {"np": np, "tf": tf}
    tree = ast.parse(open(os.path.join(REF, "solution_DeepNet", "demo.py")).read())
    for n in tree.body:
        if isinstance(n, ast.FunctionDef) and n.name in ("create_weight_matrix", "generate_multi_channel"):
            exec(compile(ast.Module([n], []), "demo.py", "exec"), dns)

    def net_pool(data, mask, table_size=7, scale_num=4):
        me = types.SimpleNamespace(table_size=table_size, scale_num=scale_num)
        me.create_weight_matrix = lambda: ns["net_create_weight_matrix"](me)
        me.weights_matrix = me.create_weight_matrix()                     # net.py:34
        return ns["net_generate_multi_channel"](me, data, mask)

    def demo_pool(data, table_size=11, scale_range=90.0, scale_num=4):
        return dns["generate_multi_channel"](data, table_size, scale_range=scale_range, scale_num=scale_num)

    net_pool.create_weight_matrix = lambda t: ns["net_create_weight_matrix"](types.SimpleNamespace(table_size=t))
    demo_pool.create_weight_matrix = dns["create_weight_matrix"]
    return net_pool, demo_pool


def pool_cases():
    """Inputs of the DT-pooling fixtures: name -> (raw depth [B,H,W] float32, table_size, scale_num)."""
    from distancetransform_depthcompletion_b200 import synth
    rng = np.random.default_rng(77)
    a = np.stack([synth.kitti_frame(5)[120:184, 200:360], synth.kitti_frame(6, beam_step=4)[120:184, 200:360]])
    b = np.stack([((rng.random((48, 96)) < 0.03) * rng.uniform(1, 80, (48, 96))).astype(np.float32),
                  np.zeros((48, 96), np.float32)])
    c = synth.nyu_frame(2)[None, 100:150, 200:283]                      # odd width
    return {"kitti_t7_s4": (a, 7, 4), "kitti_t5_s3": (a, 5, 3), "kitti_t3_s4": (a, 3, 4), "kitti_t9_s3": (a, 9, 3),
            "random_t7_s4": (b, 7, 4), "random_t11_s3": (b, 11, 3), "nyu_t7_s2": (c, 7, 2)}


def pool_inputs(x):
    """net.py:464-467, :486: validity mask x > 0.1, data x / 90 * mask, both float32 [B,H,W,1]."""
    x4 = x[..., None].astype(np.float32)
    mask = (x4 > 0.1).astype(np.float32)
    return (x4 / np.float32(90.0) * mask).astype(np.float32), mask


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def write_pool_golden():
    # DT pooling (net.py:83-123, demo.py:107-149): the reference lines on the numpy stand-in for TensorFlow
    net_pool, demo_pool = load_pooling_reference()
    pool = {}
    for name, (x, t, s) in pool_cases().items():
        data, mask = pool_inputs(x)
        lv = net_pool(data, mask, t, s)
        assert lv[0] is data and all(v is None for v in lv[s:])
        for k in range(1, s):
            pool[f"net/{name}/l{k + 1}"] = np.asarray(lv[k], np.float32)
        if t in (7, 11):
            # demo.py:108 unpacks np.shape(np.squeeze(lidar_data)) into two names: one frame per call
            dl = [demo_pool(x[i:i + 1, :, :, None].astype(np.float32), t, 90.0, s) for i in range(len(x))]
            for k in range(s):
                pool[f"demo/{name}/l{k + 1}"] = np.concatenate([np.asarray(d[k], np.float32) for d in dl])
    for t in (3, 7, 11):
        pool[f"weights/net_t{t}"] = net_pool.create_weight_matrix(t)
        pool[f"weights/demo_t{t}"] = demo_pool.create_weight_matrix(t)
    np.savez_compressed(os.path.join(OUT, "dt_pool.npz"), **pool)


def random_masks():
    """Inputs of cv2_masks.npz: 300 uint8 masks of 1..40 x 1..60 pixels (0 = source), densities 1 % .. 90 %."""
    rng = np.random.default_rng(0)
    masks = []
    for _ in range(300):
        H, W = int(rng.integers(1, 41)), int(rng.integers(1, 61))
        dens = rng.choice([0.01, 0.05, 0.2, 0.5, 0.9])
        masks.append((rng.random((H, W)) >= dens).astype(np.uint8))
    return masks


def write_cv2_golden():
    """cv2.distanceTransformWithLabels(DIST_L1, 5, DIST_LABEL_PIXEL) -- the call at tools.py:9 -- on random_masks(),
    concatenated as flat arrays with the shape of every mask; needs only cv2."""
    import cv2
    masks = random_masks()
    dts, lbls = [], []
    for m in masks:
        dt, lbl = cv2.distanceTransformWithLabels(m, cv2.DIST_L1, 5, labelType=cv2.DIST_LABEL_PIXEL)
        assert dt.dtype == np.float32 and np.array_equal(dt, np.rint(dt)) and lbl.max() < 2 ** 15
        dts.append(dt.ravel())
        lbls.append(lbl.ravel())
    np.savez_compressed(os.path.join(OUT, "cv2_masks.npz"), cv2_version=np.array(cv2.__version__),
                        shapes=np.array([m.shape for m in masks], np.int32),
                        mask=np.concatenate([m.ravel() for m in masks]),
                        dt_u16=np.concatenate(dts).astype(np.uint16), lbl_i16=np.concatenate(lbls).astype(np.int16))


def main():
    from distancetransform_depthcompletion_b200 import synth
    tools, evaluation, nyu_nearest_point, nyu_distance_transform, cv2 = load_reference()

    # ---- 1. small frames, full expected outputs (KITTI thresholds, via the raw cv2 call + tools' gather lines)
    small = {}
    rng = np.random.default_rng(11)
    cases = dict(synth.adversarial_frames())
    for t in range(12):
        H, W = int(rng.integers(2, 48)), int(rng.integers(2, 70))
        dens = float(rng.choice([0.01, 0.05, 0.2, 0.6]))
        f = ((rng.random((H, W)) < dens) * rng.uniform(1.0, 60.0, (H, W))).astype(np.float32)
        if not (f > 0.1).any():
            f[H // 2, W // 2] = 4.0
        cases[f"random_{t}"] = f
    for name, f in cases.items():
        value_mask = np.asarray(1.0 - f > 0.1).astype(np.uint8)                      # tools.py:8
        dt, lbl = cv2.distanceTransformWithLabels(value_mask, cv2.DIST_L1, 5, labelType=cv2.DIST_LABEL_PIXEL)
        with_value = f > 0.1                                                         # tools.py:22
        depth_list = f[with_value]                                                   # tools.py:24
        small[f"{name}/in"] = f
        small[f"{name}/dt"] = dt
        small[f"{name}/lbl"] = lbl
        small[f"{name}/depth"] = depth_list[lbl.reshape(1, -1) - 1].reshape(f.shape)  # tools.py:25-27
    np.savez_compressed(os.path.join(OUT, "small_frames.npz"), **small)

    # ---- 2. full-size frames through the reference functions themselves
    full = {}
    xb = synth.kitti_batch([0])                                                      # 64 beams
    ref = tools.DT_complete_batch(xb)
    dt, lbl = tools.nearest_point(xb[0, :, :, 0])
    full["kitti64_seed0/lbl"] = lbl
    full["kitti64_seed0/dt_u16"] = dt.astype(np.uint16)
    assert np.array_equal(ref[0, :, :, 0], xb[0, :, :, 0][xb[0, :, :, 0] > 0.1][lbl.reshape(-1) - 1].reshape(352, 1216))
    x8 = synth.kitti_batch([5], beam_step=8)
    dt, lbl = tools.nearest_point(x8[0, :, :, 0])
    full["kitti8_seed5/lbl"] = lbl
    full["kitti8_seed5/dt_u16"] = dt.astype(np.uint16)
    xn = synth.nyu_frame(3)
    dt, lbl = nyu_nearest_point(xn)
    full["nyu_seed3/lbl"] = lbl
    full["nyu_seed3/dt_u16"] = dt.astype(np.uint16)
    np.savez_compressed(os.path.join(OUT, "full_frames.npz"), **full)

    # ---- 3. checksums of reference outputs on more seeds (cheap to store, strong to compare)
    sums = {}
    for step in (1, 2, 4, 8):
        for seed in range(4):
            xb = synth.kitti_batch([seed], beam_step=step)
            ref = tools.DT_complete_batch(xb)
            dt, lbl = tools.nearest_point(xb[0, :, :, 0])
            sums[f"kitti_b{64 // step}_s{seed}"] = np.array([sha(ref[0, :, :, 0]), sha(dt), sha(lbl)])
    for seed in range(4):
        xn = synth.nyu_frame(seed)
        d = nyu_distance_transform(xn[None, :, :, None])
        dt, lbl = nyu_nearest_point(xn)
        sums[f"nyu_s{seed}"] = np.array([sha(d), sha(dt), sha(lbl)])
    xq = synth.nyu_frame(9, 240, 320)                                               # reference default NYU size
    d = nyu_distance_transform(xq)
    dt, lbl = nyu_nearest_point(xq)
    sums["nyu240_s9"] = np.array([sha(d), sha(dt), sha(lbl)])
    np.savez_compressed(os.path.join(OUT, "checksums.npz"), **sums)

    # ---- 4. metrics from evaluation.py on NN-filled frames
    met = {}
    for seed in range(3):
        xb = synth.kitti_batch([seed])
        fill = tools.DT_complete_batch(xb)[0, :, :, 0]
        gt = synth.kitti_gt(seed)
        R = evaluation.Result()
        R.evaluate(fill, gt)
        met[f"kitti_s{seed}"] = np.array([R.mse, R.rmse, R.mae, R.irmse, R.imae])
        R.evaluate(np.maximum(fill, 0.9), gt.astype(np.float32))
        met[f"kitti_f32gt_s{seed}"] = np.array([R.mse, R.rmse, R.mae, R.irmse, R.imae])
    for seed in range(3):
        xn, g = synth.nyu_frame(seed, return_dense=True)
        fill = nyu_distance_transform(xn)
        R = evaluation.Result_NYU()
        R.evaluate(fill, g)
        met[f"nyu_s{seed}"] = np.array([R.mse, R.rmse, R.mae, R.irmse, R.imae, R.delta1, R.delta2, R.delta3])
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **met)
    write_pool_golden()
    write_cv2_golden()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    if sys.argv[1:] == ["pool"]:          # only dt_pool.npz (the other fixtures stay byte-identical in git)
        write_pool_golden()
    elif sys.argv[1:] == ["cv2"]:         # only cv2_masks.npz (needs cv2, not the reference checkout)
        write_cv2_golden()
    else:
        main()
