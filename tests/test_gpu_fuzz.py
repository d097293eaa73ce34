"""Seeded differential fuzzing: the CUDA path (through the C ABI) against the CPU oracle on
configurations drawn at random from the whole parameter space of the prediction path
(prediction.rs:512-760): patch size, rectangle scale (uniform box sums or ragged rectangles),
tree count / depth / sparsity, node order in the file, stride, image size,
gaussian sigma, mean-shift iterations, caller seeds, frame content.  Every stage is compared as
in test_gpu_parity (leaf ids and accumulators bit-exact, trajectories and the pose identical).
Every frame and the batch run on both gate paths: patch_gate_kernel (probability codes where the
forest has box-sum rectangles) with the seed grids from gated-patch lists, and the fold inside
gate_coarse_kernel (test_gpu_parity.list_ctx / fold_ctx).  The random shapes give patch counts that
are rarely multiples of patch_gate_kernel's 1024 patches per CTA.
The draws depend only on the case number, so a failure reproduces with `-k "case17"`.
"""
import numpy as np
import pytest

import oracle
from depthhead_b200 import HoughPrediction, IntrinsicMatrix, synth
from test_gpu_parity import _compare_frame, fold_ctx, list_ctx  # noqa: F401 (module fixtures)

pytestmark = pytest.mark.gpu

N_CASES = 96


def _draw(case):
    rng = np.random.default_rng([case, 6007])
    sub_w, sub_h = (int(v) for v in rng.integers(12, 121, 2))
    if rng.random() < 0.4:
        sub_w, sub_h = 80, 80
    scale = float(rng.choice([0.1, 0.2, 0.3, 0.3, 0.5, 0.75, 1.0]))
    if int(sub_w * scale) < 1 or int(sub_h * scale) < 1:
        scale = 0.3
    sparse = rng.random() < 0.4
    forest = dict(seed=1000 + case, n_trees=int(rng.integers(1, 8)), max_depth=int(rng.integers(1, 10)),
                  sub_w=sub_w, sub_h=sub_h, rect_scale=scale,
                  stop_prob=float(rng.uniform(0.05, 0.4)) if sparse else 0.0,
                  votes_lo=int(rng.integers(1, 4)), votes_hi=int(rng.integers(4, 40)),
                  shuffle_nodes=bool(rng.random() < 0.5), ragged_rects=bool(rng.random() < 0.3),
                  tie_thresholds=bool(rng.random() < 0.2))
    h = int(rng.integers(sub_h, sub_h + 260))
    w = int(rng.integers(sub_w, sub_w + 330))
    if rng.random() < 0.25:
        h, w = 480, 640
    model = dict(stepwidth=int(rng.integers(1, 14)) if max(h, w) < 400 else int(rng.integers(4, 14)),
                 gaussian_sigma=float(rng.choice([0.5, 2.0, 8.0, 8.0, 25.0])),
                 meanshift_iterations=int(rng.choice([0, 1, 3, 20, 20, 40])))
    return rng, forest, model, h, w


def _frames(rng, h, w, case):
    full = synth.make_frames(2, seed=300 + case)
    if (h, w) == (480, 640):
        person = [full[0], full[1]]
    else:
        # crops around the person, at a random offset so the head sits anywhere (or is cut off)
        y0 = int(rng.integers(0, 480 - h + 1)) if h <= 480 else 0
        x0 = int(rng.integers(0, 640 - w + 1)) if w <= 640 else 0
        person = []
        for f in full:
            d = np.zeros((h, w), np.uint16)
            c = f[y0:y0 + h, x0:x0 + w]
            d[:c.shape[0], :c.shape[1]] = c
            person.append(d)
    noise = rng.integers(0, 65536, (h, w)).astype(np.uint16)
    noise[rng.random((h, w)) < 0.5] = 0
    return person + [noise]


@pytest.mark.parametrize("case", range(N_CASES), ids=lambda c: "case%d" % c)
def test_random_configuration(list_ctx, fold_ctx, case):
    rng, forest, model, h, w = _draw(case)
    arr = synth.make_forest(**forest)
    js = synth.forest_to_json(arr, **model)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    frames = _frames(rng, h, w, case)
    for i, d in enumerate(frames):
        mid = rot = None
        if rng.random() < 0.3:
            mid = [float(v) for v in rng.uniform([-200, -150, 500], [200, 150, 1400])]
        if rng.random() < 0.3:
            rot = [float(v) for v in rng.uniform(-1.0, 1.0, 3)]  # radians (prediction.rs:437-460)
        tr = of.predict(d, synth.KINECT_K, mid, rot, mode=oracle.MODE_SAT, keep=True)
        for c in (list_ctx, fold_ctx):
            _compare_frame(c, hp, of, d, mid, rot, trace=tr)
    # the batch entry point on the same frames (no caller seeds)
    outs = [hp.predict_batch(np.stack(frames), IntrinsicMatrix.default_kinect_intrinsic(), ctx=c) for c in (list_ctx, fold_ctx)]
    for i, d in enumerate(frames):
        tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
        for out in outs:
            assert np.array_equal(out["mid_point"][i], tr.mid_point)
            assert np.array_equal(out["rotation"][i].view(np.uint64), tr.rotation.view(np.uint64))
