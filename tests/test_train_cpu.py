"""Training callbacks (SURVEY.md section 8 f4) on the CPU: the oracle's restatement of
HoughTreeFunctions::{impurity, early_stop} (src/hough/houghforest.rs:250-311) against values worked
out by hand, and the host-side pieces of depthhead_b200.train (param_set / scale_and_replace,
sample extraction) against the oracle and the reference's own known answers."""
import math

import numpy as np
import pytest

import oracle
from depthhead_b200 import IntrinsicMatrix, synth, train


def _ln(x):
    return 0.0 if x == 0.0 else math.log(x)


def test_impurity_by_hand():
    # 6 samples: objects 0,1,2,4; left = [0,1,3], right = [2,4,5]
    is_obj = np.array([1, 1, 1, 0, 1, 0], np.uint8)
    off = np.array([[1, 2, 3], [3, 1, 0], [0, 0, 1], [9, 9, 9], [2, 5, 1], [7, 7, 7]], np.float32)
    rot = np.array([[10, 0, 5], [20, 5, 5], [0, 1, 2], [8, 8, 8], [4, 3, 1], [6, 6, 6]], np.float64)
    left, right = [0, 1, 3], [2, 4, 5]
    v, st, bad = oracle.train_impurity(is_obj, off, rot, left, right, depth=3, steepness=5.0)
    assert not bad and list(st["n"]) == [3, 3] and list(st["n_pos"]) == [2, 2]

    def entropy(p):
        return p * _ln(p) + (1 - p) * _ln(1 - p)

    def cov_det(v):  # two points: covariance of rank one, determinant exactly 0 up to rounding
        m = (v[0] + v[1]) / 2.0
        c = sum(np.outer(x - m, x - m) for x in v) / 1.0
        return (c[0, 0] * (c[1, 1] * c[2, 2] - c[1, 2] * c[2, 1]) - c[1, 0] * (c[0, 1] * c[2, 2] - c[0, 2] * c[2, 1])
                + c[2, 0] * (c[0, 1] * c[1, 2] - c[0, 2] * c[1, 1]))
    dl = cov_det(off[[0, 1]].astype(np.float64)) + cov_det(rot[[0, 1]])
    dr = cov_det(off[[2, 4]].astype(np.float64)) + cov_det(rot[[2, 4]])
    assert st["det_off"][0] + st["det_rot"][0] == dl and st["det_off"][1] + st["det_rot"][1] == dr
    reg = 0.5 * (math.log(dl) if dl > 0 else 0.0) + 0.5 * (math.log(dr) if dr > 0 else 0.0)
    want = -(0.5 * entropy(2 / 3) + 0.5 * entropy(2 / 3)) + (1 - math.exp(-(3 / 5.0))) * reg
    assert v == want
    assert oracle.train_impurity_from_stats(st, 3, 5.0) == v
    # a side without objects contributes 0 to the regression term, and ln!(0) = 0 in its entropy
    v2, st2, _ = oracle.train_impurity(is_obj, off, rot, [3, 5], [0, 1, 2, 4], depth=0, steepness=5.0)
    assert list(st2["n_pos"]) == [0, 4] and math.isnan(st2["det_off"][0])
    assert v2 == -(2 / 6 * 0.0 + 4 / 6 * 0.0) + (1 - math.exp(-0.0)) * 0.0   # depth 0: the weight 1 - e^0 is 0
    # a single object on a side: 0/0 covariance -> NaN determinant -> neither match arm -> 0
    v3, st3, _ = oracle.train_impurity(is_obj, off, rot, [0, 3], [1, 2, 4, 5], depth=2, steepness=5.0)
    assert st3["n_pos"][0] == 1 and math.isnan(st3["det_off"][0])
    assert math.isfinite(v3)


def test_early_stop():
    is_obj = np.array([0, 0, 1, 0], np.uint8)
    assert oracle.train_early_stop(is_obj, [0, 1, 3], 0, 15, 1)        # no object left (houghforest.rs:303-305)
    assert not oracle.train_early_stop(is_obj, [0, 2], 3, 15, 2)
    assert oracle.train_early_stop(is_obj, [0, 2], 15, 15, 2)          # depth >= max_depth
    assert oracle.train_early_stop(is_obj, [0, 2], 3, 15, 3)           # len < min_subset_size
    hl = train.HoughLearning(10, 80, 80, 15, 1, 100, 0.3, 10, 3, 5.0)
    for idx, depth in (([0, 1, 3], 0), ([0, 2], 3), ([0, 2], 15), ([0, 1, 2], 3)):
        assert hl.early_stop(depth, is_obj[idx]) == oracle.train_early_stop(is_obj, idx, depth, 15, 3)


def test_scale_and_replace_known_answers():
    # the reference's own test vectors (types.rs:454-474) through the vectorised port
    cases = [((100, 100), 0.5, 0.0, 0.0, (0, 0, 50, 50)), ((100, 100), 0.5, 1.0, 1.0, (50, 50, 50, 50)),
             ((100, 100), 0.5, 0.5, 0.5, (25, 25, 50, 50))]
    for (w, h), s, rx, ry, (x, y, ww, hh) in cases:
        x0, y0, x1, y1 = train.scale_and_replace(w, h, s, np.array([rx]), np.array([ry]))
        assert (int(x0[0]), int(y0[0]), int(x1[0] - x0[0]), int(y1[0] - y0[0])) == (x, y, ww, hh)
    # against the oracle's restatement on random arguments, the trained shape included
    rng = np.random.default_rng(1)
    for w, h, s in ((80, 80, 0.3), (64, 48, 0.5), (33, 57, 0.77)):
        u, v = rng.random(50), rng.random(50)
        x0, y0, x1, y1 = train.scale_and_replace(w, h, s, u, v)
        for i in range(50):
            out = np.zeros(4, np.uint32)
            r = np.array([0, 0, w, h], np.uint32)
            oracle.lib().orc_rect_scale_and_replace(r.ctypes.data, s, float(u[i]), float(v[i]), out.ctypes.data)
            assert (int(x0[i]), int(y0[i]), int(x1[i] - x0[i]), int(y1[i] - y0[i])) == tuple(int(t) for t in out)


def test_param_set_shapes():
    hl = train.HoughLearning(10, 80, 80, 15, 1, 100, 0.3, 10, 20, 5.0)
    rects, thr = hl.param_set(np.random.default_rng(0), 500)
    assert rects.shape == (500, 8) and thr.shape == (500,)
    for k in (0, 4):
        assert np.all(rects[:, k + 2] - rects[:, k] == 24) and np.all(rects[:, k + 3] - rects[:, k + 1] == 24)
        assert rects[:, k].min() >= 0 and rects[:, k + 2].max() <= 80
    assert thr.min() >= -256.0 and thr.max() < 256.0
    with pytest.raises(ValueError):
        train.HoughLearning(10, 80, 80, 15, 1, 100, 1.5, 10, 20, 5.0)
    with pytest.raises(ValueError):
        train.HoughLearning(10, 80, 80, 15, 1, 100, 0.3, 0, 20, 5.0)
    with pytest.raises(ValueError):
        train.HoughLearning(10, 80, 80, 15, 1, 100, 0.3, 10, 20, 0.0)


def test_extract_samples_against_oracle_backprojection():
    frames, centres, rots, masks = synth.make_frames(1, seed=3, with_truth=True)
    K = IntrinsicMatrix.default_kinect_intrinsic()
    org, flag, offs, rr = train.extract_samples(frames[0], masks[0], K, centres[0], rots[0], 10, 80, 80)
    assert len(org) == len(flag) == len(offs) == len(rr) > 0 and flag.any() and not flag.all()
    # every window is non-background, in sliding-window order
    for (x0, y0) in org[:50]:
        assert frames[0][y0:y0 + 80, x0:x0 + 80].any()
    assert np.all(np.diff(org[:, 1] * 10000 + org[:, 0]) > 0)
    # offsets = img_to_space_coord(centre pixel) - head centre, in f32 like the reference
    for i in np.flatnonzero(flag)[:20]:
        x, y = org[i] + 40
        p3 = np.zeros(3, np.float32)
        xy = np.array([x, y], np.float32)
        oracle.lib().orc_img_to_space(synth.KINECT_K.ctypes.data, xy.ctypes.data, float(frames[0][y, x]), p3.ctypes.data)
        assert np.array_equal((p3 - centres[0]).view(np.uint32), offs[i].view(np.uint32))
        assert masks[0][y, x] != 0
    assert np.array_equal(rr[0], rots[0].astype(np.float64))


def _avg(patch, x0, y0, x1, y1):
    # average_value_in_rect (types.rs:317-339): integer sum, then sum as f64 / count as f64
    return float(int(patch[y0:y1, x0:x1].astype(np.int64).sum())) / float((x1 - x0) * (y1 - y0))


def _cov_det(pts):
    # estimate_mean_cov (meancov_estimation.rs:359-378) and Mat3::det (:339-343) in plain Python floats
    m = [0.0, 0.0, 0.0]
    for p in pts:
        m = [m[k] + float(p[k]) for k in range(3)]
    m = [v / len(pts) for v in m]
    c = [[0.0] * 3 for _ in range(3)]
    for p in pts:
        d = [float(p[k]) - m[k] for k in range(3)]
        c = [[c[a][b] + d[a] * d[b] for b in range(3)] for a in range(3)]
    c = [[v / (len(pts) - 1) for v in row] for row in c]
    return (c[0][0] * (c[1][1] * c[2][2] - c[1][2] * c[2][1]) - c[1][0] * (c[0][1] * c[2][2] - c[0][2] * c[2][1])
            + c[2][0] * (c[0][1] * c[1][2] - c[0][2] * c[1][1]))


def _impurity_by_hand(is_obj, off, rot, left, right, depth, steepness):
    def entropy(side):
        p = sum(int(is_obj[i]) for i in side) / len(side)
        return p * _ln(p) + (1 - p) * _ln(1 - p)

    def reglog(side):
        pos = [i for i in side if is_obj[i]]
        if len(pos) < 2:   # none, or one: 0/0 covariance, NaN determinant, neither match arm
            return 0.0
        x = _cov_det(off[pos]) + _cov_det(rot[pos])
        return math.log(x) if x > 0 else 0.0
    n = len(left) + len(right)
    lf, rf = len(left) / n, len(right) / n
    return -(lf * entropy(left) + rf * entropy(right)) + (1 - math.exp(-(depth / steepness))) * (lf * reglog(left) + rf * reglog(right))


def test_oracle_trainer_grows_a_tree_by_hand():
    """HoughLearning.train_forest on oracle.OracleTrainSet: the root's candidates scored by hand, the
    root takes the smallest of them, and the grown tree partitions its samples as the driver states
    (DESIGN.md section 9): children[bit] gets binarize == bit, in set order; leaf prob = objects / samples."""
    rng = np.random.default_rng(17)
    n = 40
    patches = rng.integers(0, 2000, (n, 12, 10)).astype(np.uint16)
    patches[: n // 2, :6, :] += 1500                       # something for the features to find
    is_obj = (np.arange(n) < n // 2).astype(np.uint8)
    rng.shuffle(is_obj)
    off = rng.normal(0.0, 40.0, (n, 3)).astype(np.float32)
    rot = rng.normal(0.0, 20.0, (n, 3))
    hl = train.HoughLearning(1, 10, 12, 4, 1, 32, 0.5, 12, 4, 5.0)
    ts = oracle.OracleTrainSet(patches, is_obj, off, rot)
    arr = hl.train_forest(ts, train.CounterRng(9))
    # the driver's first draws: the subset, then the root's candidates
    r = train.CounterRng(9)
    subset = r.permutation(n)[:32]
    rects, thr = hl.param_set(r, 12)
    assert np.all(rects[:, 2] - rects[:, 0] == 5) and np.all(rects[:, 3] - rects[:, 1] == 6)
    hand = []
    for j in range(12):
        bits = np.array([_avg(patches[i], *rects[j, :4]) - _avg(patches[i], *rects[j, 4:]) > thr[j] for i in subset])
        assert np.array_equal(bits.astype(np.uint8), oracle.train_binarize(patches, subset, rects[j], thr[j]))
        left, right = subset[~bits], subset[bits]
        hand.append(np.nan if len(left) == 0 or len(right) == 0 else _impurity_by_hand(is_obj, off, rot, left, right, 0, 5.0))
    st = ts.score_level(subset, [0, 32], rects[None], thr[None], 0, 5.0)[0]
    assert np.array_equal(np.isnan(st["impurity"]), np.isnan(hand)) and np.count_nonzero(~np.isnan(hand)) >= 6
    ok = ~np.isnan(hand)
    assert np.allclose(st["impurity"][ok], np.asarray(hand)[ok], rtol=1e-12, atol=1e-12)
    best = int(np.flatnonzero(ok)[np.argmin(np.asarray(hand)[ok])])
    assert arr["tree_node_off"][1] > 0, "the root did not split"
    assert np.array_equal(arr["rects"][0], rects[best]) and arr["threshold"][0] == thr[best]
    # route the subset down the tree: every leaf holds the objects that reach it, in set order
    reach = {}

    def walk(node, idx):
        if node < 0:
            reach[~node] = idx
            return
        rr, t = arr["rects"][node], arr["threshold"][node]
        b = np.array([_avg(patches[i], *rr[:4]) - _avg(patches[i], *rr[4:]) > t for i in idx], bool)
        kids = arr["child"][node]
        walk(int(kids[0]), idx[~b])
        walk(int(kids[1]), idx[b])
    walk(0, subset)
    assert sorted(reach) == list(range(len(arr["prob"])))
    assert sum(len(v) for v in reach.values()) == 32
    for leaf, idx in reach.items():
        pos = idx[is_obj[idx] != 0]
        assert arr["prob"][leaf] == len(pos) / len(idx)
        v0, v1 = arr["vote_off"][leaf], arr["vote_off"][leaf + 1]
        assert np.array_equal(arr["offsets"][v0:v1], off[pos]) and np.array_equal(arr["rotations"][v0:v1], rot[pos])
