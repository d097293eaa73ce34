"""Training on the GPU (csrc/dh_train.cu, DESIGN.md section 9) against the CPU oracle at the shapes,
values and sizes where the scorer can go wrong: every rectangle layout of the training tables,
threshold ties to the ulp, saturated and empty patches, the reference's unreachable!() branch,
levels wider than one launch can hold, training sets built in more than one chunk, the reference's
default root, and whole forests grown on oracle.OracleTrainSet."""
import json

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, IntrinsicMatrix, capi, synth, train

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()
DEPTHS = [(0, 5.0), (4, 5.0), (15, 5.0), (0, 2.5), (4, 2.5), (15, 2.5)]


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def _windows(n_frames, seed, sw, sh, per_image=16):
    """windows of synthetic frames with their truth, half negatives and half positives per frame"""
    frames, centres, rots, masks = synth.make_frames(n_frames, seed=seed, with_truth=True)
    rng = np.random.default_rng(seed)
    P, F, O, R = [], [], [], []
    for i in range(n_frames):
        org, flag, offs, rr = train.extract_samples(frames[i], masks[i], K, centres[i], rots[i], 10, sw, sh)
        pick = np.concatenate([rng.permutation(np.flatnonzero(flag == 0))[:per_image // 2],
                               rng.permutation(np.flatnonzero(flag != 0))[:per_image // 2]])
        for j in pick:
            x0, y0 = org[j]
            P.append(frames[i][y0:y0 + sh, x0:x0 + sw]); F.append(flag[j]); O.append(offs[j]); R.append(rr[j])
    return np.stack(P), np.asarray(F, np.uint8), np.asarray(O, np.float32), np.asarray(R, np.float64)


def _mixed(sw, sh, seed, n_frames=3, n_noise=10, n_sat=3, n_zero=3):
    """windows of synthetic frames, u16 noise, saturated (65535) and all-zero patches, shuffled;
    the made-up patches carry truth at head scale"""
    P, F, O, R = _windows(n_frames, seed, sw, sh)
    rng = np.random.default_rng(seed + 1)
    n_x = n_noise + n_sat + n_zero
    extra = np.concatenate([rng.integers(0, 65536, (n_noise, sh, sw)), np.full((n_sat, sh, sw), 65535),
                            np.zeros((n_zero, sh, sw))]).astype(np.uint16)
    P = np.concatenate([P, extra])
    F = np.concatenate([F, (rng.random(n_x) < 0.5).astype(np.uint8)])
    O = np.concatenate([O, rng.normal(0, 60, (n_x, 3)).astype(np.float32)])
    R = np.concatenate([R, rng.normal(0, 15, (n_x, 3))])
    perm = rng.permutation(len(P))
    return P[perm], F[perm], O[perm], R[perm]


def _same_f64(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64))


def _assert_same_stats(g, o, what=""):
    """every field of the GPU's dh_split_stats equals the oracle's: counts exactly, doubles bit for bit, NaN where NaN"""
    for f in ("n", "n_pos"):
        assert np.array_equal(g[f], o[f]), (what, f, np.argwhere((g[f] != o[f]).any(-1))[:5].tolist())
    for f in ("det_off", "det_rot", "impurity"):
        assert _same_f64(g[f], o[f]), (what, f)


def _corners(sw, sh, rw, rh):
    """candidate rectangles at the origin, at x0 = sw - rw and at y0 = sh - rh (the last column and row of the table)"""
    O, X, Y, XY = (0, 0), (sw - rw, 0), (0, sh - rh), (sw - rw, sh - rh)
    pairs = [(O, XY), (X, Y), (XY, O), (Y, X), (O, X), (Y, O), (XY, Y), (X, XY)]
    return np.array([[a[0], a[1], a[0] + rw, a[1] + rh, b[0], b[1], b[0] + rw, b[1] + rh] for a, b in pairs], np.int32)


def _candidates(patches, nodes, sw, sh, rw, rh, m, seed):
    """per node, m candidates: rectangles at the corners of the table and random ones; thresholds at
    the exact tie a1 - a2 of three samples of the node and one ulp on either side of each, +-0,
    +-inf, NaN and U(-256, 256)"""
    rng = np.random.default_rng(seed)
    corners = _corners(sw, sh, rw, rh)
    R, T = [], []
    for k, s in enumerate(nodes):
        u = rng.random((m, 4))
        x0, y0 = (u[:, 0] * (sw - rw + 1)).astype(np.int32), (u[:, 1] * (sh - rh + 1)).astype(np.int32)
        x1, y1 = (u[:, 2] * (sw - rw + 1)).astype(np.int32), (u[:, 3] * (sh - rh + 1)).astype(np.int32)
        rects = np.stack([x0, y0, x0 + rw, y0 + rh, x1, y1, x1 + rw, y1 + rh], 1).astype(np.int32)
        thr = rng.uniform(-256.0, 256.0, m)
        for t in range(3):                                  # slots 0..8: ties of three samples of the node
            i = int(s[(t * 7 + k) % len(s)]) if len(s) else 0
            tie = oracle.train_feature(patches[i], corners[t])
            for q, v in enumerate((tie, np.nextafter(tie, np.inf), np.nextafter(tie, -np.inf))):
                rects[t * 3 + q], thr[t * 3 + q] = corners[t], v
        for q, v in enumerate((0.0, -0.0, np.inf, -np.inf, np.nan)):   # slots 9..13
            rects[9 + q], thr[9 + q] = corners[3 + q], v
        R.append(rects)
        T.append(thr)
    return np.stack(R), np.stack(T)


def _nodes_of(n, rng, is_obj):
    """everything shuffled, a third, two samples, an empty node, the objects only, the non-objects only"""
    pos, neg = np.flatnonzero(is_obj != 0), np.flatnonzero(is_obj == 0)
    return [rng.permutation(n), rng.permutation(n)[: n // 3], np.array([pos[0], neg[0]]), np.zeros(0, np.int64),
            rng.permutation(pos), neg[::2]]


def _flat(nodes):
    off = np.concatenate([[0], np.cumsum([len(x) for x in nodes])]).astype(np.uint64)
    return np.concatenate(nodes).astype(np.uint32), off


# sub-image -> rectangle.  28x28: general kernel (bw 53, pitch 56); 8x8: kWhole with a rectangle row
# inside one lane; 4x4: general, tiny rectangles; 80x80: bw 1, pitch 4, both rectangles the same;
# 81x61: odd widths (scalar loads); 128x127: the largest accepted rectangle; 25x25: pitch = bw = 56.
SHAPES = [(80, 80, 24, 24), (80, 80, 28, 28), (80, 80, 8, 8), (80, 80, 4, 4), (80, 80, 80, 80), (64, 48, 32, 24),
          (81, 61, 24, 18), (128, 127, 128, 127), (80, 80, 25, 25)]


@pytest.mark.parametrize("sw,sh,rw,rh", SHAPES, ids=["%dx%d-%dx%d" % s for s in SHAPES])
def test_score_and_split_match_the_oracle_at_every_shape(ctx, sw, sh, rw, rh):
    patches, is_obj, offs, rots = _mixed(sw, sh, seed=sw * 1000 + rw)
    n = len(patches)
    ts = train.TrainSet(patches, is_obj, offs, rots, rw, rh, ctx=ctx)
    ots = oracle.OracleTrainSet(patches, is_obj, offs, rots)
    rng = np.random.default_rng(rw * 31 + sh)
    nodes = _nodes_of(n, rng, is_obj)
    idx, off = _flat(nodes)
    m = 24
    rects, thr = _candidates(patches, nodes, sw, sh, rw, rh, m, seed=rw + sw)
    both = 0
    for depth, steep in DEPTHS:
        g = ts.score_level(idx, off, rects, thr, depth, steep)
        o = ots.score_level(idx, off, rects, thr, depth, steep)
        _assert_same_stats(g, o, (depth, steep))
        both = max(both, int(np.count_nonzero(~np.isnan(o["impurity"]))))
    if (rw, rh) != (sw, sh):      # else both rectangles are the patch: a1 - a2 = 0 and one side is always empty
        assert both >= 2 * m      # candidates with both sides populated, not only NaN
    # the bits of one chosen candidate per node, empty node included, against binarize
    for j in range(m):
        r, t = rects[:, j], thr[:, j]
        assert np.array_equal(ts.split_level(idx, off, r, t), ots.split_level(idx, off, r, t)), j
    ts.close()


def test_rejected_sizes_stay_argument_errors(ctx):
    patches, is_obj, offs, rots = _mixed(128, 128, seed=5, n_frames=1, n_noise=2, n_sat=1, n_zero=1)
    for rw, rh, code in ((129, 64, capi.DH_E_SHAPE), (64, 129, capi.DH_E_SHAPE), (128, 128, capi.DH_E_SHAPE),
                         (0, 8, capi.DH_E_SHAPE)):
        with pytest.raises(capi.DhError) as e:
            train.TrainSet(patches, is_obj, offs, rots, rw, rh, ctx=ctx)
        assert e.value.code == code, (rw, rh)
    p80 = patches[:, :80, :80].copy()
    with pytest.raises(capi.DhError) as e:
        train.TrainSet(p80, is_obj, offs, rots, 81, 8, ctx=ctx)
    assert e.value.code == capi.DH_E_SHAPE
    # a candidate rectangle one pixel past the sub-image is an argument error in both calls
    ts = train.TrainSet(p80, is_obj, offs, rots, 24, 24, ctx=ctx)
    idx, off = _flat([np.arange(len(p80))])
    for r in ([57, 0, 81, 24, 0, 0, 24, 24], [0, 0, 24, 24, 0, 57, 24, 81], [-1, 0, 23, 24, 0, 0, 24, 24]):
        rr = np.array([r], np.int32)
        with pytest.raises(capi.DhError) as e:
            ts.score_level(idx, off, rr[None], np.zeros((1, 1)), 0, 5.0)
        assert e.value.code == capi.DH_E_ARG
        with pytest.raises(capi.DhError) as e:
            ts.split_level(idx, off, rr, np.zeros(1))
        assert e.value.code == capi.DH_E_ARG
    ts.close()


def _large_offsets(seed, n_frames=4):
    """windows whose positives carry offsets spread over +-1e2 .. 1e4 mm: covariances of three or so
    such points are rank-deficient and their determinants round far below -0.001"""
    P, F, O, R = _windows(n_frames, seed, 80, 80)
    rng = np.random.default_rng(seed)
    O = (rng.choice([-1.0, 1.0], O.shape) * 10.0 ** rng.uniform(2, 4, O.shape)).astype(np.float32)
    return P, F, O, R


def test_unreachable_branch_is_skipped_like_the_oracle(ctx):
    patches, is_obj, offs, rots = _large_offsets(23)
    n = len(patches)
    ts = train.TrainSet(patches, is_obj, offs, rots, 24, 24, ctx=ctx)
    ots = oracle.OracleTrainSet(patches, is_obj, offs, rots)
    rng = np.random.default_rng(3)
    pos, neg = np.flatnonzero(is_obj != 0), np.flatnonzero(is_obj == 0)
    # small nodes of three to six positives and a few negatives
    nodes = [rng.permutation(np.concatenate([rng.choice(pos, 3 + k % 4, replace=False), rng.choice(neg, 2, replace=False)]))
             for k in range(24)]
    idx, off = _flat(nodes)
    hl = train.HoughLearning(10, 80, 80, 15, 1, 1000, 0.3, 32, 20, 5.0)
    cands = [hl.param_set(rng, 32) for _ in nodes]
    rects = np.stack([c[0] for c in cands])
    thr = rng.uniform(-60, 60, (len(nodes), 32))
    for depth, steep in ((4, 5.0), (15, 2.5)):
        g = ts.score_level(idx, off, rects, thr, depth, steep)
        o = ots.score_level(idx, off, rects, thr, depth, steep)
        assert np.count_nonzero(ots.last_bad) >= 20
        empty = (o["n"] == 0).any(-1)
        assert np.array_equal(np.isnan(g["impurity"]), empty | ots.last_bad)
        # without the skip rule these would be finite numbers
        assert np.all(np.isfinite(ots.last_value[ots.last_bad & ~empty]))
        _assert_same_stats(g, o, (depth, steep))
    ts.close()


def _content_table():
    """every node content of 0..3 distinct samples of a pool of 24, sorted: index 0 is the empty node"""
    from itertools import combinations
    out = [()]
    for k in (1, 2, 3):
        out += list(combinations(range(24), k))
    return out


@pytest.fixture(scope="module")
def wide_pool():
    """24 samples, 16 candidates and the oracle's statistics of every (node content, candidate)"""
    patches, is_obj, offs, rots = (a[:24] for a in _mixed(80, 80, seed=41, n_frames=1, n_noise=6, n_sat=1, n_zero=1))
    ots = oracle.OracleTrainSet(patches, is_obj, offs, rots)
    rng = np.random.default_rng(41)
    pool_r, _ = train.HoughLearning(10, 80, 80, 15, 1, 1000, 0.3, 16, 20, 5.0).param_set(rng, 16)
    pool_t = rng.uniform(-40, 40, 16)
    contents = _content_table()
    c_idx, c_off = _flat([np.array(c, np.int64) for c in contents])
    table = ots.score_level(c_idx, c_off, np.broadcast_to(pool_r, (len(contents), 16, 8)),
                            np.broadcast_to(pool_t, (len(contents), 16)), 4, 5.0)
    return (patches, is_obj, offs, rots), pool_r, pool_t, contents, table


@pytest.mark.parametrize("n_nodes", [65535, 65536, 70001])
def test_wide_levels_match_the_oracle(ctx, wide_pool, n_nodes):
    """levels of more nodes than one launch holds in blockIdx.y, nodes of 0..3 samples with 3 candidates each"""
    (patches, is_obj, offs, rots), pool_r, pool_t, contents, table = wide_pool
    ts = train.TrainSet(patches, is_obj, offs, rots, 24, 24, ctx=ctx)
    rng = np.random.default_rng(n_nodes)
    cid = rng.integers(1, len(contents), n_nodes)
    cid[[0, 1, n_nodes // 2]] = 0                       # empty nodes at the front and in the middle
    cid[-5:] = 0                                        # and several in a row at the end
    cand = rng.integers(0, 16, (n_nodes, 3))
    idx, off = _flat([np.array(contents[c], np.int64) for c in cid])
    g = ts.score_level(idx, off, pool_r[cand], pool_t[cand], 4, 5.0)
    assert g.shape == (n_nodes, 3)
    _assert_same_stats(g, table[cid[:, None], cand], n_nodes)
    # the split of one chosen candidate per node, across the empty ones
    chosen = cand[:, 1]
    bits_of = np.stack([oracle.train_binarize(patches, np.arange(24), pool_r[j], pool_t[j]) for j in range(16)], 1)  # [sample, cand]
    node_of_slot = np.repeat(np.arange(n_nodes), np.diff(off.astype(np.int64)))
    want = bits_of[idx, chosen[node_of_slot]]
    assert np.array_equal(ts.split_level(idx, off, pool_r[chosen], pool_t[chosen]), want)
    # a decreasing node_off is an argument error in both calls
    off_bad = off.copy()
    k = int(np.flatnonzero(np.diff(off.astype(np.int64)) > 0)[3])
    off_bad[k + 1] = off[k] - 1
    with pytest.raises(capi.DhError) as e:
        ts.split_level(idx, off_bad, pool_r[chosen], pool_t[chosen])
    assert e.value.code == capi.DH_E_ARG and "dh_train_split_level" in str(e.value)
    with pytest.raises(capi.DhError) as e:
        ts.score_level(idx, off_bad, pool_r[cand], pool_t[cand], 4, 5.0)
    assert e.value.code == capi.DH_E_ARG
    ts.close()


def test_training_tables_in_two_chunks(ctx):
    """dh_trainset_create builds its tables in chunks of 256 MiB of patches: 20 971 samples of 80x80"""
    chunk = (256 << 20) // (80 * 80 * 2)
    assert chunk == 20971
    rng = np.random.default_rng(77)
    P, F, O, R = _windows(4, 77, 80, 80)
    n = chunk + 600
    patches = rng.integers(0, 65536, (n, 80, 80), dtype=np.uint16)
    at = rng.choice(n, len(P), replace=False)
    patches[at] = P
    patches[chunk - 3:chunk + 3] = P[:6]                 # windows on both sides of the chunk boundary
    is_obj = (rng.random(n) < 0.5).astype(np.uint8)
    offs = rng.normal(0, 60, (n, 3)).astype(np.float32)
    rots = rng.normal(0, 15, (n, 3))
    ts = train.TrainSet(patches, is_obj, offs, rots, 24, 24, ctx=ctx)
    ots = oracle.OracleTrainSet(patches, is_obj, offs, rots)
    nodes = [np.arange(chunk - 40, chunk + 40), np.arange(0, 60), np.arange(n - 60, n),
             rng.permutation(np.concatenate([np.arange(0, 20), np.arange(n - 20, n), np.arange(chunk - 10, chunk + 10)])),
             np.sort(at)]
    idx, off = _flat(nodes)
    rects, thr = _candidates(patches, nodes, 80, 80, 24, 24, 24, seed=9)
    for depth, steep in ((0, 5.0), (15, 2.5)):
        _assert_same_stats(ts.score_level(idx, off, rects, thr, depth, steep), ots.score_level(idx, off, rects, thr, depth, steep))
    for j in range(0, 24, 5):
        assert np.array_equal(ts.split_level(idx, off, rects[:, j], thr[:, j]), ots.split_level(idx, off, rects[:, j], thr[:, j]))
    ts.close()


def _canonical(arr, t):
    """tree t as nested tuples from the root, independent of node / leaf numbering"""
    n0, l0 = int(arr["tree_node_off"][t]), int(arr["tree_leaf_off"][t])

    def leaf(i):
        v0, v1 = int(arr["vote_off"][l0 + i]), int(arr["vote_off"][l0 + i + 1])
        return ("leaf", float(arr["prob"][l0 + i]), arr["offsets"][v0:v1].astype(np.float32).tobytes(),
                arr["rotations"][v0:v1].astype(np.float64).tobytes())

    def node(i):
        c = arr["child"][n0 + i]
        kids = tuple(node(int(k)) if k >= 0 else leaf(int(~k)) for k in c)
        return ("node", tuple(int(x) for x in arr["rects"][n0 + i]), float(arr["threshold"][n0 + i]), kids)
    if int(arr["tree_node_off"][t + 1]) == n0:
        return leaf(0)
    return node(0)


class _SkipCounter(oracle.OracleTrainSet):
    """counts the nodes whose choice the skip rule changes: with the unreachable!() candidates
    admitted, another candidate would have won"""
    decided = 0

    def score_level(self, *a):
        st = super().score_level(*a)
        for k in range(len(st)):
            imp = st[k]["impurity"]
            raw = np.where(self.last_bad[k] & ~(st[k]["n"] == 0).any(-1), self.last_value[k], imp)
            ok, ok_raw = ~np.isnan(imp), ~np.isnan(raw)
            if ok.any() and ok_raw.any():
                a_ = int(np.flatnonzero(ok)[np.argmin(imp[ok])])
                b_ = int(np.flatnonzero(ok_raw)[np.argmin(raw[ok_raw])])
                self.decided += int(a_ != b_)
        return st


def _check_forest(ctx, hl, native_hp, ots, seed, frames):
    arr_o = hl.train_forest(ots, train.CounterRng(seed))
    arr_g = oracle.forest_arrays_from_doc(json.loads(native_hp.to_json()))
    assert arr_g["n_trees"] == hl.n_trees and int(arr_o["tree_node_off"][-1]) > 3 * hl.n_trees
    for t in range(hl.n_trees):
        assert _canonical(arr_g, t) == _canonical(arr_o, t), "tree %d differs from the one grown on the oracle" % t
    js = native_hp.to_json()
    out = native_hp.predict_batch(frames[:1], K, ctx=ctx)
    tr = oracle.OracleForest.from_json(js).predict(frames[0], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
    assert np.array_equal(out["mid_point"][0], tr.mid_point) and np.array_equal(out["rotation"][0], tr.rotation)


FORESTS = [(80, 80, 0.3), (80, 80, 0.1), (80, 80, 0.05), (64, 48, 0.5), (81, 61, 0.3)]


@pytest.mark.parametrize("sw,sh,scale", FORESTS, ids=["%dx%d-%g" % f for f in FORESTS])
def test_forest_matches_the_oracle_grown_forest(ctx, sw, sh, scale):
    hl = train.HoughLearning(10, sw, sh, 6, 2, 260, scale, 40, 10, 5.0)
    frames = synth.make_frames(1, seed=500 + sw)
    if (sw, sh) in ((80, 80), (81, 61)) and scale == 0.3:
        # HoughLearning::learn from frames: dh_train_learn on the samples the Python extraction produced
        n_fr = 9
        f, c, r, m = synth.make_frames(n_fr, seed=sw + 7, with_truth=True)
        data = [dict(depth=f[i], mask=m[i], intrinsic=K, pos3d=c[i], rot=r[i]) for i in range(n_fr)]
        hl.learn(8.0, data, seed=13, ctx=ctx, native=True)
        ots = oracle.OracleTrainSet(*hl.last_samples)
        _check_forest(ctx, hl, hl.learn_native(8.0, data, seed=13, ctx=ctx), ots, 14, frames)
        patches, is_obj, offs, rots = hl.last_samples
    else:
        patches, is_obj, offs, rots = _windows(20, seed=sw + int(scale * 100), sw=sw, sh=sh)
    _check_forest(ctx, hl, hl.train_native(8.0, patches, is_obj, offs, rots, seed=3, ctx=ctx),
                  oracle.OracleTrainSet(patches, is_obj, offs, rots), 3, frames)


def test_forest_with_skipped_candidates_matches_the_oracle(ctx):
    patches, is_obj, offs, rots = _large_offsets(29, n_frames=20)
    hl = train.HoughLearning(10, 80, 80, 7, 3, 280, 0.3, 48, 4, 5.0)
    ots = _SkipCounter(patches, is_obj, offs, rots)
    _check_forest(ctx, hl, hl.train_native(8.0, patches, is_obj, offs, rots, seed=8, ctx=ctx), ots, 8,
                  synth.make_frames(1, seed=600))
    assert ots.decided > 0, "the skip rule decided no node"


def test_default_root_matches_the_oracle(ctx):
    """the reference's default root: 5200 samples, 2000 candidates of 24x24 rectangles in 80x80"""
    P, F, O, R = _windows(40, 61, 80, 80, per_image=40)
    rng = np.random.default_rng(61)
    n = 5200
    reps = rng.integers(0, len(P), n - len(P))
    noise = rng.integers(0, 64, (len(reps), 80, 80)).astype(np.uint16)   # distinct copies of the windows
    patches = np.concatenate([P, np.minimum(P[reps].astype(np.int64) + noise, 65535).astype(np.uint16)])
    is_obj = np.concatenate([F, F[reps]])
    offs = np.concatenate([O, O[reps] + rng.normal(0, 5, (len(reps), 3)).astype(np.float32)])
    rots = np.concatenate([R, R[reps]])
    ts = train.TrainSet(patches, is_obj, offs, rots, 24, 24, ctx=ctx)
    ots = oracle.OracleTrainSet(patches, is_obj, offs, rots)
    hl = train.HoughLearning(10, 80, 80, 15, 1, 5200, 0.3, 2000, 20, 5.0)
    rects, thr = hl.param_set(train.CounterRng(5), 2000)
    idx, off = _flat([rng.permutation(n)])
    g = ts.score_level(idx, off, rects[None], thr[None], 0, 5.0)
    o = ots.score_level(idx, off, rects[None], thr[None], 0, 5.0)
    _assert_same_stats(g, o)
    imp = g[0]["impurity"]
    ok = ~np.isnan(imp)
    assert ok.sum() > 500
    # the candidate dh_train_forest takes: the smallest impurity, the first of equals
    best = int(np.flatnonzero(ok)[np.argmin(imp[ok])])
    oi = o[0]["impurity"]
    assert best == int(np.flatnonzero(~np.isnan(oi))[np.argmin(oi[~np.isnan(oi)])])
    ts.close()
