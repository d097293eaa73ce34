"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.

Bars (BASELINE.json north_star): leaf index per patch x tree bit-exact; votes exact (integer bins
and u32 sums — tighter than the 1e-5 relative the north star allows); seeds identical; final head
centre / rotation identical (the bar is 1 mm / 0.1 degree, i.e. the same 3-degree bin).
"""
import os

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth
from test_prob_codes_cpu import codes_of, thresholds

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def context_with(**env):
    """a Context created with the given DH_* switches set, or unset where the value is None (the
    constructor reads them; the process environment is restored afterwards)"""
    old = {k: os.environ.get(k) for k in env}
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        return Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


# Passes of DH_GATE_SPLIT_MIN frames or more gate their patches in patch_gate_kernel (probability codes
# in the leaf words decide most patches, the gated-patch lists feed gate_coarse_kernel<true, .>); smaller
# passes fold every patch's probabilities in phase A of gate_coarse_kernel<false, .>, one launch less.
@pytest.fixture(scope="module")
def list_ctx():
    c = context_with(DH_GATE_SPLIT_MIN=1)
    yield c
    c.close()


@pytest.fixture(scope="module")
def fold_ctx():
    c = context_with(DH_GATE_SPLIT_MIN=1 << 30)
    yield c
    c.close()


def _filter_acc(keys, vals, origin, dim):
    """non-zero cells inside the cube [origin, origin + dim)^3"""
    if len(vals) == 0 or dim == 0:
        return keys.reshape(-1, 3)[:0], vals[:0]
    rel = keys.astype(np.int64) - np.asarray(origin, np.int64)
    m = (vals > 0) & np.all((rel >= 0) & (rel < dim), axis=1)
    return keys[m], vals[m]


def _compare_frame(ctx, hp, of, depth, midp_guess=None, rot_guess=None, check_patches=True, intrinsic=None, trace=None):
    """every stage of one frame against the oracle; intrinsic: a float32 3x3 matrix for both sides
    (None = the Kinect default); trace: the oracle's trace of this frame with these arguments
    (keep=True), when the caller already has it"""
    k = synth.KINECT_K if intrinsic is None else np.asarray(intrinsic, np.float32)
    ctx.enable_debug(True)
    res = hp.predict_parameter_parallel(depth, K if intrinsic is None else IntrinsicMatrix(k), midp_guess, rot_guess, ctx=ctx)
    tr = of.predict(depth, k, midp_guess, rot_guess, mode=oracle.MODE_SAT, keep=True) if trace is None else trace
    npx, npy, T = ctx.debug_dims()
    assert (npx, npy, T) == (tr.npx, tr.npy, of.n_trees)
    # --- leaf index per patch x tree: bit-exact
    leaf = ctx.debug_leaf_indices()
    assert np.array_equal(leaf, tr.leaf), "leaf ids differ at %d of %d" % (np.sum(leaf != tr.leaf), leaf.size)
    if check_patches:
        p3, gate = ctx.debug_patches()
        assert np.array_equal(gate, tr.gate)
        g = gate.astype(bool)
        assert np.array_equal(p3[g].view(np.uint32), tr.p3[g].view(np.uint32)), "p3 not bit-exact"
    # --- coarse grids + seeds
    gp, gr, sm, sr = ctx.debug_seeds()
    assert np.array_equal(gp, tr.guess_pos)
    assert np.array_equal(gr, tr.guess_rot)
    assert np.array_equal(sm, tr.seed_mid)
    assert np.array_equal(sr, tr.seed_rot)
    # --- accumulators: every cell of the dense cube around the final position must equal the
    #     reference's SparseArray3D (and the cube must contain the final 20^3 window)
    final = (tr.mid_point.astype(np.int64), np.round(tr.rotation / 3.14159 * 60 + 60).astype(np.int64))
    for which, (ok, ov) in enumerate(((tr.mid_keys, tr.mid_vals), (tr.rot_keys, tr.rot_vals))):
        gk, gv, org, dim = ctx.debug_votes(which)
        if of.meanshift_iterations == 0:
            assert dim == 0
            continue
        assert dim >= 20 + 2 * 6  # the 20-cell window of the seed and a margin
        ek, ev = _filter_acc(ok, ov, org, dim)
        assert np.array_equal(gk, ek), "accumulator %d keys differ (%d vs %d cells)" % (which, len(gk), len(ek))
        assert np.array_equal(gv, ev), "accumulator %d sums differ" % which
    # --- mean-shift trajectories: the GPU stops as soon as a position repeats (fixed point or
    #     cycle) and reads the final position off the history; the reference keeps iterating.
    for which, (otrace, seed) in enumerate(((tr.ms_mid, tr.seed_mid), (tr.ms_rot, tr.seed_rot))):
        gtrace = ctx.debug_meanshift(which)
        n = len(gtrace)
        assert n <= len(otrace)
        assert np.array_equal(gtrace, otrace[:n])
        if n and n < len(otrace) and not (tr.ms_mid_zero, tr.ms_rot_zero)[which]:
            seq = [tuple(seed)] + [tuple(p) for p in gtrace]
            j = seq.index(seq[-1])
            assert j < len(seq) - 1, "early exit without a repeated position"
            period = (len(seq) - 1) - j
            for m in range(n + 1, len(otrace) + 1):
                assert tuple(otrace[m - 1]) == seq[j + (m - j) % period], "periodic extension mismatch"
    f0, f1 = ctx.debug_meanshift_flags()
    assert bool(f0 & 1) == tr.ms_mid_zero and bool(f1 & 1) == tr.ms_rot_zero
    # --- result
    assert np.array_equal(res.mid_point, tr.mid_point)
    assert np.array_equal(res.rotation.view(np.uint64), tr.rotation.view(np.uint64))
    assert res.bounding_box == (0, 0, 0, 0)
    ctx.enable_debug(False)
    return res, tr


def test_small_forest_every_stage(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    for d in frames:
        _compare_frame(ctx, hp, of, d)


@pytest.mark.parametrize("stride,depth,trees", [(5, 10, 10), (7, 8, 5), (16, 12, 3)])
def test_mid_forest(ctx, stride, depth, trees):
    arr = synth.make_forest(seed=21 + stride, n_trees=trees, max_depth=depth, shuffle_nodes=True)
    js = synth.forest_to_json(arr, stepwidth=stride)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    for d in synth.make_frames(2, seed=100 + stride):
        _compare_frame(ctx, hp, of, d)


def test_sparse_trees_and_ragged_rects(ctx):
    arr = synth.make_forest(seed=5, n_trees=6, max_depth=12, stop_prob=0.25, ragged_rects=True, shuffle_nodes=True)
    js = synth.forest_to_json(arr, stepwidth=6)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    for d in synth.make_frames(2, seed=77):
        _compare_frame(ctx, hp, of, d)


def test_exact_ties_in_the_node_test(ctx):
    """Thresholds exactly on (and one ulp around) values avg1 - avg2 can take, identical
    rectangles, flat and staircase frames: the filtered integer predicate must fall back to the
    IEEE-division path and still agree with the reference arithmetic bit for bit."""
    arr = synth.make_forest(seed=17, n_trees=8, max_depth=10, tie_thresholds=True)
    js = synth.forest_to_json(arr, stepwidth=5)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    h, w = 480, 640
    flat = np.full((h, w), 1000, np.uint16)
    stairs = (1000 + (np.arange(w)[None, :] // 24) + 0 * np.arange(h)[:, None]).astype(np.uint16)
    ramp = (500 + np.arange(w)[None, :] + np.arange(h)[:, None]).astype(np.uint16)
    for d in (flat, stairs, ramp, synth.make_frames(1, seed=5)[0]):
        _compare_frame(ctx, hp, of, d)


def _threshold_menus(T):
    """leaf probability sub-menus ((value, weight) lists), one forest each, whose sums of T leaves
    concentrate on the code thresholds of T trees (test_prob_codes_cpu.thresholds)"""
    up, dn = 1.0, -1.0
    _, pass_codes, fail_codes = thresholds(T)
    nx = np.nextafter
    code178 = [0.7 - 1.0 / 300, nx(179 / 256, dn)]
    code179 = [179 / 256, nx(179 / 256, up), 0.7, nx(0.7, up), nx(0.7, dn), nx(180 / 256, dn)]
    code180 = [180 / 256, nx(180 / 256, up), 0.7 + 1.0 / 300]
    q_pass = min(max((pass_codes - 0.5 - 179 * T) / T, 0.0), 1.0)           # mean S = pass_codes - 1/2
    q_fail = min(max((fail_codes + 0.5 - T - 178 * T) / T, 0.0), 1.0)       # mean S + T = fail_codes + 1/2
    return [
        [(v, 1.0) for v in (0.7, nx(0.7, up), nx(0.7, dn))],                 # every code 179: ulp decisions
        [(v, (1 - q_pass) / 6) for v in code179] + [(v, q_pass / 3) for v in code180],
        [(v, (1 - q_fail) / 2) for v in code178] + [(v, q_fail / 6) for v in code179],
        [(179 / 256, 0.8), (180 / 256, 0.2)],                                # exact folds: S / 256 is the sum
    ]


def _threshold_forest(T, k, menu):
    """depth-6 trees whose leaves draw from `menu`, plus 0.0 and 1.0 (the ends of the code range) at 1 % each"""
    arr = synth.make_forest(seed=40 + 7 * T + k, n_trees=T, max_depth=6)
    rng = np.random.default_rng([T, k])
    vals = np.array([v for v, _ in menu] + [0.0, 1.0])
    w = np.array([p for _, p in menu])
    w = np.concatenate([0.98 * w / w.sum(), [0.01, 0.01]])
    prob = vals[rng.choice(len(vals), len(arr["prob"]), p=w)]
    nv = np.diff(arr["vote_off"])
    arr["prob"] = np.where((nv == 0) & (prob > 0), 0.0, prob).astype(np.float64)  # prob > 0 needs votes (prediction.rs:594)
    return arr


@pytest.mark.parametrize("n_trees", [1, 3, 5, 10, 20])
def test_patch_gate_at_the_threshold(list_ctx, fold_ctx, n_trees):
    """prob > 0.7 (prediction.rs:582-584) with leaf probabilities on, one ulp around and 1/300 around 0.7,
    on the code boundaries 179/256 and 180/256 and one ulp around them, and 0.0 and 1.0, drawn so that
    the sums of T leaves sit on the code thresholds.  Every frame runs on both gate paths: on list_ctx,
    patch_gate_kernel<false> decides a patch from its code sum S when S >= gate_pass_codes or
    S + T <= gate_fail_codes and folds the rest; on fold_ctx, phase A of gate_coarse_kernel<false, false>
    folds every patch.  Both must give the reference's gate flags, p3 bits and everything after them."""
    T = n_trees
    smin, pass_codes, fail_codes = thresholds(T)
    frames = synth.make_frames(2, seed=61)
    cls = dict.fromkeys(("S = pass", "S = pass - 1, folds below", "S + T = fail", "S + T = fail + 1",
                         "undecided, passes", "undecided, fails", "fold = gate_min_sum"), 0)
    for k, menu in enumerate(_threshold_menus(T)):
        arr = _threshold_forest(T, k, menu)
        js = synth.forest_to_json(arr, stepwidth=6)
        hp = HoughPrediction.from_json(js)
        of = oracle.OracleForest.from_json(js)
        for d in frames:
            tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=True)
            _compare_frame(fold_ctx, hp, of, d, trace=tr)
            launches = fold_ctx.counters()["launches"]
            _compare_frame(list_ctx, hp, of, d, trace=tr)
            # the list path ran: patch_gate_kernel is the one extra launch
            assert list_ctx.counters()["launches"] == launches + 1
            # what the code decision saw (the leaf words' codes have no accessor: restated from the oracle's leaf ids)
            leaf = tr.leaf[tr.leaf[:, 0] >= 0]
            prob = arr["prob"][leaf]
            S = codes_of(prob).sum(axis=1)
            fold = np.zeros(len(leaf))
            for t in range(T):
                fold = fold + prob[:, t]
            ref = fold / T > 0.7
            assert np.array_equal(ref, tr.gate[tr.leaf[:, 0] >= 0] == 1)
            undecided = (S < pass_codes) & (S + T > fail_codes)
            cls["S = pass"] += int(np.sum(S == pass_codes))
            cls["S = pass - 1, folds below"] += int(np.sum((S == pass_codes - 1) & undecided & ~ref))
            cls["S + T = fail"] += int(np.sum(S + T == fail_codes))
            cls["S + T = fail + 1"] += int(np.sum(S + T == fail_codes + 1))
            cls["undecided, passes"] += int(np.sum(undecided & ref))
            cls["undecided, fails"] += int(np.sum(undecided & ~ref))
            cls["fold = gate_min_sum"] += int(np.sum(fold == smin))
    if T == 20:
        cls.pop("fold = gate_min_sum")  # no sum of these values lands on 14.000000000000002
    assert all(cls.values()), cls


def test_caller_seeds(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    d = frames[0]
    auto, tr = _compare_frame(ctx, hp, of, d)
    # seed near the head: find a dense region from the oracle's own accumulator
    k = tr.mid_keys[np.argmax(tr.mid_vals)] if len(tr.mid_vals) else np.array([0, 0, 900])
    _compare_frame(ctx, hp, of, d, midp_guess=[float(k[0]) + 3.7, float(k[1]) - 2.2, float(k[2]) + 5.5],
                   rot_guess=[0.2, -0.35, 0.05])
    _compare_frame(ctx, hp, of, d, midp_guess=[12.5, -40.25, 950.0], rot_guess=None)
    _compare_frame(ctx, hp, of, d, midp_guess=None, rot_guess=[-1.0, 1.0, 0.5])


def test_sigma_iterations_stepwidth_setters(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    hp.update_sigma(3.0)
    of.update_sigma(3.0)
    hp.meanshift_iterations = 7
    of.meanshift_iterations = 7
    hp.stepwidth = 13
    of.stepwidth = 13
    _compare_frame(ctx, hp, of, frames[1])
    hp.update_sigma(-2.0)  # ignored (prediction.rs:321)
    assert hp.sigma() == 3.0
    hp.meanshift_iterations = 0
    of.meanshift_iterations = 0
    _compare_frame(ctx, hp, of, frames[1])


def test_edge_frames(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    h, w = 480, 640
    empty = np.zeros((h, w), np.uint16)                       # everything is background
    full = np.full((h, w), 65535, np.uint16)                  # maximum depth everywhere (u32 SAT wraps)
    one = empty.copy()
    one[240, 320] = 1234                                      # a single valid pixel
    rng = np.random.default_rng(5)
    noise = rng.integers(0, 65536, (h, w)).astype(np.uint16)  # random u16
    for d in (empty, full, one, noise):
        _compare_frame(ctx, hp, of, d)


def test_ragged_image_sizes(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    rng = np.random.default_rng(9)
    for (h, w) in ((80, 80), (81, 97), (123, 211), (480, 637)):
        d = np.where(rng.random((h, w)) < 0.6, rng.integers(400, 1500, (h, w)), 0).astype(np.uint16)
        _compare_frame(ctx, hp, of, d)


def test_leaf_static_gates(ctx):
    arr = synth.make_forest(seed=8, n_trees=3, max_depth=8)
    js = synth.forest_to_json(arr, stepwidth=10)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    v, r, o = hp.debug_leaf_static(ctx)
    n_rot = n_off = 0
    for leaf in range(hp.n_leaves):
        ev, tr_rot, tr_off = of.leaf_static(leaf)
        nv = int(arr["vote_off"][leaf + 1] - arr["vote_off"][leaf])
        if nv == 0:
            assert v[leaf] == 0 and r[leaf] == 0 and o[leaf] == 0
            continue
        assert v[leaf] == ev
        assert bool(r[leaf]) == bool(tr_rot <= 400.0)
        assert bool(o[leaf]) == bool(tr_off <= np.float32(5200.0))
        n_rot += int(r[leaf])
        n_off += int(o[leaf])
    assert 0 < n_rot < hp.n_leaves and 0 < n_off < hp.n_leaves  # both outcomes exercised


def test_batch_matches_single_and_oracle(ctx):
    arr = synth.make_forest(seed=2, n_trees=10, max_depth=9)
    js = synth.forest_to_json(arr, stepwidth=5)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    frames = synth.make_frames(11, seed=31)
    ctx.set_chunk_frames(4)  # 3 chunks, the last one ragged
    out = hp.predict_batch(frames, K, ctx=ctx)
    cnt = ctx.counters()
    assert cnt["frames"] == 11 and cnt["launches"] > 0
    ctx.set_chunk_frames(0)
    for i, d in enumerate(frames):
        tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(out["mid_point"][i], tr.mid_point)
        assert np.array_equal(out["rotation"][i], tr.rotation)
        single = hp.predict_parameter_parallel(d, K, ctx=ctx)
        assert np.array_equal(single.mid_point, out["mid_point"][i])
        assert np.array_equal(single.rotation, out["rotation"][i])


def test_device_resident_batch(ctx):
    import torch
    arr = synth.make_forest(seed=4, n_trees=5, max_depth=8)
    hp = HoughPrediction.from_arrays(arr, stepwidth=5)
    frames = synth.make_frames(6, seed=41)
    host = hp.predict_batch(frames, K, ctx=ctx)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    out = hp.predict_batch(None, K, ctx=ctx, device_ptr=dev.data_ptr(), n=6, w=640, h=480)
    assert np.array_equal(out["mid_point"], host["mid_point"])
    assert np.array_equal(out["rotation"], host["rotation"])
    # frames that start on an odd 2-byte boundary: no 16-byte pixel loads in the front-end kernels
    flat = torch.zeros(frames.size + 8, dtype=torch.int16, device="cuda")
    for off in (1, 3):
        flat[off:off + frames.size] = torch.from_numpy(frames.view(np.int16).reshape(-1)).cuda()
        torch.cuda.synchronize()
        out = hp.predict_batch(None, K, ctx=ctx, device_ptr=flat.data_ptr() + 2 * off, n=6, w=640, h=480)
        assert np.array_equal(out["mid_point"], host["mid_point"]) and np.array_equal(out["rotation"], host["rotation"])


def test_json_and_arrays_loaders_agree(ctx, small_case):
    arr, js, frames = small_case
    a = HoughPrediction.from_json(js)
    b = HoughPrediction.from_arrays(arr, stepwidth=10)
    ra = a.predict_batch(frames, K, ctx=ctx)
    rb = b.predict_batch(frames, K, ctx=ctx)
    assert np.array_equal(ra["mid_point"], rb["mid_point"]) and np.array_equal(ra["rotation"], rb["rotation"])


def test_predict_mask_and_hough_image(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    for d in frames[:2]:
        assert np.array_equal(hp.predict_mask(d, ctx=ctx), of.predict_mask(d))
        assert np.array_equal(hp.hough_image_raw(d, K, ctx=ctx), of.hough_image_raw(d, synth.KINECT_K))
    hp.stepwidth = 7
    of.stepwidth = 7
    assert np.array_equal(hp.predict_mask(frames[2], ctx=ctx), of.predict_mask(frames[2]))


def test_build_hough_image_and_from2dhough(ctx, small_case):
    """build_hough_image with its gaussian blur and predict_parameter_from2dhough
    (prediction.rs:343-367, 760-845) against the oracle, on the image shapes of the box-image test;
    the blur alone on images that exercise the clamped borders, saturation and the arg-max tie rule"""
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    for d in frames[:2]:
        got = hp.build_hough_image(d, K, ctx=ctx)
        assert np.array_equal(got, of.build_hough_image(d, synth.KINECT_K))
        res = hp.predict_parameter_from2dhough(d, K, ctx=ctx)
        mid, xy = of.predict_parameter_from2dhough(d, synth.KINECT_K)
        assert np.array_equal(res.mid_point.view(np.uint32), mid.view(np.uint32)) and np.all(res.rotation == 0.0)
        assert res.bounding_box == (0, 0, 0, 0)
    # an empty frame: the vote image is all zero, max_by_key returns the LAST pixel
    z = np.zeros((480, 640), np.uint16)
    res = hp.predict_parameter_from2dhough(z, K, ctx=ctx)
    mid, xy = of.predict_parameter_from2dhough(z, synth.KINECT_K)
    assert xy == (639, 479) and np.array_equal(res.mid_point, mid)
    # other sigmas (kernel radius ceil(2 sigma)) and other shapes
    for sigma, (sub, scale, stride, hw) in zip((1.5, 3.0, 0.4, 11.0, 8.0), [((80, 80), 0.3, 5, (480, 640)), ((80, 80), 0.3, 7, (203, 331)),
                                                                              ((64, 48), 0.5, 4, (150, 296)), ((40, 56), 0.13, 3, (97, 120)),
                                                                              ((96, 96), 0.9, 9, (200, 264))]):
        a2 = synth.make_forest(seed=17, n_trees=3, max_depth=6, sub_w=sub[0], sub_h=sub[1], rect_scale=scale)
        js2 = synth.forest_to_json(a2, stepwidth=stride)
        hp2 = HoughPrediction.from_json(js2)
        of2 = oracle.OracleForest.from_json(js2)
        hp2.update_sigma(sigma)
        of2.update_sigma(sigma)
        full = synth.make_frames(2, seed=5)
        y0, x0 = (480 - hw[0]) // 2, (640 - hw[1]) // 2
        for d in np.ascontiguousarray(full[:, y0:y0 + hw[0], x0:x0 + hw[1]]):
            got = hp2.build_hough_image(d, K, ctx=ctx)
            want = of2.build_hough_image(d, synth.KINECT_K)
            assert np.array_equal(got, want), (sigma, hw, int(np.sum(got != want)))
            res = hp2.predict_parameter_from2dhough(d, K, ctx=ctx)
            mid, _ = of2.predict_parameter_from2dhough(d, synth.KINECT_K)
            assert np.array_equal(res.mid_point.view(np.uint32), mid.view(np.uint32))


def test_shape_errors(ctx, small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    small = np.zeros((60, 60), np.uint16)
    with pytest.raises(capi.DhError) as e:
        hp.predict_parameter_parallel(small, K, ctx=ctx)
    assert e.value.code == capi.DH_E_SHAPE


def test_full_size_properties(ctx):
    """BASELINE configs[1] shape (10 trees, depth 15, stride 5) — size-independent properties:
    batch == per-frame, chunking-independent, permutation-equivariant, deterministic."""
    arr = synth.make_forest(seed=1, n_trees=10, max_depth=15)
    hp = HoughPrediction.from_arrays(arr, stepwidth=5)
    frames = synth.make_frames(24, seed=7)
    a = hp.predict_batch(frames, K, ctx=ctx)
    ctx.set_chunk_frames(5)
    b = hp.predict_batch(frames, K, ctx=ctx)
    ctx.set_chunk_frames(0)
    assert np.array_equal(a["mid_point"], b["mid_point"]) and np.array_equal(a["rotation"], b["rotation"])
    perm = np.random.default_rng(0).permutation(len(frames))
    c = hp.predict_batch(frames[perm], K, ctx=ctx)
    assert np.array_equal(c["mid_point"], a["mid_point"][perm]) and np.array_equal(c["rotation"], a["rotation"][perm])
    cnt = ctx.counters()
    assert cnt["evals"] == cnt["valid_patches"] * 10
    assert cnt["node_visits"] == cnt["evals"] * 15  # full depth-15 trees: every walk visits 15 nodes
    # spot-check three frames end to end against the oracle
    of = oracle.OracleForest(arr, 5, 80, 80, 8.0, 20)
    for i in (0, 11, 23):
        tr = of.predict(frames[i], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(a["mid_point"][i], tr.mid_point) and np.array_equal(a["rotation"][i], tr.rotation)


def test_against_committed_golden_vectors(ctx):
    """the CUDA path against tests/golden/oracle_small.npz directly (no oracle run in this test):
    leaf ids, gate, both seed grids, seeds and the final pose of every golden case"""
    import importlib.util
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(here, "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    g = np.load(os.path.join(here, "golden", "oracle_small.npz"))
    ctx.enable_debug(True)
    try:
        for name, fk, step, fseed, n in mg.CASES:
            arr = synth.make_forest(**fk)
            hp = HoughPrediction.from_arrays(arr, stepwidth=step)
            for i, d in enumerate(synth.make_frames(n, seed=fseed)):
                res = hp.predict_parameter_parallel(d, K, ctx=ctx)
                p = "%s/%d/" % (name, i)
                assert np.array_equal(ctx.debug_leaf_indices(), g[p + "leaf"]), (name, i)
                assert np.array_equal(ctx.debug_patches()[1], g[p + "gate"]), (name, i)
                gp, gr, sm, sr = ctx.debug_seeds()
                assert np.array_equal(gp, g[p + "guess_pos"]) and np.array_equal(gr, g[p + "guess_rot"]), (name, i)
                assert np.array_equal(sm, g[p + "seed_mid"]) and np.array_equal(sr, g[p + "seed_rot"]), (name, i)
                assert np.array_equal(res.mid_point, g[p + "mid_point"]), (name, i)
                assert np.array_equal(res.rotation.view(np.uint64), g[p + "rotation"].view(np.uint64)), (name, i)
    finally:
        ctx.enable_debug(False)
