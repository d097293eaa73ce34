"""GPU parity for the remaining BASELINE.json configs and for every kernel variant.

configs[2] (Biwi-shaped sequence sharded by frame), configs[3] (large forest: 50 trees, depth 20,
dense stride-1 sampling) and configs[4] (vote-heavy: a million votes per frame) are run against
the oracle at sizes it finishes in seconds, and at (or near) full size through size-independent
properties: batch == single frame, chunking / sharding independence, permutation equivariance,
work-counter identities.  The variant test forces each path the library selects for some input
(LSU node fetch, general rectangles instead of box sums, box sums made in the tile, two-pass
summed-area table, box-image launch shapes, 512-thread traversal, the patch gate with and without
probability codes, lanes and chunks) and repeats the stage-by-stage comparison.
"""
import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, synth
from test_gpu_parity import _compare_frame

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def _small_frames(n, h, w, seed):
    """crops of the synthetic 640x480 frames around the person (keeps non-background content)"""
    full = synth.make_frames(n, seed=seed)
    y0, x0 = (480 - h) // 2, (640 - w) // 2
    return np.ascontiguousarray(full[:, y0:y0 + h, x0:x0 + w])


VARIANTS = [
    {"DH_TEX": "0"},                                # general rectangles need the LSU path when the texture is off
    {"DH_UNIFORM": "0"},                            # general 8-tap traversal on a uniform forest
    {"DH_UNIFORM": "0", "DH_TEX": "0"},
    {"DH_SAT_BANDS": "0", "DH_BOX_IMAGE": "0"},     # two-pass summed-area table
    {"DH_BOX_IMAGE": "0"},                          # uniform forest on the summed-area table (box sums made in the tile)
    {"DH_BOX_BANDS": "1"},                          # box image: one band per frame / five bands instead of the launch heuristic
    {"DH_BOX_BANDS": "5"},
    {"DH_BOX_WHOLE": "0"},                          # box image through warp-wide prefix sums (the path of widths not divisible by 8)
    {"DH_TRAV_THREADS": "512"},                     # 512-thread traversal tiles
    {"DH_LANES": "1"},
    {"DH_LANES": "4", "DH_CHUNK_FRAMES": "2"},
    {"DH_GATE_SPLIT_MIN": "64"},                    # the library's default: small passes gate inside the seed-grid kernel
    {"DH_PROB_CODES": "0"},                         # no probability codes in the node table: the patch gate runs as its own kernel
    {"DH_PROB_CODES": "0", "DH_GATE_CTAS": "2"},
    {"DH_PROB_CODES": "0", "DH_GATE_SPLIT_MIN": "64"},  # patch gate inside the seed-grid kernel, leaf words without codes
    {"DH_GATE_CTAS": "1"},                          # one seed-grid CTA per frame walks every slice of the gated-patch list
    {"DH_GATE_CTAS": "2", "DH_TRAV_THREADS": "512"},
    {"DH_BOX_IMAGE": "0", "DH_UNIFORM": "0", "DH_GATE_CTAS": "3"},
]


GATE_SLICE = 512  # entries of a frame's gated-patch list per seed-grid slice (kGateThreads)


def _noise_frame(seed):
    """random u16 depth with half of the pixels zeroed: a few thousand gated patches per VGA frame"""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 65536, (480, 640)).astype(np.uint16)
    d[rng.random((480, 640)) < 0.5] = 0
    return d


@pytest.mark.parametrize("env", VARIANTS, ids=lambda e: ",".join("%s=%s" % kv for kv in e.items()))
def test_kernel_variants(monkeypatch, env):
    gate_ctas = int(env.get("DH_GATE_CTAS", 0))
    if gate_ctas:
        # DH_GATE_CTAS shapes the seed-grid launch over the gated-patch lists, which passes of at least
        # DH_GATE_SPLIT_MIN frames use: every pass here does
        monkeypatch.setenv("DH_GATE_SPLIT_MIN", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = Context(0)  # the switches are read when a context is created, uploads a model or sizes its scratch
    try:
        for kw in (dict(seed=3, n_trees=4, max_depth=7), dict(seed=5, n_trees=3, max_depth=8, stop_prob=0.2, ragged_rects=True)):
            arr = synth.make_forest(**kw)
            js = synth.forest_to_json(arr, stepwidth=6)
            hp = HoughPrediction.from_json(js)
            of = oracle.OracleForest.from_json(js)
            frames = np.concatenate([synth.make_frames(5, seed=21), _noise_frame(21)[None]])
            _compare_frame(c, hp, of, frames[0])
            _compare_frame(c, hp, of, frames[5])
            if gate_ctas:
                # the noise frame's list has more slices than the frame has seed-grid CTAs: a CTA walks several
                assert c.counters()["gate_patches"] > gate_ctas * GATE_SLICE, c.counters()
            out = hp.predict_batch(frames, K, ctx=c)
            for i, d in enumerate(frames):
                tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
                assert np.array_equal(out["mid_point"][i], tr.mid_point) and np.array_equal(out["rotation"][i], tr.rotation)
            if gate_ctas:
                # the pass took the list path: one launch more (patch_gate_kernel) than with the gate inside the
                # seed-grid kernel
                launches = c.counters()["launches"]
                monkeypatch.setenv("DH_GATE_SPLIT_MIN", "64")
                ref = Context(0)
                try:
                    assert hp.predict_batch(frames, K, ctx=ref).tobytes() == out.tobytes()
                    assert launches == ref.counters()["launches"] + 1
                finally:
                    ref.close()
                    monkeypatch.setenv("DH_GATE_SPLIT_MIN", "1")
    finally:
        c.close()


def test_large_batch_crosses_both_gate_paths(monkeypatch):
    """library defaults: a batch of 80 frames gates its patches in patch_gate_kernel (probability codes in
    the leaf words, seed grids from slices of the gated-patch lists), single frames gate inside the
    seed-grid kernel; both must give the oracle's poses"""
    monkeypatch.delenv("DH_GATE_SPLIT_MIN", raising=False)
    c = Context(0)
    try:
        arr = synth.make_forest(seed=9, n_trees=5, max_depth=8)
        js = synth.forest_to_json(arr, stepwidth=8)
        hp = HoughPrediction.from_json(js)
        of = oracle.OracleForest.from_json(js)
        frames = synth.make_frames(80, seed=71)
        out = hp.predict_batch(frames, K, ctx=c)
        assert c.counters()["gate_patches"] > 80 * 100  # the gate passes a few hundred patches per frame
        for i in (0, 1, 17, 40, 79):
            tr = of.predict(frames[i], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
            assert np.array_equal(out["mid_point"][i], tr.mid_point) and np.array_equal(out["rotation"][i], tr.rotation), i
            res = hp.predict_parameter_parallel(frames[i], K, ctx=c)
            assert np.array_equal(res.mid_point, tr.mid_point) and np.array_equal(res.rotation, tr.rotation), i
        assert len({tuple(r) for r in out["rotation"].tolist()}) > 3
    finally:
        c.close()


@pytest.mark.parametrize("sub,scale,stride,hw", [
    ((80, 80), 0.3, 5, (480, 640)),     # the trained shape: 24x24 rectangles in 80x80 patches
    ((80, 80), 0.3, 7, (203, 331)),     # width not a multiple of 8: scalar pixel loads, ragged strips
    ((64, 48), 0.5, 4, (150, 296)),     # 32x24 rectangles, 2x2 taps cover a patch
    ((40, 56), 0.13, 3, (97, 120)),     # 5x7 rectangles: 8x8 = 64 taps per background test
    ((96, 96), 0.9, 9, (200, 264)),     # 86x86 rectangles: long ring, narrow box image
])
def test_box_image_shapes(ctx, sub, scale, stride, hw):
    """box-sum image front end (box_image_kernel + traversal modes 4/5) on rectangle / patch / image
    shapes that exercise strips, bands, the scalar load path and the tap cover of the background test"""
    arr = synth.make_forest(seed=17, n_trees=3, max_depth=6, sub_w=sub[0], sub_h=sub[1], rect_scale=scale)
    js = synth.forest_to_json(arr, stepwidth=stride)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    frames = _small_frames(3, hw[0], hw[1], seed=5) if hw != (480, 640) else synth.make_frames(2, seed=5)
    for d in frames:
        _compare_frame(ctx, hp, of, d)
    assert ctx.counters()["launches"] > 0
    # a frame of isolated pixels: most tiles are background, single set pixels decide patches
    rng = np.random.default_rng(3)
    d = np.zeros(hw, np.uint16)
    ys, xs = rng.integers(0, hw[0], 12), rng.integers(0, hw[1], 12)
    d[ys, xs] = rng.integers(1, 65535, 12)
    _compare_frame(ctx, hp, of, d)
    # saturated frame: every rectangle sum at its maximum
    _compare_frame(ctx, hp, of, np.full(hw, 65535, np.uint16))
    # many frames at once: bands and strips of a batch
    batch = np.stack([frames[i % len(frames)] for i in range(9)])
    out = hp.predict_batch(batch, K, ctx=ctx)
    for i, dd in enumerate(batch):
        tr = of.predict(dd, synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(out["mid_point"][i], tr.mid_point) and np.array_equal(out["rotation"][i], tr.rotation)


def test_config3_large_forest_dense_stride_vs_oracle(ctx):
    """configs[3] shape — many sparse deep trees, stride 1 — on a cropped frame the oracle can afford."""
    arr = synth.make_forest(seed=9, n_trees=50, max_depth=20, stop_prob=0.3)
    hp = HoughPrediction.from_arrays(arr, stepwidth=1)
    of = oracle.OracleForest(arr, 1, 80, 80, 8.0, 20)
    for d in _small_frames(2, 128, 160, seed=5):
        _compare_frame(ctx, hp, of, d)


def test_config3_large_forest_full_size_properties(ctx):
    """50 trees, depth 20, stride 1 on full 640x480 frames: 224 000 patches x 50 trees per frame."""
    arr = synth.make_forest(seed=9, n_trees=50, max_depth=20, stop_prob=0.3)
    hp = HoughPrediction.from_arrays(arr, stepwidth=1)
    frames = synth.make_frames(3, seed=8)
    a = hp.predict_batch(frames, K, ctx=ctx)
    cnt = ctx.counters()
    assert cnt["patches"] == 3 * 224000
    assert cnt["evals"] == cnt["valid_patches"] * 50
    assert cnt["evals"] <= cnt["node_visits"] <= cnt["evals"] * 20
    ctx.set_chunk_frames(2)
    b = hp.predict_batch(frames[::-1].copy(), K, ctx=ctx)
    ctx.set_chunk_frames(0)
    assert np.array_equal(a["mid_point"], b["mid_point"][::-1]) and np.array_equal(a["rotation"], b["rotation"][::-1])
    for i in range(3):
        s = hp.predict_parameter_parallel(frames[i], K, ctx=ctx)
        assert np.array_equal(s.mid_point, a["mid_point"][i]) and np.array_equal(s.rotation, a["rotation"][i])


def test_config4_vote_heavy_vs_oracle(ctx):
    """configs[4] shape — leaves with 32..128 votes — on a cropped frame, every stage compared."""
    arr = synth.make_forest(seed=13, n_trees=10, max_depth=8, votes_lo=32, votes_hi=128)
    hp = HoughPrediction.from_arrays(arr, stepwidth=2)
    of = oracle.OracleForest(arr, 2, 80, 80, 8.0, 20)
    for d in _small_frames(2, 160, 200, seed=6):
        _compare_frame(ctx, hp, of, d)


def test_config4_vote_heavy_full_size(ctx):
    """stride 1, 10 trees, 32..128 votes per leaf on full frames: over a million votes per frame
    through the coarse-grid, cube and mean-shift kernels; one frame checked against the oracle."""
    arr = synth.make_forest(seed=13, n_trees=10, max_depth=8, votes_lo=32, votes_hi=128)
    hp = HoughPrediction.from_arrays(arr, stepwidth=1)
    frames = synth.make_frames(3, seed=12)
    a = hp.predict_batch(frames, K, ctx=ctx)
    cnt = ctx.counters()
    assert (cnt["centre_votes"] + cnt["rot_votes"]) / 3 >= 1_000_000
    perm = np.array([2, 0, 1])
    b = hp.predict_batch(frames[perm], K, ctx=ctx)
    assert np.array_equal(b["mid_point"], a["mid_point"][perm]) and np.array_equal(b["rotation"], a["rotation"][perm])
    of = oracle.OracleForest(arr, 1, 80, 80, 8.0, 20)
    tr = of.predict(frames[1], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
    assert np.array_equal(a["mid_point"][1], tr.mid_point) and np.array_equal(a["rotation"][1], tr.rotation)


def test_config2_sequence_sharded_by_frame(ctx):
    """configs[2]: a Biwi-shaped sequence cut into contiguous shards (depthhead_b200.shard) gives
    byte-identical results to the unsharded run, shard by shard, for 1/2/4/8-way splits."""
    from depthhead_b200 import shard
    arr = synth.make_forest(seed=1, n_trees=10, max_depth=12)
    hp = HoughPrediction.from_arrays(arr, stepwidth=5)
    n = 37
    frames = synth.make_frames(n, seed=3, sequence=True)
    whole = hp.predict_batch(frames, K, ctx=ctx)
    for world in (2, 4, 8):
        parts = []
        for rank in range(world):
            lo, hi = shard.shard_range(n, rank, world)
            parts.append(hp.predict_batch(frames[lo:hi], K, ctx=ctx) if hi > lo else whole[:0])
        got = np.concatenate(parts)
        assert got.tobytes() == whole.tobytes()
    of = oracle.OracleForest(arr, 5, 80, 80, 8.0, 20)
    for i in (0, 18, 36):
        tr = of.predict(frames[i], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(whole["mid_point"][i], tr.mid_point) and np.array_equal(whole["rotation"][i], tr.rotation)


def _ramp_forest(n_trees=6):
    """Trees without nodes (a single leaf each) whose centre votes pile up exponentially along x:
    cell x of [0, 32) receives about 1.25^x votes per patch.  Mean-shift seeded at the thin end
    climbs the ramp by several cells per round, far more than the 10 cells of margin around the
    seed's window."""
    mult = np.maximum(1, np.round(1.25 ** np.arange(32))).astype(np.int64)
    xs = np.repeat(np.arange(32), mult)                      # one entry per vote
    per = int(np.ceil(len(xs) / n_trees))
    assert per <= 1000                                       # valtoadd = 1000 / n must stay >= 1
    offsets, rotations, vote_off = [], [], [0]
    for t in range(n_trees):
        part = xs[t * per:(t + 1) * per]
        if len(part) < 2:
            part = np.array([31, 31])
        o = np.zeros((len(part), 3), np.float32)
        o[:, 0] = -part.astype(np.float32) - 0.5             # np = p3 - o lands in cell trunc(p3.x) + x
        offsets.append(o)
        rotations.append(np.tile(np.array([[9.0, -12.0, 3.0]]), (len(part), 1)))
        vote_off.append(vote_off[-1] + len(part))
    z = np.zeros(n_trees + 1, np.int64)
    return dict(n_trees=n_trees, tree_node_off=z, tree_leaf_off=np.arange(n_trees + 1, dtype=np.int64),
                rects=np.zeros((0, 8), np.int64), threshold=np.zeros(0), child=np.zeros((0, 2), np.int32),
                prob=np.ones(n_trees), vote_off=np.asarray(vote_off, np.int64),
                offsets=np.ascontiguousarray(np.concatenate(offsets)),
                rotations=np.ascontiguousarray(np.concatenate(rotations)), sub_w=80, sub_h=80, max_depth=0)


def test_drifting_mean_shift_rebuilds_the_cube(ctx):
    """The window walks out of the seed-centred accumulator cube: the cube is rebuilt around the
    current position (more than once) and the trajectory still matches the oracle round by round."""
    arr = _ramp_forest()
    js = synth.forest_to_json(arr, stepwidth=5, meanshift_iterations=30)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    d = np.full((90, 90), 1000, np.uint16)                   # 2 x 2 patches, all valid, p3 ~ (-500, -357, 1000)
    tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=True)
    x0 = int(tr.mid_keys[:, 0].min())
    y0, z0 = int(tr.mid_keys[0, 1]), int(tr.mid_keys[0, 2])
    total = 0
    for start in (x0 - 6, x0 + 2):
        guess = [float(start), float(y0), float(z0)]
        res, t2 = _compare_frame(ctx, hp, of, d, midp_guess=guess, rot_guess=[0.15, -0.2, 0.05])
        assert abs(int(res.mid_point[0]) - start) > 14       # the position really left the first cube
        total += ctx.counters()["cube_rebuilds"]
    assert total >= 2


def test_two_devices_in_one_process():
    """one dh_ctx per GPU in ONE process (the forest object is shared): both devices give the
    oracle's answers; skipped on single-GPU boxes"""
    try:
        c1 = Context(1)
    except Exception:
        pytest.skip("needs a second GPU")
    c0 = Context(0)
    try:
        arr = synth.make_forest(seed=2, n_trees=5, max_depth=9)
        hp = HoughPrediction.from_arrays(arr, stepwidth=5)
        of = oracle.OracleForest(arr, 5, 80, 80, 8.0, 20)
        frames = synth.make_frames(6, seed=14)
        a = hp.predict_batch(frames, K, ctx=c1)       # the second device first: nothing was configured there yet
        b = hp.predict_batch(frames, K, ctx=c0)
        assert a.tobytes() == b.tobytes()
        for i in (0, 5):
            tr = of.predict(frames[i], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
            assert np.array_equal(a["mid_point"][i], tr.mid_point) and np.array_equal(a["rotation"][i], tr.rotation)
        r1 = hp.predict_parameter_parallel(frames[2], K, ctx=c1)
        assert np.array_equal(r1.mid_point, a["mid_point"][2])
    finally:
        c0.close()
        c1.close()


def test_single_frame_graph_replay_equals_eager_launches(monkeypatch):
    """dh_predict replays a captured CUDA graph from its third call with unchanged model / shape /
    intrinsics; seeds, frames, and every setter that is baked into the graph must still take effect"""
    arr = synth.make_forest(seed=6, n_trees=4, max_depth=8)
    frames = synth.make_frames(5, seed=33)
    K2 = IntrinsicMatrix([[575.816, 0.0, 320.0], [0.0, 575.816, 240.0], [0.0, 0.0, 1.0]])

    def run(flag):
        monkeypatch.setenv("DH_GRAPH", flag)
        c = Context(0)
        hp = HoughPrediction.from_arrays(arr, stepwidth=6)
        out = []
        try:
            res = None
            for rep in range(3):                       # eager, capture, replay ...
                for d in frames:
                    res = hp.predict_parameter_parallel(d, K, None if res is None or rep == 1 else res.mid_point,
                                                        None if res is None else res.rotation, ctx=c)
                    out.append((res.mid_point.copy(), res.rotation.copy()))
            for change in ("stepwidth", "iterations", "sigma", "K", "crop"):
                if change == "stepwidth":
                    hp.stepwidth = 9
                elif change == "iterations":
                    hp.meanshift_iterations = 3
                elif change == "sigma":
                    hp.update_sigma(5.0)
                kk = K2 if change in ("K", "crop") else K
                for rep in range(3):
                    for d in frames[:2]:
                        dd = d[:400, :600].copy() if change == "crop" else d
                        res = hp.predict_parameter_parallel(dd, kk, ctx=c)
                        out.append((res.mid_point.copy(), res.rotation.copy()))
        finally:
            c.close()
        return out
    a, b = run("1"), run("0")
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]), i
    of = oracle.OracleForest(arr, 6, 80, 80, 8.0, 20)
    tr = of.predict(frames[0], synth.KINECT_K, mode=oracle.MODE_SAT, keep=False)
    assert np.array_equal(a[0][0], tr.mid_point) and np.array_equal(a[0][1], tr.rotation)


def test_graph_replay_survives_a_growing_batch_between_single_calls(monkeypatch):
    """dh_predict's captured graph must not point at anything dh_predict_batch reallocates: single
    calls, a batch, more single calls (graph captured), a LARGER batch (the batch's pinned result
    buffer grows), single calls again — equal to the same sequence with eager launches."""
    arr = synth.make_forest(seed=8, n_trees=3, max_depth=7)
    frames = synth.make_frames(40, seed=51)

    def run(flag):
        monkeypatch.setenv("DH_GRAPH", flag)
        c = Context(0)
        c.set_chunk_frames(16)
        hp = HoughPrediction.from_arrays(arr, stepwidth=8)
        out = []
        try:
            out.append(hp.predict_batch(frames[:20], K, ctx=c).copy())
            for d in frames[:3]:
                r = hp.predict_parameter_parallel(d, K, ctx=c)
                out.append((r.mid_point.copy(), r.rotation.copy()))
            out.append(hp.predict_batch(frames[:40], K, ctx=c).copy())   # grows the batch result staging
            for d in frames[3:7]:
                r = hp.predict_parameter_parallel(d, K, ctx=c)
                out.append((r.mid_point.copy(), r.rotation.copy()))
            out.append(hp.predict_batch(frames[:5], K, ctx=c).copy())
            r = hp.predict_parameter_parallel(frames[9], K, ctx=c)
            out.append((r.mid_point.copy(), r.rotation.copy()))
        finally:
            c.close()
        return out
    a, b = run("1"), run("0")
    for i, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, tuple):
            assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]), i
        else:
            assert np.array_equal(x["mid_point"], y["mid_point"]) and np.array_equal(x["rotation"], y["rotation"]), i
    # single call 3 + k equals row 3 + k of the 40-frame batch
    for k in range(4):
        assert np.array_equal(a[5 + k][0], a[4]["mid_point"][3 + k]) and np.array_equal(a[5 + k][1], a[4]["rotation"][3 + k])


@pytest.mark.parametrize("threads", [None, "512"], ids=["default", "512"])
def test_default_walk_tree_shapes(monkeypatch, threads):
    """The default walk (box-sum tile, the first levels through the LSU path, the rest through the
    texture path) with the library's tiles and with 512-thread tiles: full trees of odd and even depth,
    sparse trees (leaves at every depth, children that are leaves), trees that are a single leaf,
    shuffled node order, exact ties (the fast pass hands them to the IEEE-division pass), and the work
    counter node_visits, which must count every node of a walk once, ties included."""
    if threads is None:
        monkeypatch.delenv("DH_TRAV_THREADS", raising=False)
    else:
        monkeypatch.setenv("DH_TRAV_THREADS", threads)
    c = Context(0)
    try:
        frames = synth.make_frames(3, seed=61)
        cases = [dict(seed=31, n_trees=3, max_depth=7), dict(seed=32, n_trees=3, max_depth=8),
                 dict(seed=33, n_trees=6, max_depth=11, stop_prob=0.3, shuffle_nodes=True),
                 dict(seed=34, n_trees=5, max_depth=1), dict(seed=35, n_trees=4, max_depth=2, stop_prob=0.5),
                 dict(seed=36, n_trees=8, max_depth=10, tie_thresholds=True)]
        for kw in cases:
            arr = synth.make_forest(**kw)
            js = synth.forest_to_json(arr, stepwidth=6)
            hp = HoughPrediction.from_json(js)
            of = oracle.OracleForest.from_json(js)
            for d in frames[:2]:
                _compare_frame(c, hp, of, d)
            if kw.get("tie_thresholds"):
                stairs = (1000 + (np.arange(640)[None, :] // 24) + 0 * np.arange(480)[:, None]).astype(np.uint16)
                _compare_frame(c, hp, of, stairs)
                _compare_frame(c, hp, of, np.full((480, 640), 1000, np.uint16))
            # node visits = sum over evaluations of the depth of the leaf reached
            out = hp.predict_batch(frames, K, ctx=c)
            cnt = c.counters()
            depth_of_leaf = _leaf_depths(arr)
            want = 0
            for d in frames:
                tr = of.predict(d, synth.KINECT_K, mode=oracle.MODE_SAT, keep=True)
                valid = tr.leaf[:, 0] >= 0
                want += int(depth_of_leaf[tr.leaf[valid]].sum())
            assert cnt["node_visits"] == want, kw
    finally:
        c.close()


def _leaf_depths(arr):
    """depth (number of node visits of a walk that ends there) of every global leaf id"""
    n_leaves = int(arr["tree_leaf_off"][-1])
    out = np.zeros(n_leaves, np.int64)
    for t in range(int(arr["n_trees"])):
        n0, l0 = int(arr["tree_node_off"][t]), int(arr["tree_leaf_off"][t])
        n_nodes = int(arr["tree_node_off"][t + 1]) - n0
        if n_nodes == 0:
            continue
        stack = [(0, 1)]
        while stack:
            i, d = stack.pop()
            for b in range(2):
                ch = int(arr["child"][n0 + i, b]) if arr["child"].ndim == 2 else int(arr["child"][2 * (n0 + i) + b])
                if ch >= 0:
                    stack.append((ch, d + 1))
                else:
                    out[l0 + (~ch)] = d
    return out


def test_seeded_sequences_equal_frame_by_frame_prediction(ctx):
    """dh_predict_sequences: frame t of every sequence in one pass, seeded on the device with the
    pose of frame t - 1 (examples/live_prediction.rs:75-88) == dh_predict frame by frame with those
    seeds == the oracle with those seeds; host and device input, groups smaller than the batch."""
    import torch
    arr = synth.make_forest(seed=12, n_trees=4, max_depth=8)
    js = synth.forest_to_json(arr, stepwidth=8)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    n_seq, T = 5, 6
    frames = np.stack([synth.make_frames(T, seed=400 + s, sequence=True, start_index=625 * s) for s in range(n_seq)])
    frames[3, 2] = 0            # an empty frame in the middle of a sequence: pose (0, 0, 0) -> z <= 500 -> no centre seed for the next frame
    got = hp.predict_sequences(frames, K, min_seed_z=500.0, ctx=ctx)
    assert got.shape == (n_seq, T)
    for s in range(n_seq):
        mid, rot = None, None
        for t in range(T):
            mg = mid if (mid is not None and mid[2] > np.float32(500.0)) else None
            res = hp.predict_parameter_parallel(frames[s, t], K, mg, rot, ctx=ctx)
            assert np.array_equal(got[s, t]["mid_point"], res.mid_point) and np.array_equal(got[s, t]["rotation"], res.rotation), (s, t)
            if s < 2:
                tr = of.predict(frames[s, t], synth.KINECT_K, mg, rot, mode=oracle.MODE_SAT, keep=False)
                assert np.array_equal(res.mid_point, tr.mid_point) and np.array_equal(res.rotation, tr.rotation)
            mid, rot = res.mid_point, res.rotation
    # device-resident input, and groups of 2 sequences per pass
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    c2 = Context(0)
    try:
        c2.set_chunk_frames(2)
        got2 = hp.predict_sequences(None, K, 500.0, ctx=c2, device_ptr=dev.data_ptr(), n_seq=n_seq, frames_per_seq=T, w=640, h=480)
    finally:
        c2.close()
    assert np.array_equal(got2["mid_point"], got["mid_point"]) and np.array_equal(got2["rotation"], got["rotation"])
    # min_seed_z = -inf: always seeded with the previous centre; differs from the 500 mm rule only after the empty frame
    got3 = hp.predict_sequences(frames, K, min_seed_z=float("-inf"), ctx=ctx)
    assert np.array_equal(got3[:3]["mid_point"], got[:3]["mid_point"])
    # one frame per sequence == the unseeded batch
    one = hp.predict_sequences(frames[:, :1], K, ctx=ctx)
    bat = hp.predict_batch(np.ascontiguousarray(frames[:, 0]), K, ctx=ctx)
    assert np.array_equal(one[:, 0]["mid_point"], bat["mid_point"]) and np.array_equal(one[:, 0]["rotation"], bat["rotation"])
