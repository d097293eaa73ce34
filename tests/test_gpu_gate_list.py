"""GPU tests of the back end that passes of DH_GATE_SPLIT_MIN frames or more take (64 by default, which
is what batches, bench.py and long track passes run): patch_gate_kernel decides the patch gate from the
8-bit probability codes in the leaf words (the exact f64 fold for the undecided band) and writes every
frame's gated-patch list; gate_coarse_kernel<true, .> then builds the seed grids from slices of 512
list entries, a few CTAs per frame.  Both come in a one-K and a per-frame-K (kFrameK) instantiation.

Every call here is checked to have run that path: it makes one launch per pass more (patch_gate_kernel)
than the same call on a context whose DH_GATE_SPLIT_MIN exceeds the pass, and returns the same poses.
The contexts copy host frames without the run-length rewrite (DH_HOST_ENCODE=0), so that launch counts
do not depend on the machine's host threads.  Results must equal dh_predict frame by frame (passes of
one frame fold every patch inside gate_coarse_kernel) and the CPU oracle, bit for bit."""
import numpy as np
import pytest

import oracle
from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi, synth
from test_gpu_configs import _ramp_forest
from test_gpu_frame_args import _assert_same, _matrices, _seeds, _single, model  # noqa: F401 (module fixture)
from test_gpu_parity import _compare_frame, context_with, fold_ctx, list_ctx  # noqa: F401 (module fixtures)
from test_gpu_tracks import _first_seeds, _live_loop, _track_frames

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()
GATE_SLICE = 512  # entries of a frame's gated-patch list per seed-grid slice (kGateThreads)


@pytest.fixture(scope="module")
def ctx():
    """the library's default split (the test session may lower it through the environment)"""
    c = context_with(DH_GATE_SPLIT_MIN=None, DH_HOST_ENCODE=0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ref():
    """every pass folds the patch gate inside gate_coarse_kernel<false, .>"""
    c = context_with(DH_GATE_SPLIT_MIN=1 << 30, DH_HOST_ENCODE=0)
    yield c
    c.close()


def _on_both(ctx, ref, call, list_passes=1):
    """call(context) on ctx and on ref: the same results, and list_passes more launches on ctx"""
    got = call(ctx)
    launches = ctx.counters()["launches"]
    want = call(ref)
    assert launches == ref.counters()["launches"] + list_passes, (launches, ref.counters()["launches"], list_passes)
    _assert_same(got, want, "list path against the fold")
    return got


def _chunk(contexts, frames):
    for c in contexts:
        c.set_chunk_frames(frames)


def _on_device(frames):
    import torch
    dev = torch.from_numpy(np.ascontiguousarray(frames).view(np.int16)).cuda()
    torch.cuda.synchronize()
    return dev


def _assert_oracle(of, frame, Kf, mg, rg, got, what):
    tr = of.predict(frame, Kf, mg, rg, mode=oracle.MODE_SAT, keep=False)
    assert np.array_equal(got["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32)), what
    assert np.array_equal(got["rotation"].view(np.uint64), tr.rotation.view(np.uint64)), what


def test_per_frame_intrinsics_on_the_list_path(ctx, ref, model):
    """72 frames in one pass, 24 matrices (the general 3x3 among them) and mixed seeds: host, device and
    Biwi input run patch_gate_kernel<true> and gate_coarse_kernel<true, true>"""
    js, hp = model
    of = oracle.OracleForest.from_json(js)
    n = 72
    frames = synth.make_frames(n, seed=811)
    Ks = _matrices(24)[np.arange(n) % 24]
    mid, rot, hm, hr = _seeds(n, np.random.default_rng(12))
    want = _single(hp, ctx, frames, Ks, mid, rot, hm, hr)
    dev = _on_device(frames)
    blob, off = biwi.pack_files([biwi.encode_depth(f) for f in frames])
    _chunk((ctx, ref), n)
    try:
        for where, call in (
                ("host", lambda c: hp.predict_frames(frames, Ks, mid, rot, hm, hr, ctx=c)),
                ("device", lambda c: hp.predict_frames(None, Ks, mid, rot, hm, hr, ctx=c, device_ptr=dev.data_ptr(), n=n, w=640, h=480)),
                ("Biwi", lambda c: biwi.predict_files(hp, blob, off, 640, 480, Ks, ctx=c, midp_guess=mid, rot_guess=rot,
                                                      has_midp=hm, has_rot=hr))):
            _assert_same(_on_both(ctx, ref, call), want, where)
    finally:
        _chunk((ctx, ref), 0)
    one_k = hp.predict_frames(frames, K, mid, rot, hm, hr, ctx=ctx)
    assert (want["mid_point"] != one_k["mid_point"]).any(axis=1).sum() >= n // 2  # the matrices do move the poses
    for i in range(n):
        _assert_oracle(of, frames[i], Ks[i], mid[i] if hm[i] else None, rot[i] if hr[i] else None, want[i], i)


def _pass_sizes(lengths, F):
    """frames per pass of dh_predict_tracks (dh_ctx.cu plan_tracks): longest track first, F slots, an
    ended track's slot takes the next waiting track"""
    order = sorted((s for s in range(len(lengths)) if lengths[s]), key=lambda s: -lengths[s])
    slots = [[s, 0] for s in order[:F]]
    nxt, sizes = len(slots), []
    while any(s[0] >= 0 for s in slots):
        sizes.append(sum(s[0] >= 0 for s in slots))
        for s in slots:
            if s[0] < 0:
                continue
            s[1] += 1
            if s[1] == lengths[s[0]]:
                s[0], s[1] = (order[nxt] if nxt < len(order) else -1), 0
                nxt += 1
    return sizes


def test_tracks_whose_passes_straddle_the_split(ctx, ref, model):
    """80 tracks of 0 to 9 frames, each with its own K and starting seeds: the first passes hold 64 frames
    or more (list path, kFrameK), the later ones fewer (the fold); host, device and Biwi input, in passes
    of every live track and in passes of 64 slots"""
    js, hp = model
    rng = np.random.default_rng(77)
    lengths = [int(v) for v in rng.integers(0, 10, 80)]
    n_seq = len(lengths)
    frames = _track_frames(lengths, 1300)
    Ks = _matrices(n_seq)
    mid, rot, hm, hr = _first_seeds(n_seq, np.random.default_rng(13))
    want, seeds = _live_loop(hp, ctx, frames, lengths, Ks, mid, rot, hm, hr)
    dev = _on_device(frames)
    blob, off = biwi.pack_files([biwi.encode_depth(f) for f in frames])
    for chunk in (0, 64):
        sizes = _pass_sizes(lengths, chunk or n_seq)
        long_passes = sum(s >= 64 for s in sizes)
        assert 0 < long_passes < len(sizes), sizes
        _chunk((ctx, ref), chunk)
        try:
            for where, call in (
                    ("host", lambda c: hp.predict_tracks(frames, lengths, Ks, mid, rot, hm, hr, ctx=c)),
                    ("device", lambda c: hp.predict_tracks(None, lengths, Ks, mid, rot, hm, hr, ctx=c, device_ptr=dev.data_ptr(),
                                                           w=640, h=480)),
                    ("Biwi", lambda c: biwi.predict_track_files(hp, blob, off, lengths, 640, 480, Ks, mid, rot, hm, hr, ctx=c))):
                _assert_same(_on_both(ctx, ref, call, long_passes), want, "%s, chunk %d" % (where, chunk))
        finally:
            _chunk((ctx, ref), 0)
    # the oracle on frames of the first pass (every live track's first frame) and of short passes
    of = oracle.OracleForest.from_json(js)
    first = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    picks = [int(first[s]) for s in np.flatnonzero(np.array(lengths) > 0)[:4]]
    picks += [int(first[s]) + lengths[s] - 1 for s in np.flatnonzero(np.array(lengths) == 9)[:3]]
    track_of = np.repeat(np.arange(n_seq), lengths)
    for f in picks:
        mg, rg = seeds[f]
        _assert_oracle(of, frames[f], Ks[track_of[f]], mg, rg, want[f], f)


def _slice_forest():
    """box-sum trees on 12x12 windows whose every leaf has prob 1.0 and at least one vote: a patch gates
    if and only if its window has a non-zero pixel"""
    arr = synth.make_forest(seed=23, n_trees=3, max_depth=5, sub_w=12, sub_h=12, rect_scale=0.5, votes_lo=1, votes_hi=6)
    nv = np.diff(arr["vote_off"])
    take = [np.arange(arr["vote_off"][l], arr["vote_off"][l + 1]) if nv[l] else np.array([0]) for l in range(len(nv))]
    arr["offsets"] = np.ascontiguousarray(np.concatenate([arr["offsets"][t] for t in take]))
    arr["rotations"] = np.ascontiguousarray(np.concatenate([arr["rotations"][t] for t in take]))
    arr["vote_off"] = np.concatenate([[0], np.cumsum([len(t) for t in take])]).astype(np.int64)
    arr["prob"] = np.ones(len(nv))
    return arr


SLICE_COUNTS = [0, 1, GATE_SLICE - 1, GATE_SLICE, GATE_SLICE + 1, 2 * GATE_SLICE - 1, 2 * GATE_SLICE, 2 * GATE_SLICE + 1, 1536]


def _slice_frames(counts, seed):
    """588x396 frames (48 x 32 = 1536 windows of 12x12 at stride 12, which do not overlap), the centre
    pixel of `count` randomly chosen windows set"""
    rng = np.random.default_rng(seed)
    out = np.zeros((len(counts), 396, 588), np.uint16)
    for i, n in enumerate(counts):
        lit = rng.permutation(1536)[:n]
        out[i, 6 + 12 * (lit // 48), 6 + 12 * (lit % 48)] = rng.integers(600, 1400, n)
    return out


@pytest.mark.parametrize("gate_ctas", [None, 1, 2, 3], ids=["default", "1", "2", "3"])
def test_gated_list_slice_boundaries(ref, list_ctx, gate_ctas):
    """gated-patch lists of 0, 1, 511, 512, 513, 1023, 1024, 1025 and all 1536 entries in one pass of 72
    frames, walked by the launch heuristic's CTAs and by 1, 2 and 3 CTAs per frame"""
    arr = _slice_forest()
    js = synth.forest_to_json(arr, stepwidth=12)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    counts = SLICE_COUNTS * 8
    frames = _slice_frames(counts, 5 + (gate_ctas or 0))
    dev = _on_device(frames)
    c = context_with(DH_GATE_SPLIT_MIN=None, DH_HOST_ENCODE=0, DH_GATE_CTAS=gate_ctas or 0)
    try:
        out = _on_both(c, ref, lambda cc: hp.predict_batch(None, K, ctx=cc, device_ptr=dev.data_ptr(), n=len(counts), w=588, h=396))
        cnt = c.counters()
        assert cnt["patches"] == 1536 * len(counts) and cnt["gate_patches"] == sum(counts), cnt
        for i, d in enumerate(frames):
            _assert_oracle(of, d, synth.KINECT_K, None, None, out[i], i)
        if gate_ctas in (None, 1):
            # single frames on the list path: the whole frame list for one CTA, or one CTA per possible slice
            single = list_ctx if gate_ctas is None else context_with(DH_GATE_SPLIT_MIN=1, DH_GATE_CTAS=1)
            try:
                for i, n in enumerate(SLICE_COUNTS):
                    _, tr = _compare_frame(single, hp, of, frames[i])
                    assert int(tr.gate.sum()) == n and single.counters()["gate_patches"] == n
            finally:
                if single is not list_ctx:
                    single.close()
    finally:
        c.close()


def test_cube_rebuilds_inside_a_list_pass(ctx, ref):
    """72 frames with seeds along the vote ramp of test_gpu_configs._ramp_forest: mean-shift leaves the
    seed-centred accumulator cube and rebuilds it, in a pass whose persistent mean-shift CTAs take many
    frames each"""
    arr = _ramp_forest()
    js = synth.forest_to_json(arr, stepwidth=5, meanshift_iterations=30)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    n = 72
    frames = np.full((n, 90, 90), 1000, np.uint16)
    tr = of.predict(frames[0], synth.KINECT_K, mode=oracle.MODE_SAT, keep=True)
    x0 = int(tr.mid_keys[:, 0].min())
    y0, z0 = int(tr.mid_keys[0, 1]), int(tr.mid_keys[0, 2])
    mid = np.array([[x0 - 8 + 0.75 * i, y0 + (i % 5) - 2, z0 + (i % 3)] for i in range(n)], np.float32)
    rot = np.tile(np.array([0.15, -0.2, 0.05]), (n, 1))
    want = np.zeros(n, capi.RESULT_DTYPE)
    rebuilds = 0
    for i in range(n):
        r = hp.predict_parameter_parallel(frames[i], K, mid[i], rot[i], ctx=ctx)
        want[i]["mid_point"], want[i]["rotation"] = r.mid_point, r.rotation
        rebuilds += ctx.counters()["cube_rebuilds"]
    _chunk((ctx, ref), n)
    try:
        got = _on_both(ctx, ref, lambda c: hp.predict_frames(frames, K, mid, rot, ctx=c))
        batch_rebuilds = ctx.counters()["cube_rebuilds"]
    finally:
        _chunk((ctx, ref), 0)
    assert batch_rebuilds > 0 and batch_rebuilds == rebuilds, (batch_rebuilds, rebuilds)
    _assert_same(got, want, "ramp")
    for i in range(n):
        _assert_oracle(of, frames[i], synth.KINECT_K, mid[i], rot[i], got[i], i)


def _capped_codes(prob):
    """plan_nodes_kernel's code for any probability: floor(prob * 256) rounded toward zero into [0, 255]"""
    return np.clip(np.floor(prob * 256.0), 0, 255).astype(np.int64)


@pytest.mark.parametrize("n_trees", [2, 5])
def test_probabilities_outside_the_unit_interval(list_ctx, fold_ctx, n_trees):
    """leaves with prob 1.5 and -0.25 among ordinary ones: the loader takes them and the context turns the
    codes off, because a capped code sum would decide such patches against the fold (at T = 2, the leaves
    (1.5, 0.0) give S + T = 257 <= 358, a sure fail, but fold to 1.5 >= 1.4)"""
    from test_prob_codes_cpu import thresholds
    T = n_trees
    _, pass_codes, fail_codes = thresholds(T)
    arr = synth.make_forest(seed=90 + T, n_trees=T, max_depth=6)
    rng = np.random.default_rng(T)
    prob = np.array([1.5, -0.25, 0.0, 0.7, 0.9, 1.0])[rng.integers(0, 6, len(arr["prob"]))]
    nv = np.diff(arr["vote_off"])
    arr["prob"] = np.where((nv == 0) & (prob > 0), 0.0, prob).astype(np.float64)  # prob > 0 needs votes (prediction.rs:594)
    js = synth.forest_to_json(arr, stepwidth=6)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    wrong_fail = wrong_pass = 0
    for d in synth.make_frames(2, seed=95):
        _, tr = _compare_frame(fold_ctx, hp, of, d)
        launches = fold_ctx.counters()["launches"]
        _compare_frame(list_ctx, hp, of, d, trace=tr)
        assert list_ctx.counters()["launches"] == launches + 1  # patch_gate_kernel ran
        leaf = tr.leaf[tr.leaf[:, 0] >= 0]
        S = _capped_codes(arr["prob"][leaf]).sum(axis=1)
        ref_gate = tr.gate[tr.leaf[:, 0] >= 0] == 1
        wrong_fail += int(np.sum((S + T <= fail_codes) & ref_gate))
        wrong_pass += int(np.sum((S >= pass_codes) & ~ref_gate))
    # patches that codes would have decided wrongly (the leaf words' codes have no accessor: restated here)
    assert wrong_fail > 0 and (T == 2 or wrong_pass > 0), (wrong_fail, wrong_pass)


def test_default_split_point(ctx, ref):
    """device input at the library's default: 63 frames fold the gate inside gate_coarse_kernel, 64 run
    patch_gate_kernel, one launch more; both equal single-frame calls"""
    arr = synth.make_forest(seed=9, n_trees=5, max_depth=8)
    hp = HoughPrediction.from_arrays(arr, stepwidth=8)
    frames = synth.make_frames(64, seed=72)
    dev = _on_device(frames)
    want = _single(hp, ctx, frames, K.mat)
    launches = {}
    for n in (63, 64):
        got = _on_both(ctx, ref, lambda c: hp.predict_batch(None, K, ctx=c, device_ptr=dev.data_ptr(), n=n, w=640, h=480),
                       1 if n >= 64 else 0)
        launches[n] = ctx.counters()["launches"]
        _assert_same(got, want[:n], "%d frames" % n)
    assert launches[64] == launches[63] + 1, launches
