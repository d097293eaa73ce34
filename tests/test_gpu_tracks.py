"""GPU tests of dh_predict_tracks / dh_predict_tracks_biwi: tracks of any length, each with its own
intrinsics and starting seeds, every later frame seeded from the frame before it by the live rule of
examples/live_prediction.rs:75-88.  Results must equal, bit for bit on mid_point and rotation, a host
loop of predict_parameter_parallel that applies the rule, whatever the chunk size (which decides
only where a frame runs), for host, device-resident and Biwi input."""
import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()
LENGTHS = [7, 1, 0, 12, 3, 5]
MIN_Z = np.float32(500.0)


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def model(ctx):
    """the trained forest of test_gpu_frame_args.py (4 trees of depth 8 on synthetic heads, stride 10)"""
    from depthhead_b200 import train
    tf, tc, tr_, tm = synth.make_frames(40, seed=101, with_truth=True)
    data = [dict(depth=tf[i], mask=tm[i], intrinsic=K, pos3d=tc[i], rot=tr_[i]) for i in range(len(tf))]
    js = train.HoughLearning(10, 80, 80, 8, 4, 1200, 0.3, 150, 20, 5.0).learn_native(8.0, data, seed=7, ctx=ctx).to_json()
    return js, HoughPrediction.from_json(js)


def _matrices(n):
    """n intrinsics that differ, one of them a general 3x3 (non-zero off-diagonal and bottom-row terms)"""
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 480.0 + 7.5 * i
        Ks[i] = [[f, 0.0, 300.0 + 2.0 * i], [0.0, f * 1.01, 230.0 + 1.5 * i], [0.0, 0.0, 1.0]]
    Ks[n // 2] = [[561.5, 3.25, 318.0], [-2.5, 557.0, 243.5], [1.0e-4, -2.0e-4, 1.0]]
    return Ks


def _track_frames(lengths, seed):
    """smooth sequences, one per track, concatenated in track order; frame 1 of the longest track is empty
    (its z is 0, so the next frame gets no centre seed)"""
    parts = [synth.make_frames(n, seed=seed + s, sequence=True, start_index=700 * s) for s, n in enumerate(lengths) if n]
    frames = np.ascontiguousarray(np.concatenate(parts))
    off = np.concatenate([[0], np.cumsum(lengths)])
    longest = int(np.argmax(lengths))
    if lengths[longest] > 2:
        frames[off[longest] + 1] = 0
    return frames


def _first_seeds(n, rng):
    """seeds of the first frames: both, centre only, rotation only and none (over LENGTHS: every kind on a
    track that has frames)"""
    mid = rng.uniform(-200.0, 200.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    rot = rng.uniform(-1.0, 1.0, (n, 3))
    kind = np.array([3, 1, 2, 0, 2, 1])[np.arange(n) % 6]
    return mid, rot, (kind & 1) == 1, (kind & 2) == 2


def _live_loop(hp, ctx, frames, lengths, Ks, mid=None, rot=None, hm=None, hr=None):
    """predict_parameter_parallel frame by frame with the live rule: RESULT_DTYPE[total], and every
    frame's seeds (midp or None, rot or None)"""
    out = np.zeros(len(frames), capi.RESULT_DTYPE)
    seeds = []
    f = 0
    for s, n in enumerate(lengths):
        prev = None
        for t in range(n):
            if prev is None:
                mg = mid[s] if mid is not None and hm[s] else None
                rg = rot[s] if rot is not None and hr[s] else None
            else:
                mg = prev.mid_point if prev.mid_point[2] > MIN_Z else None
                rg = prev.rotation
            kk = IntrinsicMatrix(Ks[s] if Ks.ndim == 3 else Ks)
            prev = hp.predict_parameter_parallel(frames[f], kk, mg, rg, ctx=ctx)
            out[f]["mid_point"], out[f]["rotation"] = prev.mid_point, prev.rotation
            seeds.append((mg, rg))
            f += 1
    return out, seeds


def _assert_same(got, want, what):
    assert got.shape == want.shape, what
    for name, view in (("mid_point", np.uint32), ("rotation", np.uint64)):
        a, b = np.ascontiguousarray(got[name]).view(view), np.ascontiguousarray(want[name]).view(view)
        bad = np.argwhere((a != b).any(axis=1)).ravel()
        assert len(bad) == 0, "%s: %s differs at frames %s" % (what, name, bad[:8].tolist())
    assert np.all(got["bounding_box"] == 0) and np.all(got["_pad"] == 0), what


def _on_device(frames):
    import torch
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    return dev


@pytest.fixture(scope="module")
def ragged(ctx, model):
    _, hp = model
    n = len(LENGTHS)
    frames = _track_frames(LENGTHS, 900)
    Ks = _matrices(n)
    mid, rot, hm, hr = _first_seeds(n, np.random.default_rng(11))
    want, seeds = _live_loop(hp, ctx, frames, LENGTHS, Ks, mid, rot, hm, hr)
    return frames, Ks, (mid, rot, hm, hr), want, seeds


@pytest.mark.parametrize("chunk", [0, 1, 2, 4])
def test_ragged_tracks_equal_the_live_rule_loop(ctx, model, ragged, chunk):
    """six tracks (one of them empty), six matrices, mixed starting seeds; chunks of 1, 2 and 4 refill
    slots and leave one-frame passes; host, device-resident and Biwi input"""
    _, hp = model
    frames, Ks, seeds, want, _ = ragged
    total = len(frames)
    dev = _on_device(frames)
    files = [biwi.encode_depth(f) for f in frames]
    blob, off = biwi.pack_files(files)
    ctx.set_chunk_frames(chunk)
    try:
        _assert_same(hp.predict_tracks(frames, LENGTHS, Ks, *seeds, ctx=ctx), want, "host, chunk %d" % chunk)
        assert ctx.counters()["frames"] == total
        _assert_same(hp.predict_tracks(None, LENGTHS, Ks, *seeds, ctx=ctx, device_ptr=dev.data_ptr(), w=640, h=480), want,
                     "device, chunk %d" % chunk)
        assert ctx.counters()["frames"] == total
        _assert_same(biwi.predict_track_files(hp, blob, off, LENGTHS, 640, 480, Ks, *seeds, ctx=ctx), want, "Biwi, chunk %d" % chunk)
        assert ctx.counters()["frames"] == total
    finally:
        ctx.set_chunk_frames(0)


def test_seeds_and_matrices_matter(ctx, model, ragged):
    """the starting seeds and the matrices visibly change the poses (so the test above tests them)"""
    _, hp = model
    frames, Ks, seeds, want, _ = ragged
    plain = hp.predict_tracks(frames, LENGTHS, K, ctx=ctx)
    assert (plain["mid_point"] != want["mid_point"]).any(axis=1).sum() >= len(frames) // 3
    unseeded = hp.predict_tracks(frames, LENGTHS, Ks, ctx=ctx)
    first = np.concatenate([[0], np.cumsum(LENGTHS)[:-1]])[np.array(LENGTHS) > 0]
    changed = (unseeded["rotation"][first] != want["rotation"][first]).any(axis=1) | \
        (unseeded["mid_point"][first] != want["mid_point"][first]).any(axis=1)
    assert changed.sum() >= 2, changed


def test_three_frames_equal_the_oracle(ctx, model, ragged):
    """frames of the longest track, with the seeds the track gave them, against the CPU oracle"""
    js, _ = model
    of = oracle.OracleForest.from_json(js)
    frames, Ks, _, want, seeds = ragged
    s = int(np.argmax(LENGTHS))
    f0 = int(np.sum(LENGTHS[:s]))
    for t in (0, 3, LENGTHS[s] - 1):
        mg, rg = seeds[f0 + t]
        tr = of.predict(frames[f0 + t], Ks[s], mg, rg, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(want[f0 + t]["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32)), t
        assert np.array_equal(want[f0 + t]["rotation"].view(np.uint64), tr.rotation.view(np.uint64)), t


@pytest.mark.parametrize("chunk", [0, 3])
def test_equal_lengths_one_k_no_seeds_equal_predict_sequences(ctx, model, chunk):
    """4 tracks of 5 frames: exactly dh_predict_sequences, with the same counters (launches included);
    chunk 3 runs the tracks in two groups, as dh_predict_sequences does"""
    _, hp = model
    n_seq, T = 4, 5
    frames = np.stack([synth.make_frames(T, seed=500 + s, sequence=True, start_index=600 * s) for s in range(n_seq)])
    frames[2, 1] = 0
    flat = np.ascontiguousarray(frames.reshape(n_seq * T, 480, 640))
    dev = _on_device(flat)
    ctx.set_chunk_frames(chunk)
    try:
        for where in ("host", "device"):
            src = dict(device_ptr=dev.data_ptr(), w=640, h=480) if where == "device" else {}
            seq_src = dict(device_ptr=dev.data_ptr(), n_seq=n_seq, frames_per_seq=T, w=640, h=480) if where == "device" else {}
            want = hp.predict_sequences(None if src else frames, K, min_seed_z=500.0, ctx=ctx, **seq_src)
            cnt_seq = ctx.counters()
            got = hp.predict_tracks(None if src else flat, [T] * n_seq, K, min_seed_z=500.0, ctx=ctx, **src)
            cnt_tracks = ctx.counters()
            _assert_same(got, np.ascontiguousarray(want.reshape(-1)), where)
            assert cnt_tracks == cnt_seq, (where, cnt_seq, cnt_tracks)
            assert cnt_tracks["frames"] == n_seq * T
            # one matrix as an [n_seq,3,3] array is the same call
            _assert_same(hp.predict_tracks(None if src else flat, [T] * n_seq, np.tile(K.mat, (n_seq, 1, 1)), ctx=ctx, **src),
                         np.ascontiguousarray(want.reshape(-1)), where + ", K per track")
            assert ctx.counters()["launches"] == cnt_seq["launches"]
    finally:
        ctx.set_chunk_frames(0)


@pytest.mark.parametrize("chunk", [0, 1])
def test_damaged_biwi_file_names_the_lowest_frame(ctx, model, chunk):
    """a damaged file in a short track and one in the longest track (which runs first): DH_E_ARG names
    the lower global index, whichever ran first"""
    _, hp = model
    lengths = [3, 9, 2]
    frames = _track_frames(lengths, 950)
    files = [biwi.encode_depth(f) for f in frames]
    Ks = _matrices(3)
    ctx.set_chunk_frames(chunk)
    try:
        for short, longest, want in ((1, 3 + 6, 1), (12 + 1, 3 + 1, 4)):
            bad = list(files)
            bad[short] = bad[short][:len(bad[short]) // 2]
            bad[longest] = bad[longest][:len(bad[longest]) // 3]
            blob, off = biwi.pack_files(bad)
            with pytest.raises(capi.DhError) as e:
                biwi.predict_track_files(hp, blob, off, lengths, 640, 480, Ks, ctx=ctx)
            assert e.value.code == capi.DH_E_ARG and "Biwi frame %d " % want in str(e.value), str(e.value)
        # the context is usable afterwards
        blob, off = biwi.pack_files(files)
        _assert_same(biwi.predict_track_files(hp, blob, off, lengths, 640, 480, Ks, ctx=ctx),
                     hp.predict_tracks(frames, lengths, Ks, ctx=ctx), "after the errors")
    finally:
        ctx.set_chunk_frames(0)


def test_launches_per_pass_depend_on_neither_chunk_nor_matrices(ctx, model):
    """device-resident frames: launches / passes is the same at chunk 0 (4 passes) and chunk 1 (12
    passes), with one matrix and with three; the frames counter is the total"""
    _, hp = model
    lengths = [4, 4, 4]
    frames = _track_frames(lengths, 970)
    dev = _on_device(frames)
    mid, rot, hm, hr = _first_seeds(3, np.random.default_rng(2))
    hm[:] = True  # starting seeds: the general pass loop even with one matrix
    per_pass = []
    for chunk, passes in ((0, 4), (1, 12)):
        ctx.set_chunk_frames(chunk)
        try:
            for Ks in (K, _matrices(3)):
                hp.predict_tracks(None, lengths, Ks, mid, rot, hm, hr, ctx=ctx, device_ptr=dev.data_ptr(), w=640, h=480)
                cnt = ctx.counters()
                assert cnt["frames"] == 12
                assert cnt["launches"] % passes == 0, (chunk, cnt["launches"])
                per_pass.append(cnt["launches"] // passes)
        finally:
            ctx.set_chunk_frames(0)
    assert per_pass[1:] == per_pass[:-1] and per_pass[0] > 0, per_pass


def test_empty_calls(ctx, model):
    _, hp = model
    assert len(hp.predict_tracks(np.zeros((0, 480, 640), np.uint16), [], np.zeros((0, 3, 3), np.float32), ctx=ctx)) == 0
    assert len(hp.predict_tracks(np.zeros((0, 480, 640), np.uint16), [0, 0], K, ctx=ctx)) == 0
    assert ctx.counters()["frames"] == 0
