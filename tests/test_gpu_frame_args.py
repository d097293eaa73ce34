"""GPU tests of dh_predict_frames / dh_predict_frames_biwi: a batch in which every frame has its own
intrinsics and seeds must equal, bit for bit on mid_point and rotation, dh_predict called frame by
frame with the same arguments — across the host, run-length host and device-resident input paths,
several chunks over both lanes, distinct and degenerate matrices, and every kind of seed."""
import os

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def model(ctx):
    """a forest trained on synthetic heads (as smoke() does: 4 trees of depth 8, stride 10), so that
    poses follow the head and the intrinsics and seeds visibly change them"""
    from depthhead_b200 import train
    tf, tc, tr_, tm = synth.make_frames(40, seed=101, with_truth=True)
    data = [dict(depth=tf[i], mask=tm[i], intrinsic=K, pos3d=tc[i], rot=tr_[i]) for i in range(len(tf))]
    js = train.HoughLearning(10, 80, 80, 8, 4, 1200, 0.3, 150, 20, 5.0).learn_native(8.0, data, seed=7, ctx=ctx).to_json()
    return js, HoughPrediction.from_json(js)


def _matrices(n):
    """n intrinsics: focal lengths and principal points that vary, and one general 3x3 with non-zero
    off-diagonal terms (including the bottom row)"""
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 480.0 + 7.5 * i
        Ks[i] = [[f, 0.0, 300.0 + 2.0 * i], [0.0, f * 1.01, 230.0 + 1.5 * i], [0.0, 0.0, 1.0]]
    Ks[n // 2] = [[561.5, 3.25, 318.0], [-2.5, 557.0, 243.5], [1.0e-4, -2.0e-4, 1.0]]
    return Ks


def _seeds(n, rng):
    """a mix of (None, None), centre only, rotation only and both, some far outside the image"""
    mid = rng.uniform(-300.0, 300.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    rot = rng.uniform(-1.5, 1.5, (n, 3))
    mid[3::7] = [4.0e4, -6.0e4, 9.0e5]
    rot[5::7] = [40.0, -25.0, 700.0]
    kind = np.arange(n) % 4
    return mid, rot, (kind & 1) == 1, (kind & 2) == 2


def _single(hp, ctx, frames, Ks, mid=None, rot=None, hm=None, hr=None):
    """dh_predict frame by frame: RESULT_DTYPE[n]"""
    out = np.zeros(len(frames), capi.RESULT_DTYPE)
    for i, d in enumerate(frames):
        kk = IntrinsicMatrix(Ks[i] if Ks.ndim == 3 else Ks)
        mg = mid[i] if mid is not None and (hm is None or hm[i]) else None
        rg = rot[i] if rot is not None and (hr is None or hr[i]) else None
        r = hp.predict_parameter_parallel(d, kk, mg, rg, ctx=ctx)
        out[i]["mid_point"], out[i]["rotation"] = r.mid_point, r.rotation
    return out


def _assert_same(got, want, what):
    assert got.shape == want.shape, what
    for name, view in (("mid_point", np.uint32), ("rotation", np.uint64)):
        a, b = np.ascontiguousarray(got[name]).view(view), np.ascontiguousarray(want[name]).view(view)
        bad = np.argwhere((a != b).any(axis=1)).ravel()
        assert len(bad) == 0, "%s: %s differs at frames %s" % (what, name, bad[:8].tolist())
    assert np.all(got["bounding_box"] == 0) and np.all(got["_pad"] == 0), what


def _encode_context():
    old = os.environ.get("DH_HOST_ENCODE")
    os.environ["DH_HOST_ENCODE"] = "1"
    try:
        return Context(0)
    finally:
        if old is None:
            del os.environ["DH_HOST_ENCODE"]
        else:
            os.environ["DH_HOST_ENCODE"] = old


def test_one_matrix_no_seeds_equals_predict_batch(ctx, model):
    """10 VGA frames in chunks of 3 (two lanes, a tail chunk of 1): host frames, the run-length host
    path and device-resident frames; the counters equal dh_predict_batch's"""
    import torch
    _, hp = model
    frames = synth.make_frames(10, seed=31)
    enc = _encode_context()
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    try:
        for c, where in ((ctx, "host"), (enc, "run-length host"), (ctx, "device")):
            c.set_chunk_frames(3)
            src = dict(device_ptr=dev.data_ptr(), n=10, w=640, h=480) if where == "device" else {}
            arg = None if where == "device" else frames
            want = hp.predict_batch(arg, K, ctx=c, **src)
            cnt_batch = c.counters()
            got = hp.predict_frames(arg, K, ctx=c, **src)
            cnt_frames = c.counters()
            if where == "run-length host":
                assert c.transfer_info()["encoded_chunks"] > 0
            _assert_same(got, want, where)
            if where == "run-length host":  # chunks taken raw by the second copy stream launch no expansion
                cnt_batch.pop("launches"), cnt_frames.pop("launches")
            assert cnt_frames == cnt_batch, (where, cnt_batch, cnt_frames)
            # the same matrix as an [n,3,3] array
            _assert_same(hp.predict_frames(arg, np.tile(K.mat, (10, 1, 1)), ctx=c, **src), want, where + ", K per frame")
            c.set_chunk_frames(0)
    finally:
        ctx.set_chunk_frames(0)
        enc.close()


def test_distinct_matrices_equal_dh_predict_and_the_oracle(ctx, model):
    js, hp = model
    of = oracle.OracleForest.from_json(js)
    frames = synth.make_frames(24, seed=32)
    Ks = _matrices(24)
    want = _single(hp, ctx, frames, Ks)
    for chunk in (0, 7):  # one pass, and passes of 7 frames over two lanes
        ctx.set_chunk_frames(chunk)
        try:
            _assert_same(hp.predict_frames(frames, Ks, ctx=ctx), want, "24 matrices, chunk %d" % chunk)
        finally:
            ctx.set_chunk_frames(0)
    one_k = hp.predict_batch(frames, K, ctx=ctx)
    assert (want["mid_point"] != one_k["mid_point"]).any(axis=1).sum() >= 12  # the matrices do change the poses
    for i in (0, 12, 23):  # 12: the general matrix
        tr = of.predict(frames[i], Ks[i], mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(want[i]["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32)), i
        assert np.array_equal(want[i]["rotation"].view(np.uint64), tr.rotation.view(np.uint64)), i


def test_seeds_mixed_with_matrices(ctx, model):
    """None, centre only, rotation only and both, some far outside the image, with 24 matrices;
    also with device-resident frames and small passes (the in-kernel patch gate below 64 frames)"""
    import torch
    _, hp = model
    n = 28
    frames = synth.make_frames(n, seed=33)
    Ks = _matrices(n)
    mid, rot, hm, hr = _seeds(n, np.random.default_rng(5))
    want = _single(hp, ctx, frames, Ks, mid, rot, hm, hr)
    _assert_same(hp.predict_frames(frames, Ks, mid, rot, hm, hr, ctx=ctx), want, "seeds, host frames")
    unseeded = hp.predict_frames(frames, Ks, ctx=ctx)
    assert (want["rotation"] != unseeded["rotation"]).any(axis=1)[hr].sum() >= n // 4  # the seeds do change the poses
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    ctx.set_chunk_frames(5)
    try:
        got = hp.predict_frames(None, Ks, mid, rot, hm, hr, ctx=ctx, device_ptr=dev.data_ptr(), n=n, w=640, h=480)
    finally:
        ctx.set_chunk_frames(0)
    _assert_same(got, want, "seeds, device frames, chunks of 5")
    # seeds given for every frame (masks None), one matrix
    _assert_same(hp.predict_frames(frames[:6], K, mid[:6], rot[:6], ctx=ctx), _single(hp, ctx, frames[:6], K.mat, mid[:6], rot[:6]),
                 "seeds for every frame")


def test_live_rule_equals_predict_sequences(ctx, model):
    """seeds built on the host from the previous frame's result by the rule of
    examples/live_prediction.rs:75-88 give what dh_predict_sequences computes"""
    _, hp = model
    n_seq, T = 4, 5
    frames = np.stack([synth.make_frames(T, seed=500 + s, sequence=True, start_index=600 * s) for s in range(n_seq)])
    frames[2, 1] = 0
    want = hp.predict_sequences(frames, K, min_seed_z=500.0, ctx=ctx)
    prev = None
    for t in range(T):
        if prev is None:
            got = hp.predict_frames(np.ascontiguousarray(frames[:, t]), K, ctx=ctx)
        else:
            got = hp.predict_frames(np.ascontiguousarray(frames[:, t]), K, np.ascontiguousarray(prev["mid_point"]),
                                    np.ascontiguousarray(prev["rotation"]), prev["mid_point"][:, 2] > np.float32(500.0),
                                    np.ones(n_seq, bool), ctx=ctx)
        _assert_same(got, np.ascontiguousarray(want[:, t]), "pass %d" % t)
        prev = got


def test_biwi_files_with_a_matrix_per_file(ctx, model):
    """one dh_predict_frames_biwi call equals dh_predict_batch_biwi per group of equal K; a damaged
    file is DH_E_ARG naming the first bad frame"""
    _, hp = model
    n = 12
    frames = synth.make_frames(n, seed=34)
    files = [biwi.encode_depth(f) for f in frames]
    groups = _matrices(3)
    which = np.arange(n) % 3
    Ks = groups[which]
    blob, off = biwi.pack_files(files)
    got = biwi.predict_files(hp, blob, off, 640, 480, Ks, ctx=ctx)
    for g in range(3):
        idx = np.flatnonzero(which == g)
        b2, o2 = biwi.pack_files([files[i] for i in idx])
        _assert_same(got[idx], biwi.predict_files(hp, b2, o2, 640, 480, IntrinsicMatrix(groups[g]), ctx=ctx), "group %d" % g)
    mid, rot, hm, hr = _seeds(n, np.random.default_rng(9))
    _assert_same(biwi.predict_files(hp, blob, off, 640, 480, Ks, ctx=ctx, midp_guess=mid, rot_guess=rot, has_midp=hm, has_rot=hr),
                 _single(hp, ctx, frames, Ks, mid, rot, hm, hr), "Biwi files with seeds")
    bad = list(files)
    bad[7] = bad[7][:len(bad[7]) // 2]
    bad[9] = bad[9][:len(bad[9]) // 3]
    b3, o3 = biwi.pack_files(bad)
    with pytest.raises(capi.DhError) as e:
        biwi.predict_files(hp, b3, o3, 640, 480, Ks, ctx=ctx)
    assert e.value.code == capi.DH_E_ARG and "Biwi frame 7 " in str(e.value)


def test_singular_and_non_finite_matrices(ctx, model):
    _, hp = model
    frames = synth.make_frames(6, seed=35)
    Ks = _matrices(6)
    Ks[0] = 0.0                                          # all zero
    Ks[1] = [[560, 0, 320], [1120, 0, 640], [0, 0, 1]]   # rank 2
    Ks[2, 0, 0] = np.nan
    Ks[3, 1, 2] = np.inf
    Ks[4, 2, 2] = 0.0                                    # singular through the last row
    _assert_same(hp.predict_frames(frames, Ks, ctx=ctx), _single(hp, ctx, frames, Ks), "degenerate matrices")


def test_boundaries_and_setters(ctx, model):
    js, _ = model
    hp = HoughPrediction.from_json(js)  # its own model: the setters below change it
    frames = synth.make_frames(5, seed=36)
    Ks = _matrices(5)
    mid, rot, hm, hr = _seeds(5, np.random.default_rng(3))
    # n = 1
    _assert_same(hp.predict_frames(frames[:1], Ks[:1], mid[:1], rot[:1], np.ones(1, bool), np.ones(1, bool), ctx=ctx),
                 _single(hp, ctx, frames[:1], Ks[:1], mid[:1], rot[:1]), "n = 1")
    # n = 0
    assert len(hp.predict_frames(np.zeros((0, 480, 640), np.uint16), np.zeros((0, 3, 3), np.float32), ctx=ctx)) == 0
    # frames of exactly the sub-image size: no patch at all
    y0, x0 = 200, 280
    small = np.ascontiguousarray(frames[:, y0:y0 + 80, x0:x0 + 80])
    _assert_same(hp.predict_frames(small, Ks, mid, rot, hm, hr, ctx=ctx), _single(hp, ctx, small, Ks, mid, rot, hm, hr), "80 x 80")
    # stepwidth, sigma and iterations changed between calls
    prev = None
    for change in (None, ("stepwidth", 7), ("sigma", 3.0), ("meanshift_iterations", 5), ("meanshift_iterations", 0)):
        if change and change[0] == "sigma":
            hp.update_sigma(change[1])
        elif change:
            setattr(hp, change[0], change[1])
        got = hp.predict_frames(frames, Ks, mid, rot, hm, hr, ctx=ctx)
        _assert_same(got, _single(hp, ctx, frames, Ks, mid, rot, hm, hr), "after %s" % (change,))
        plain = hp.predict_frames(frames, Ks, ctx=ctx)  # unseeded: the poses must follow the new stride
        if change and change[0] == "stepwidth":
            assert not (np.array_equal(plain["mid_point"], prev["mid_point"]) and np.array_equal(plain["rotation"], prev["rotation"]))
        prev = plain


def test_launches_depend_on_neither_frames_nor_matrices(ctx, model):
    """device-resident frames in one pass: 1 frame, 32 frames with one matrix and 32 frames with 32
    matrices launch the same kernels, and as many as dh_predict_batch"""
    import torch
    _, hp = model
    frames = synth.make_frames(32, seed=37)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    loc = lambda n: dict(device_ptr=dev.data_ptr(), n=n, w=640, h=480)
    mid, rot, hm, hr = _seeds(32, np.random.default_rng(1))
    launches = []
    for n, Ks in ((1, K), (32, K), (32, _matrices(32))):
        hp.predict_frames(None, Ks, mid[:n], rot[:n], hm[:n], hr[:n], ctx=ctx, **loc(n))
        cnt = ctx.counters()
        assert cnt["frames"] == n
        launches.append(cnt["launches"])
        hp.predict_batch(None, K, ctx=ctx, **loc(n))
        launches.append(ctx.counters()["launches"])
    assert launches[1:] == launches[:-1] and launches[0] > 0, launches
