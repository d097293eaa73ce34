"""GPU tests of the 2-D entry points with a K per frame (dh_build_hough_image_frames) and from Biwi files
(dh_build_hough_image_frames_biwi, dh_predict_mask_batch_biwi).  Raw and blurred vote images are
compared byte for byte and from2d mid_points as uint32 bits with the single-frame calls, with the
one-K batch per group of equal K and, on a subset, with the CPU oracle."""
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
def model():
    """4-tree depth-6 forest at stride 10 (as test_gpu_hough2d_batch.py)"""
    arr = synth.make_forest(seed=3, n_trees=4, max_depth=6)
    js = synth.forest_to_json(arr, stepwidth=10)
    return js, HoughPrediction.from_json(js)


def _matrices(n):
    """n intrinsics: focal lengths and principal points that vary, and one general 3x3 with non-zero
    off-diagonal terms (including the bottom row) at n // 2"""
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 480.0 + 7.5 * i
        Ks[i] = [[f, 0.0, 300.0 + 2.0 * i], [0.0, f * 1.01, 230.0 + 1.5 * i], [0.0, 0.0, 1.0]]
    Ks[n // 2] = [[561.5, 3.25, 318.0], [-2.5, 557.0, 243.5], [1.0e-4, -2.0e-4, 1.0]]
    return Ks


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


def _single(hp, ctx, frames, Ks):
    """(raw, blurred, from2d mid_point) from the single-frame calls, frame i with Ks[i]"""
    kk = [IntrinsicMatrix(Ks[i] if Ks.ndim == 3 else Ks) for i in range(len(frames))]
    raw = np.stack([hp.hough_image_raw(d, kk[i], ctx=ctx) for i, d in enumerate(frames)])
    blur = np.stack([hp.build_hough_image(d, kk[i], ctx=ctx) for i, d in enumerate(frames)])
    mids = np.stack([hp.predict_parameter_from2dhough(d, kk[i], ctx=ctx).mid_point for i, d in enumerate(frames)])
    return raw, blur, mids


def _frames(hp, ctx, frames, Ks, **src):
    """(raw, blurred, from2d mid_point) from the three _frames wrappers"""
    raw = hp.hough_image_raw_frames(frames, Ks, ctx=ctx, **src)
    blur, res = hp.build_hough_image_frames(frames, Ks, ctx=ctx, from2d=True, **src)
    only = hp.predict_parameter_from2dhough_frames(frames, Ks, ctx=ctx, **src)
    assert np.array_equal(only.view(np.uint8), res.view(np.uint8))
    assert np.all(res["rotation"] == 0.0) and np.all(res["bounding_box"] == 0) and np.all(res["_pad"] == 0)
    return raw, blur, res["mid_point"]


def _batch(hp, ctx, frames, k, **src):
    raw = hp.hough_image_raw_batch(frames, k, ctx=ctx, **src)
    blur, res = hp.build_hough_image_batch(frames, k, ctx=ctx, from2d=True, **src)
    return raw, blur, res["mid_point"]


def _assert_same(got, want, what):
    for name, a, b in zip(("raw votes", "blurred votes", "from2d mid_point"), got, want):
        if name == "from2d mid_point":
            a, b = np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32)
        assert a.shape == b.shape, (what, name, a.shape, b.shape)
        bad = np.argwhere(a != b)
        assert len(bad) == 0, "%s: %s differs at %d places, first %s" % (what, name, len(bad), bad[0].tolist())


def test_one_matrix_repeated_equals_the_batch(ctx, model):
    """10 VGA frames in chunks of 3 (two lanes, a tail of 1): results equal dh_build_hough_image_batch, with
    one IntrinsicMatrix and with it repeated as [n,3,3]; device-resident frames: every counter equal too"""
    import torch
    _, hp = model
    frames = synth.make_frames(10, seed=61)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    ctx.set_chunk_frames(3)
    try:
        for where in ("host", "device"):
            src = dict(device_ptr=dev.data_ptr(), n=10, w=640, h=480) if where == "device" else {}
            arg = None if where == "device" else frames
            want = _batch(hp, ctx, arg, K, **src)
            assert want[0].max() > 0 and want[1].max() > 0
            _assert_same(_frames(hp, ctx, arg, K, **src), want, where + ", one IntrinsicMatrix")
            _assert_same(_frames(hp, ctx, arg, np.tile(K.mat, (10, 1, 1)), **src), want, where + ", K repeated")
            if where == "device":
                for blur in (False, True):
                    calls = ((hp.hough_image_raw_batch, hp.hough_image_raw_frames) if not blur else
                             (lambda *a, **kw: hp.build_hough_image_batch(*a, from2d=True, **kw),
                              lambda *a, **kw: hp.build_hough_image_frames(*a, from2d=True, **kw)))
                    calls[0](None, K, ctx=ctx, **src)
                    cnt_batch = ctx.counters()
                    calls[1](None, np.tile(K.mat, (10, 1, 1)), ctx=ctx, **src)
                    assert ctx.counters() == cnt_batch, (blur, cnt_batch, ctx.counters())
    finally:
        ctx.set_chunk_frames(0)


def test_24_matrices_over_three_image_chunks(ctx, model):
    """240 VGA frames, frame i with matrix i % 24: image chunks are capped at 109 VGA frames, so the call
    runs chunks of 109, 109 and 22 over both lanes.  Equal to the single-frame calls, to one _batch call
    per group of equal K, and on a subset to the oracle."""
    js, hp = model
    of = oracle.OracleForest.from_json(js)
    n = 240
    frames = synth.make_frames(n, seed=62)
    groups = _matrices(24)
    which = np.arange(n) % 24
    Ks = np.ascontiguousarray(groups[which])
    got = _frames(hp, ctx, frames, Ks)
    _assert_same(got, _single(hp, ctx, frames, Ks), "24 matrices vs single-frame calls")
    for g in range(24):
        idx = np.flatnonzero(which == g)
        _assert_same([a[idx] for a in got], _batch(hp, ctx, np.ascontiguousarray(frames[idx]), IntrinsicMatrix(groups[g])),
                     "group %d vs its _batch call" % g)
    one_k = _batch(hp, ctx, frames, K)
    assert (got[0] != one_k[0]).any(axis=(1, 2)).sum() >= n // 2  # the matrices do change the images
    assert (got[2] != one_k[2]).any(axis=1).sum() >= n // 4
    for i in (0, 12, 108, 109, 218, 219, 239):  # 12: the general matrix; 108 / 109 and 218 / 219: chunk edges
        k = Ks[i]
        assert np.array_equal(got[0][i], of.hough_image_raw(frames[i], k)), i
        assert np.array_equal(got[1][i], of.build_hough_image(frames[i], k)), i
        mid, _ = of.predict_parameter_from2dhough(frames[i], k)
        assert np.array_equal(got[2][i].view(np.uint32), np.asarray(mid, np.float32).view(np.uint32)), i


@pytest.mark.parametrize("out_dev", [False, True], ids=["host_out", "device_out"])
@pytest.mark.parametrize("where", ["host", "device", "run_length"])
def test_input_and_output_locations(ctx, model, where, out_dev):
    """12 frames with 12 matrices in chunks of 5: host frames, device frames and the run-length host path;
    images to host and to device memory"""
    import torch
    _, hp = model
    n = 12
    frames = synth.make_frames(n, seed=63)
    Ks = _matrices(n)
    want = _single(hp, ctx, frames, Ks)
    c = _encode_context() if where == "run_length" else ctx
    src = {}
    if where == "device":
        dev = torch.from_numpy(frames.view(np.int16)).cuda()
        torch.cuda.synchronize()
        src = dict(device_ptr=dev.data_ptr(), n=n, w=640, h=480)
    arg = None if where == "device" else frames

    def run(fn, **kw):
        if not out_dev:
            return fn(arg, Ks, ctx=c, **src, **kw)
        out = torch.full((n, 480, 640), 77, dtype=torch.int16, device="cuda")
        torch.cuda.synchronize()
        r = fn(arg, Ks, ctx=c, **src, out_device_ptr=out.data_ptr(), **kw)
        img = out.cpu().numpy().view(np.uint16)
        if isinstance(r, tuple):
            assert r[0] is None
            return img, r[1]
        assert r is None
        return img

    c.set_chunk_frames(5)
    try:
        raw = run(hp.hough_image_raw_frames)
        blur, res = run(hp.build_hough_image_frames, from2d=True)
        if where == "run_length":
            assert c.transfer_info()["encoded_chunks"] > 0
        _assert_same((raw, blur, res["mid_point"]), want, "%s in, %s out" % (where, "device" if out_dev else "host"))
        if out_dev:
            blur2 = run(hp.build_hough_image_frames)
            assert np.array_equal(blur2, want[1])
    finally:
        c.set_chunk_frames(0)
        if c is not ctx:
            c.close()


def test_biwi_files(ctx, model):
    """130 Biwi files (more than one capped image chunk of 109 VGA frames) with 24 matrices: one call
    equals the frames call on the decoded frames, and the mask call equals dh_predict_mask_batch;
    images to host and to device memory"""
    import torch
    _, hp = model
    n = 130
    frames = synth.make_frames(n, seed=64)
    Ks = np.ascontiguousarray(_matrices(24)[np.arange(n) % 24])
    blob, off = biwi.encode_frames(frames)
    want = _frames(hp, ctx, frames, Ks)
    blur, res = biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, from2d=True, ctx=ctx)
    raw = biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, blur=False, ctx=ctx)
    only = biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, from2d=True, images=False, ctx=ctx)
    assert only[0] is None and np.array_equal(only[1].view(np.uint8), res.view(np.uint8))
    _assert_same((raw, blur, res["mid_point"]), want, "Biwi files vs frames call")
    mask = biwi.predict_mask_files(hp, blob, off, 640, 480, ctx=ctx)
    mask_want = hp.predict_mask_batch(frames, ctx=ctx)
    assert mask.max() > 0 and np.array_equal(mask, mask_want)
    out = torch.zeros((n, 480, 640), dtype=torch.int16, device="cuda")
    out8 = torch.zeros((n, 480, 640), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, ctx=ctx, out_device_ptr=out.data_ptr()) is None
    assert biwi.predict_mask_files(hp, blob, off, 640, 480, ctx=ctx, out_device_ptr=out8.data_ptr()) is None
    assert np.array_equal(out.cpu().numpy().view(np.uint16), want[1])
    assert np.array_equal(out8.cpu().numpy(), mask_want)
    # one K for every file: the same as the one-K batch
    raw1 = biwi.build_hough_image_files(hp, blob, off, 640, 480, K, blur=False, ctx=ctx)
    blur1, res1 = biwi.build_hough_image_files(hp, blob, off, 640, 480, K, from2d=True, ctx=ctx)
    _assert_same((raw1, blur1, res1["mid_point"]), _batch(hp, ctx, frames, K), "Biwi files, one K")


def test_damaged_biwi_files_and_wrong_sizes(ctx, model):
    _, hp = model
    n = 12
    frames = synth.make_frames(n, seed=65)
    files = [biwi.encode_depth(f) for f in frames]
    Ks = _matrices(n)
    bad = list(files)
    bad[7] = bad[7][:len(bad[7]) // 2]
    bad[9] = bad[9][:len(bad[9]) // 3]
    blob, off = biwi.pack_files(bad)
    for call in (lambda: biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, from2d=True, ctx=ctx),
                 lambda: biwi.build_hough_image_files(hp, blob, off, 640, 480, Ks, blur=False, ctx=ctx),
                 lambda: biwi.predict_mask_files(hp, blob, off, 640, 480, ctx=ctx)):
        with pytest.raises(capi.DhError) as e:
            call()
        assert e.value.code == capi.DH_E_ARG and "Biwi frame 7 " in str(e.value), str(e.value)
    good, goff = biwi.pack_files(files)
    for call in (lambda: biwi.build_hough_image_files(hp, good, goff, 320, 240, Ks, ctx=ctx),
                 lambda: biwi.predict_mask_files(hp, good, goff, 320, 240, ctx=ctx)):
        with pytest.raises(capi.DhError) as e:
            call()
        assert e.value.code == capi.DH_E_ARG and "Biwi frame 0 has a header" in str(e.value), str(e.value)
    # the context still works, and the good files give the frames call's results
    _assert_same(_frames(hp, ctx, frames, Ks), _single(hp, ctx, frames, Ks), "after the errors")


def test_degenerate_matrices(ctx, model):
    _, hp = model
    frames = synth.make_frames(6, seed=66)
    Ks = _matrices(6)
    Ks[0] = 0.0                                          # all zero
    Ks[1] = [[560, 0, 320], [1120, 0, 640], [0, 0, 1]]   # rank 2
    Ks[2, 0, 0] = np.nan
    Ks[3, 1, 2] = np.inf
    Ks[4, 2, 2] = 0.0                                    # singular through the last row
    _assert_same(_frames(hp, ctx, frames, Ks), _single(hp, ctx, frames, Ks), "degenerate matrices")


def test_launches_depend_on_neither_frames_nor_matrices(ctx, model):
    """device-resident frames: at n = 1 and n = 32, in one pass and in passes of 7, one matrix and 32
    matrices launch as many kernels as the one-K batch at the same n and chunk size"""
    import torch
    _, hp = model
    frames = synth.make_frames(32, seed=67)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    loc = lambda n: dict(device_ptr=dev.data_ptr(), n=n, w=640, h=480)
    try:
        for chunk in (0, 7):
            ctx.set_chunk_frames(chunk)
            for n in (1, 32):
                for name, batch, per_frame in (
                        ("raw", lambda k: hp.hough_image_raw_batch(None, k, ctx=ctx, **loc(n)),
                         lambda k: hp.hough_image_raw_frames(None, k, ctx=ctx, **loc(n))),
                        ("blurred + from2d", lambda k: hp.build_hough_image_batch(None, k, ctx=ctx, from2d=True, **loc(n)),
                         lambda k: hp.build_hough_image_frames(None, k, ctx=ctx, from2d=True, **loc(n))),
                        ("from2d", lambda k: hp.predict_parameter_from2dhough_batch(None, k, ctx=ctx, **loc(n)),
                         lambda k: hp.predict_parameter_from2dhough_frames(None, k, ctx=ctx, **loc(n)))):
                    batch(K)
                    want = ctx.counters()["launches"]
                    for Ks in (K, _matrices(n)):
                        per_frame(Ks)
                        cnt = ctx.counters()
                        assert cnt["frames"] == n and cnt["launches"] == want > 0, (chunk, n, name, want, cnt)
    finally:
        ctx.set_chunk_frames(0)


def test_boundaries_and_setters(ctx, model):
    js, _ = model
    hp = HoughPrediction.from_json(js)  # its own model: the setters below change it
    of = oracle.OracleForest.from_json(js)
    frames = synth.make_frames(5, seed=68)
    Ks = _matrices(5)
    # n = 1, against the oracle too
    got = _frames(hp, ctx, frames[:1], Ks[:1])
    _assert_same(got, _single(hp, ctx, frames[:1], Ks[:1]), "n = 1")
    assert np.array_equal(got[1][0], of.build_hough_image(frames[0], Ks[0]))
    # n = 0
    empty = np.zeros((0, 480, 640), np.uint16)
    assert hp.hough_image_raw_frames(empty, np.zeros((0, 3, 3), np.float32), ctx=ctx).shape == (0, 480, 640)
    assert len(hp.predict_parameter_from2dhough_frames(empty, K, ctx=ctx)) == 0
    assert biwi.predict_mask_files(hp, np.zeros(16, np.uint8), np.zeros(1, np.uint64), 640, 480, ctx=ctx).shape == (0, 480, 640)
    # frames of exactly the sub-image size: no patch at all
    small = np.ascontiguousarray(frames[:, 200:280, 280:360])
    got = _frames(hp, ctx, small, Ks)
    _assert_same(got, _single(hp, ctx, small, Ks), "80 x 80")
    assert got[0].max() == 0
    # sigma and stepwidth changed between calls
    prev = _frames(hp, ctx, frames, Ks)
    for change in (("sigma", 3.0), ("stepwidth", 7)):
        if change[0] == "sigma":
            hp.update_sigma(change[1])
            of.update_sigma(change[1])
        else:
            hp.stepwidth = of.stepwidth = change[1]
        got = _frames(hp, ctx, frames, Ks)
        _assert_same(got, _single(hp, ctx, frames, Ks), "after %s" % (change,))
        assert np.array_equal(got[1][2], of.build_hough_image(frames[2], Ks[2])), change
        assert not np.array_equal(got[1], prev[1]), change
        prev = got
