"""GPU tests of the batched 2-D entry points: predict_mask_batch, hough_image_raw_batch,
build_hough_image_batch and predict_parameter_from2dhough_batch.  Every mask, raw vote image,
blurred image and from2d mid_point (compared as uint32) must equal, bit for bit, both the CPU
oracle frame by frame and the single-frame GPU calls."""
import os

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small():
    """4-tree depth-6 forest at stride 10 and five VGA frames, the third all zero"""
    arr = synth.make_forest(seed=3, n_trees=4, max_depth=6)
    js = synth.forest_to_json(arr, stepwidth=10)
    frames = synth.make_frames(4, seed=11)
    frames = np.ascontiguousarray(np.concatenate([frames[:2], np.zeros((1, 480, 640), np.uint16), frames[2:]]))
    return js, frames


def _crop(frames, h, w):
    y0, x0 = (frames.shape[1] - h) // 2, (frames.shape[2] - w) // 2
    return np.ascontiguousarray(frames[:, y0:y0 + h, x0:x0 + w])


def _oracle(of, frames):
    mask = np.stack([of.predict_mask(d) for d in frames])
    raw = np.stack([of.hough_image_raw(d, synth.KINECT_K) for d in frames])
    blur = np.stack([of.build_hough_image(d, synth.KINECT_K) for d in frames])
    mids, xys = zip(*[of.predict_parameter_from2dhough(d, synth.KINECT_K) for d in frames])
    return mask, raw, blur, np.stack(mids).astype(np.float32), list(xys)


def _single(hp, ctx, frames):
    mask = np.stack([hp.predict_mask(d, ctx=ctx) for d in frames])
    raw = np.stack([hp.hough_image_raw(d, K, ctx=ctx) for d in frames])
    blur = np.stack([hp.build_hough_image(d, K, ctx=ctx) for d in frames])
    mids = np.stack([hp.predict_parameter_from2dhough(d, K, ctx=ctx).mid_point for d in frames])
    return mask, raw, blur, mids


def _batch(hp, ctx, frames):
    mask = hp.predict_mask_batch(frames, ctx=ctx)
    raw = hp.hough_image_raw_batch(frames, K, ctx=ctx)
    blur, res = hp.build_hough_image_batch(frames, K, ctx=ctx, from2d=True)
    only = hp.predict_parameter_from2dhough_batch(frames, K, ctx=ctx)
    assert np.array_equal(only.view(np.uint8), res.view(np.uint8))
    assert np.all(res["rotation"] == 0.0) and np.all(res["bounding_box"] == 0) and np.all(res["_pad"] == 0)
    return mask, raw, blur, res["mid_point"]


def _assert_same(got, want, what):
    names = ("mask", "raw votes", "blurred votes", "from2d mid_point")
    for name, a, b in zip(names, got, want):
        if name == names[3]:
            a, b = np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32)
        assert a.shape == b.shape, (what, name, a.shape, b.shape)
        bad = np.argwhere(a != b)
        assert len(bad) == 0, "%s: %s differs at %d places, first %s" % (what, name, len(bad), bad[0].tolist())


def _check(hp, of, ctx, frames, what):
    got = _batch(hp, ctx, frames)
    want = _oracle(of, frames)
    _assert_same(got, want[:4], what + " vs oracle")
    _assert_same(got, _single(hp, ctx, frames), what + " vs single-frame calls")
    return got, want


def test_small_case_with_an_empty_frame(ctx, small):
    js, frames = small
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    got, want = _check(hp, of, ctx, frames, "small case")
    assert got[0].max() > 0 and got[1].max() > 0
    # the all-zero frame: an all-zero vote image, whose arg-max is the LAST pixel
    assert got[2][2].max() == 0 and want[4][2] == (639, 479)


@pytest.mark.parametrize("stride", [1, 5, 7, 10])
@pytest.mark.parametrize("ragged", [True, False], ids=["sat", "box_image"])
def test_front_ends_and_strides(ctx, ragged, stride):
    """general rectangles (summed-area-table front end) and one rectangle size (box-image front end)"""
    arr = synth.make_forest(seed=21, n_trees=5, max_depth=8, ragged_rects=ragged)
    js = synth.forest_to_json(arr, stepwidth=stride)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    frames = synth.make_frames(3, seed=40 + stride)
    if stride == 1:
        frames = _crop(frames, 200, 240)
    got, _ = _check(hp, of, ctx, frames, "ragged=%s stride=%d" % (ragged, stride))
    assert got[0].max() > 0


def test_vote_heavy_forest_at_stride_1(ctx):
    arr = synth.make_forest(seed=13, n_trees=10, max_depth=8, votes_lo=32, votes_hi=128)
    js = synth.forest_to_json(arr, stepwidth=1)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    got, _ = _check(hp, of, ctx, _crop(synth.make_frames(3, seed=5), 200, 200), "vote-heavy stride 1")
    assert got[1].max() > 0


@pytest.mark.parametrize("sigma,sub,scale,stride,hw", [(1.5, (80, 80), 0.3, 5, (480, 640)), (3.0, (80, 80), 0.3, 7, (203, 331)),
                                                      (0.4, (64, 48), 0.5, 4, (150, 296)), (11.0, (40, 56), 0.13, 3, (97, 120)),
                                                      (8.0, (96, 96), 0.9, 9, (200, 264))])
def test_odd_shapes_and_sigmas(ctx, sigma, sub, scale, stride, hw):
    arr = synth.make_forest(seed=17, n_trees=3, max_depth=6, sub_w=sub[0], sub_h=sub[1], rect_scale=scale)
    js = synth.forest_to_json(arr, stepwidth=stride)
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    hp.update_sigma(sigma)
    of.update_sigma(sigma)
    _check(hp, of, ctx, _crop(synth.make_frames(3, seed=5), *hw), "sigma %s shape %s" % (sigma, hw))


def test_frames_of_the_subimage_size(ctx, small):
    """w = subimage_width, h = subimage_height: no patch at all (P = 0)"""
    js, frames = small
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    got, want = _check(hp, of, ctx, _crop(frames, 80, 80), "sub-image sized frames")
    assert got[0].max() == 0 and got[1].max() == 0 and all(xy == (79, 79) for xy in want[4])


def test_several_chunks_both_lanes_and_a_tail(ctx, small):
    js, frames = small
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    many = np.ascontiguousarray(np.concatenate([frames, frames[::-1]]))  # 10 frames
    ctx.set_chunk_frames(3)
    try:
        _check(hp, of, ctx, many, "chunks of 3")
    finally:
        ctx.set_chunk_frames(0)


@pytest.mark.parametrize("out_dev", [False, True], ids=["host_out", "device_out"])
@pytest.mark.parametrize("in_dev", [False, True], ids=["host_in", "device_in"])
def test_input_and_output_locations(ctx, small, in_dev, out_dev):
    import torch
    js, frames = small
    hp = HoughPrediction.from_json(js)
    want = _single(hp, ctx, frames)
    n, h, w = frames.shape
    src = {}
    if in_dev:
        dev = torch.from_numpy(frames.view(np.int16)).cuda()
        src = dict(device_ptr=dev.data_ptr(), n=n, w=w, h=h)
    arg = None if in_dev else frames

    def run(fn, dtype, **kw):
        if not out_dev:
            return fn(arg, ctx=ctx, **src, **kw)
        out = torch.full((n, h, w), 77, dtype=torch.uint8 if dtype == np.uint8 else torch.int16, device="cuda")
        torch.cuda.synchronize()
        r = fn(arg, ctx=ctx, **src, out_device_ptr=out.data_ptr(), **kw)
        img = out.cpu().numpy().view(dtype)
        if isinstance(r, tuple):  # (None, from2d results): nothing on the host but the results
            assert r[0] is None
            return img, r[1]
        assert r is None
        return img

    if in_dev:
        torch.cuda.synchronize()
    mask = run(hp.predict_mask_batch, np.uint8)
    raw = run(lambda a, **kw: hp.hough_image_raw_batch(a, K, **kw), np.uint16)
    blur, res = run(lambda a, **kw: hp.build_hough_image_batch(a, K, from2d=True, **kw), np.uint16)
    only = hp.predict_parameter_from2dhough_batch(arg, K, ctx=ctx, **src)
    assert np.array_equal(only.view(np.uint8), res.view(np.uint8))
    _assert_same((mask, raw, blur, res["mid_point"]), want, "in_dev=%s out_dev=%s" % (in_dev, out_dev))
    if out_dev:  # the blurred image alone to device memory, no from2d
        out = torch.zeros((n, h, w), dtype=torch.int16, device="cuda")
        torch.cuda.synchronize()
        assert hp.build_hough_image_batch(arg, K, ctx=ctx, **src, out_device_ptr=out.data_ptr()) is None
        assert np.array_equal(out.cpu().numpy().view(np.uint16), want[2])


def test_encoded_host_path(small):
    """16 VGA host frames in a context that rewrites host chunks as run-length files"""
    js, _ = small
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    frames = synth.make_frames(16, seed=23)
    old = os.environ.get("DH_HOST_ENCODE")
    os.environ["DH_HOST_ENCODE"] = "1"
    try:
        c = Context(0)
    finally:
        if old is None:
            del os.environ["DH_HOST_ENCODE"]
        else:
            os.environ["DH_HOST_ENCODE"] = old
    try:
        got = _batch(hp, c, frames)
        assert c.transfer_info()["encoded_chunks"] > 0
        _assert_same(got, _single(hp, c, frames), "encoded host path vs single-frame calls")
        want = _oracle(of, frames[:3])
        _assert_same([g[:3] for g in got], want[:4], "encoded host path vs oracle")
    finally:
        c.close()


def test_sigma_and_stepwidth_changes_between_calls(ctx, small):
    """the blur taps are cached per model and sigma: update_sigma and a new stepwidth must show"""
    js, frames = small
    hp = HoughPrediction.from_json(js)
    of = oracle.OracleForest.from_json(js)
    f3 = frames[:2]
    first = _check(hp, of, ctx, f3, "sigma 8")[0]
    hp.update_sigma(3.0)
    of.update_sigma(3.0)
    second = _check(hp, of, ctx, f3, "sigma 3")[0]
    assert not np.array_equal(first[2], second[2])
    hp.stepwidth = 7
    of.stepwidth = 7
    third = _check(hp, of, ctx, f3, "sigma 3, stride 7")[0]
    assert not np.array_equal(second[1], third[1])


def test_launches_do_not_depend_on_frames_and_counters(ctx, small):
    """a 1-frame call and a 32-frame call of one chunk launch the same kernels (device-resident
    frames: host frames of a large batch may take the run-length path, which adds its expansion)"""
    import torch
    js, frames = small
    hp = HoughPrediction.from_json(js)
    many = np.ascontiguousarray(np.concatenate([frames] * 7)[:32])
    dev = torch.from_numpy(many.view(np.int16)).cuda()
    torch.cuda.synchronize()
    loc = lambda n: dict(device_ptr=dev.data_ptr(), n=n, w=640, h=480)
    calls = (lambda n: hp.predict_mask_batch(None, ctx=ctx, **loc(n)), lambda n: hp.hough_image_raw_batch(None, K, ctx=ctx, **loc(n)),
             lambda n: hp.build_hough_image_batch(None, K, ctx=ctx, from2d=True, **loc(n)),
             lambda n: hp.predict_parameter_from2dhough_batch(None, K, ctx=ctx, **loc(n)))
    for i, call in enumerate(calls):
        call(1)
        one = ctx.counters()
        call(32)
        cnt = ctx.counters()
        assert cnt["launches"] == one["launches"] > 0, (i, one, cnt)
        assert cnt["frames"] == 32 and one["frames"] == 1
        assert cnt["patches"] == 32 * one["patches"] > 0
        assert cnt["valid_patches"] > 0 and cnt["evals"] == cnt["valid_patches"] * hp.n_trees and cnt["node_visits"] > 0
        for k in ("gate_patches", "hits", "centre_votes", "rot_votes", "meanshift_iters", "cube_rebuilds"):
            assert cnt[k] == 0, (i, k, cnt)
    ctx.enable_stage_timing(True)
    try:
        hp.build_hough_image_batch(many, K, ctx=ctx, from2d=True)
        ms = ctx.stage_ms()
    finally:
        ctx.enable_stage_timing(False)
    assert ms["sat"] > 0 and ms["traverse"] > 0 and ms["vote"] > 0 and ms["h2d"] > 0 and ms["d2h"] > 0, ms
    assert ms["gate"] == 0 and ms["meanshift"] == 0, ms


def test_empty_batch_and_shape_errors(ctx, small):
    js, frames = small
    hp = HoughPrediction.from_json(js)
    assert hp.predict_mask_batch(np.zeros((0, 480, 640), np.uint16), ctx=ctx).shape == (0, 480, 640)
    assert len(hp.predict_parameter_from2dhough_batch(np.zeros((0, 480, 640), np.uint16), K, ctx=ctx)) == 0
    with pytest.raises(capi.DhError) as e:
        hp.build_hough_image_batch(np.zeros((2, 60, 60), np.uint16), K, ctx=ctx)
    assert e.value.code == capi.DH_E_SHAPE
