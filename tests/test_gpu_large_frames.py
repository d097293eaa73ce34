"""GPU parity on frames larger than VGA, up to the largest accepted side (32768 pixels).

Depth cameras deliver 848x480, 1280x720, 640x576 or 1024x1024 frames, and the library picks several
code paths from the frame size alone: the two-pass summed-area table from 1024 columns on, the widest
banded table at 1023, box images whose strips spread over several CTAs from 1880 columns on, the
seed-grid cell by division instead of multiply-high from 14655 pixels on, the image back end at its
chunk cap and pose passes capped by the per-frame scratch budget.  Every stage is compared bit for
bit against the CPU oracle on these shapes, with an intrinsic matrix scaled to the frame so that the
synthetic head lies inside the image."""
import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth
from test_gpu_parity import _compare_frame

pytestmark = pytest.mark.gpu

SUB = 80                       # make_forest's default patch size
RECT = 24                      # ... and its rectangle size (rect_scale 0.3), the box-image front end's
# uniform 24x24 rectangles take the box-sum image; ragged rectangles take the summed-area table
FORESTS = {"box_image": (dict(seed=51, n_trees=4, max_depth=8), 5),
           "sat": (dict(seed=52, n_trees=3, max_depth=7, ragged_rects=True), 6)}


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def _scaled_K(w, h, scale=1.0, shift=0.0):
    """the Kinect matrix scaled to a w x h frame, as synth.make_frames projects its person"""
    return np.array([[560.0 * w / 640.0 * scale, 0.0, w / 2.0 + shift],
                     [0.0, 560.0 * h / 480.0 * scale, h / 2.0 - shift],
                     [0.0, 0.0, 1.0]], np.float32)


def _models(forest):
    kw, stride = FORESTS[forest]
    js = synth.forest_to_json(synth.make_forest(**kw), stepwidth=stride)
    return HoughPrediction.from_json(js), oracle.OracleForest.from_json(js), stride


def _noise(w, h, seed):
    """random u16 depth with half of the pixels zeroed: most patches are valid and many pass the gate"""
    rng = np.random.default_rng([seed, w, h])
    d = rng.integers(0, 65536, (h, w)).astype(np.uint16)
    d[rng.random((h, w)) < 0.5] = 0
    return d


def _grid_patches(w, h, stride, sub=SUB):
    return (w - sub + stride - 1) // stride, (h - sub + stride - 1) // stride


SHAPES = [
    (848, 480),      # real sensors; 848 + 1 <= 1024: banded summed-area table
    (1280, 720),     # w + 1 > 1024: two-pass table (sat_rows_kernel + sat_cols_kernel)
    (1024, 1024),    # the first width on the two-pass table
    (640, 576),
    (1023, 600),     # w + 1 = 1024: the widest banded table (1024-thread band sums, 132 KB of shared memory);
                     # width not a multiple of 8
    (1879, 200),     # box image 1856 wide = 8 strips of 232 columns: one CTA per (frame, band), 8 warps
    (1880, 200),     # box image 1857 wide = 9 strips: 2 warps per CTA, a frame's strips over several CTAs
    (1920, 1080),    # 9 strips at full HD
    (1917, 1079),    # odd width: scalar pixel loads
    # the seed-grid cell x * 20 / w (y * 20 / h) is a multiply-high when ensure_scratch finds an exact constant,
    # i.e. 20 * (d - 1) * d < 2^32: magic_w / magic_h are nonzero up to 14654 and 0 (real division) from 14655 on
    (14654, 100),    # the last divisor with a multiply-high constant ...
    (14655, 100),    # ... and the first one whose seed-grid cell is a division, along x
    (100, 14655),    # ... and along y
    (32768, 96),     # the largest accepted side: 142 strips, long rows of the table
    (96, 32768),     # a tall table, many bands
]


@pytest.mark.parametrize("forest", list(FORESTS))
@pytest.mark.parametrize("w,h", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_every_stage_at_large_shapes(ctx, w, h, forest):
    """leaf ids, gates, p3, seed grids, seeds, accumulator cells, mean-shift trajectories and poses of a
    person frame, a noise frame and a saturated frame; then the same frames as one batch"""
    hp, of, stride = _models(forest)
    K = _scaled_K(w, h)
    frames = [synth.make_frames(1, seed=900 + w + h, w=w, h=h)[0], _noise(w, h, 900), np.full((h, w), 65535, np.uint16)]
    traces = [_compare_frame(ctx, hp, of, d, intrinsic=K)[1] for d in frames]
    npx, npy = _grid_patches(w, h, stride)
    assert traces[0].npx * traces[0].npy == npx * npy
    # the premises of the row
    plan = ctx.tile_plan()
    assert (plan["tiles_x"] - 1) * plan["patches_x"] < npx <= plan["tiles_x"] * plan["patches_x"], plan
    assert (plan["tiles_y"] - 1) * plan["patches_y"] < npy <= plan["tiles_y"] * plan["patches_y"], plan
    # tile rows: sh + 1 taps of the summed-area table, sh - rh + 1 of the box-sum image
    assert plan["tile_h"] - (plan["patches_y"] - 1) * stride == (SUB - RECT + 1 if forest == "box_image" else SUB + 1), plan
    assert sum(int(t.guess_pos.sum()) for t in traces) > 0, "no centre vote reached the seed grid"
    assert sum(int(t.gate.sum()) for t in traces) > 0
    out = hp.predict_batch(np.stack(frames), IntrinsicMatrix(K), ctx=ctx)
    assert ctx.counters()["patches"] == len(frames) * npx * npy
    for i, tr in enumerate(traces):
        assert np.array_equal(out["mid_point"][i], tr.mid_point), i
        assert np.array_equal(out["rotation"][i].view(np.uint64), tr.rotation.view(np.uint64)), i


def test_side_limits(ctx):
    """sides up to 32768 pixels, and at least 20 (the 20x20 seed grid): DH_E_SHAPE beyond"""
    hp, _, _ = _models("box_image")
    for w, h in ((32769, 96), (96, 32769)):
        d = _noise(w, h, 3)
        K = IntrinsicMatrix(_scaled_K(w, h))
        with pytest.raises(capi.DhError) as e:
            hp.predict_parameter_parallel(d, K, ctx=ctx)
        assert e.value.code == capi.DH_E_SHAPE, (w, h)
        with pytest.raises(capi.DhError) as e:
            hp.predict_batch(d[None], K, ctx=ctx)
        assert e.value.code == capi.DH_E_SHAPE, (w, h)
    arr = synth.make_forest(seed=54, n_trees=3, max_depth=6, sub_w=12, sub_h=12)
    js = synth.forest_to_json(arr, stepwidth=2)
    hp12, of12 = HoughPrediction.from_json(js), oracle.OracleForest.from_json(js)
    rng = np.random.default_rng(11)
    d = rng.integers(400, 1500, (20, 20)).astype(np.uint16)
    _compare_frame(ctx, hp12, of12, d, intrinsic=_scaled_K(20, 20))
    for h, w in ((20, 19), (19, 20)):
        with pytest.raises(capi.DhError) as e:
            hp12.predict_parameter_parallel(np.ascontiguousarray(d[:h, :w]), IntrinsicMatrix(_scaled_K(w, h)), ctx=ctx)
        assert e.value.code == capi.DH_E_SHAPE, (w, h)


@pytest.mark.parametrize("forest", list(FORESTS))
def test_batch_paths_at_720p(monkeypatch, ctx, forest):
    """12 frames of 1280x720 through the run-length host path, the plain host path, device input at an odd
    2-byte offset and predict_frames with a matrix per frame: identical to each other, to single-frame calls
    and to the oracle"""
    import torch
    w, h, n = 1280, 720, 12
    hp, of, _ = _models(forest)
    K = _scaled_K(w, h)
    frames = np.stack([synth.make_frames(1, seed=300 + i, w=w, h=h)[0] if i % 2 == 0 else _noise(w, h, 300 + i)
                       for i in range(n)])
    outs = {}
    for enc in ("1", "0"):
        monkeypatch.setenv("DH_HOST_ENCODE", enc)
        c = Context(0)
        try:
            outs[enc] = hp.predict_batch(frames, IntrinsicMatrix(K), ctx=c)
            assert (c.transfer_info()["encoded_chunks"] > 0) == (enc == "1")
        finally:
            c.close()
    flat = torch.zeros(frames.size + 8, dtype=torch.int16, device="cuda")
    flat[3:3 + frames.size] = torch.from_numpy(frames.view(np.int16).reshape(-1)).cuda()
    torch.cuda.synchronize()
    dev = hp.predict_batch(None, IntrinsicMatrix(K), ctx=ctx, device_ptr=flat.data_ptr() + 2 * 3, n=n, w=w, h=h)
    assert outs["1"].tobytes() == outs["0"].tobytes() == dev.tobytes()
    for i in (0, 5, 11):
        tr = of.predict(frames[i], K, mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(dev["mid_point"][i], tr.mid_point), i
        assert np.array_equal(dev["rotation"][i].view(np.uint64), tr.rotation.view(np.uint64)), i
    # a matrix per frame: focal lengths from 0.88 to 1.1 times the scaled one, principal points shifted
    Ks = np.stack([_scaled_K(w, h, 1.0 + 0.02 * (i - 6), 3.0 * (i - 6)) for i in range(n)])
    per = hp.predict_frames(frames, Ks, ctx=ctx)
    for i in range(n):
        s = hp.predict_parameter_parallel(frames[i], IntrinsicMatrix(Ks[i]), ctx=ctx)
        assert np.array_equal(per["mid_point"][i], s.mid_point), i
        assert np.array_equal(per["rotation"][i].view(np.uint64), s.rotation.view(np.uint64)), i
    for i in (0, 5, 11):
        tr = of.predict(frames[i], Ks[i], mode=oracle.MODE_SAT, keep=False)
        assert np.array_equal(per["mid_point"][i], tr.mid_point), i
        assert np.array_equal(per["rotation"][i].view(np.uint64), tr.rotation.view(np.uint64)), i
    assert not np.array_equal(per["mid_point"], dev["mid_point"])  # the matrices reached the kernels


def test_image_batches_in_two_chunks_at_1080p(ctx):
    """20 frames of 1920x1080 through the 2-D back ends: a chunk of 16 frames (the image scratch cap) and a
    ragged one of 4; every mask, raw and blurred vote image and from2d mid_point against the oracle"""
    w, h, n = 1920, 1080, 20
    cap = (256 << 20) // (8 * w * h + 8)  # image_chunk_cap: 256 MiB of u32 sums and two u16 planes per lane
    assert cap == 16 and n % cap != 0
    arr = synth.make_forest(seed=55, n_trees=4, max_depth=8)
    js = synth.forest_to_json(arr, stepwidth=7)
    hp, of = HoughPrediction.from_json(js), oracle.OracleForest.from_json(js)
    K = _scaled_K(w, h)
    frames = np.stack([synth.make_frames(1, seed=500 + i, w=w, h=h)[0] if i % 3 else _noise(w, h, 500 + i)
                       for i in range(n)])
    mask = hp.predict_mask_batch(frames, ctx=ctx)
    raw = hp.hough_image_raw_batch(frames, IntrinsicMatrix(K), ctx=ctx)
    blur, res = hp.build_hough_image_batch(frames, IntrinsicMatrix(K), ctx=ctx, from2d=True)
    only = hp.predict_parameter_from2dhough_batch(frames, IntrinsicMatrix(K), ctx=ctx)
    assert np.array_equal(only.view(np.uint8), res.view(np.uint8))
    assert np.all(res["rotation"] == 0.0)
    for i, d in enumerate(frames):
        for name, got, want in (("mask", mask[i], of.predict_mask(d)), ("raw", raw[i], of.hough_image_raw(d, K)),
                                ("blurred", blur[i], of.build_hough_image(d, K))):
            bad = np.argwhere(got != want)
            assert len(bad) == 0, "frame %d: %s differs at %d pixels, first %s" % (i, name, len(bad), bad[0].tolist())
        mid, _ = of.predict_parameter_from2dhough(d, K)
        assert np.array_equal(res["mid_point"][i].view(np.uint32), mid.view(np.uint32)), i
    assert raw[16:].max() > 0 and mask[16:].max() > 0  # the ragged chunk has content


def test_pose_pass_capped_by_the_scratch_budget(ctx):
    """4096x4096 at stride 1 with 20 trees: the per-frame scratch budget of ensure_scratch (12 GiB per lane)
    holds 6 frames, so a batch of 8 runs in passes smaller than the requested chunk.  Per-frame correctness
    at large shapes is the shape table's; here the capped passes must equal passes of one frame and
    single-frame calls."""
    w = h = 4096
    n, T, stride = 8, 20, 1
    npx, npy = _grid_patches(w, h, stride)
    assert npx == npy == 4016
    vote_box_cells = 32 ** 3
    per_frame = ((h + 1) * ((w + 4) & ~3) * 4 + npx * npy * T * 4 + npx * npy * 29 + w * h * 4 +
                 2 * vote_box_cells * 4 + 40000)
    cap = (12 << 30) // per_frame
    assert cap == 6 and cap < n
    arr = synth.make_forest(seed=56, n_trees=T, max_depth=8)
    hp = HoughPrediction.from_arrays(arr, stepwidth=stride)
    K = IntrinsicMatrix(_scaled_K(w, h))
    frames = np.stack([_noise(w, h, 700 + i) if i in (5, 7) else synth.make_frames(1, seed=700 + i, w=w, h=h)[0]
                       for i in range(n)])
    a = hp.predict_batch(frames, K, ctx=ctx)
    cnt = ctx.counters()
    assert cnt["patches"] == n * npx * npy
    assert cnt["valid_patches"] > 0 and cnt["evals"] == cnt["valid_patches"] * T
    ctx.set_chunk_frames(1)
    try:
        b = hp.predict_batch(frames, K, ctx=ctx)
    finally:
        ctx.set_chunk_frames(0)
    assert a.tobytes() == b.tobytes()
    for i in (0, 5, 7):
        s = hp.predict_parameter_parallel(frames[i], K, ctx=ctx)
        assert np.array_equal(a["mid_point"][i], s.mid_point), i
        assert np.array_equal(a["rotation"][i].view(np.uint64), s.rotation.view(np.uint64)), i
    assert np.any(a["mid_point"][[5, 7]] != 0)
