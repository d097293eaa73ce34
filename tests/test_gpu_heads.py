"""GPU tests of dh_predict_frames_heads (DESIGN.md §7 "Several heads per frame"): head 0 against
dh_predict_frames byte for byte, every head and its count against the CPU oracle's orc_predict_heads bit
for bit (both patch-gate paths, a synthetic and a trained forest, mixed intrinsics and caller seeds, tries
whose mean-shift leaves its cube), heads found on two-person frames, and results that do not depend on the
input path or the chunking."""
import os

import numpy as np
import pytest

from oracle import heads as heads_oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth, train
from depthhead_b200.api import DEFAULT_MIN_CELL_VOTES

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def trained(ctx):
    """the forest dh_train_learn grows from one-person synthetic frames (as test_gpu_frame_args' model)"""
    tf, tc, tr_, tm = synth.make_frames(40, seed=101, with_truth=True)
    data = [dict(depth=tf[i], mask=tm[i], intrinsic=K, pos3d=tc[i], rot=tr_[i]) for i in range(len(tf))]
    js = train.HoughLearning(10, 80, 80, 8, 4, 1200, 0.3, 150, 20, 5.0).learn_native(8.0, data, seed=7, ctx=ctx).to_json()
    return js, HoughPrediction.from_json(js)


@pytest.fixture(scope="module")
def synthetic():
    js = synth.forest_to_json(synth.make_forest(seed=0), stepwidth=10)
    return js, HoughPrediction.from_json(js)


def _matrices(n):
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 520.0 + 5.5 * (i % 13)
        Ks[i] = [[f, 0.0, 310.0 + (i % 7)], [0.0, f * 1.01, 236.0 + 0.5 * (i % 5)], [0.0, 0.0, 1.0]]
    return Ks


def _seeds(n, rng):
    """(None, None), centre only, rotation only and both, by frame"""
    mid = rng.uniform(-200.0, 200.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    rot = rng.uniform(-1.0, 1.0, (n, 3))
    kind = np.arange(n) % 4
    return mid, rot, (kind & 1) == 1, (kind & 2) == 2


def _same(a, b):
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


@pytest.mark.parametrize("max_heads", [1, 2, 4, 8])
def test_head0_is_predict_frames(ctx, trained, max_heads):
    _, hp = trained
    frames, _, _ = synth.make_person_frames(70, seed=3)
    Ks = _matrices(70)
    mid, rot, hm, hr = _seeds(70, np.random.default_rng(1))
    want = hp.predict_frames(frames, Ks, mid, rot, hm, hr, ctx=ctx)
    heads, n_heads = hp.predict_frames_heads(frames, Ks, mid, rot, hm, hr, max_heads=max_heads, min_cell_votes=1, ctx=ctx)
    assert heads.shape == (70, max_heads) and _same(heads[:, 0]["pose"], want)
    assert np.all((n_heads >= 1) & (n_heads <= max_heads))
    for i in range(70):
        assert not heads[i, n_heads[i]:].tobytes().strip(b"\0"), i
    if max_heads > 1:
        assert (n_heads > 1).any()


def _oracle_heads(js, frames, Ks, mid, rot, hm, hr, max_heads, votes, radius):
    of = heads_oracle.HeadsForest.from_json(js)
    out = []
    for i in range(len(frames)):
        out.append(of.predict_heads(frames[i], Ks[i], max_heads, votes, radius, midp_guess=mid[i] if hm[i] else None,
                                    rot_guess=rot[i] if hr[i] else None))
    return out


def _compare(heads, n_heads, want, what):
    moved = 0
    for i, (oh, on, tries) in enumerate(want):
        assert int(n_heads[i]) == on, (what, i, int(n_heads[i]), on, tries)
        g = heads[i]
        for k in range(on):
            assert _same(g[k]["pose"]["mid_point"], oh[k]["mid_point"]), (what, i, k, g[k], oh[k])
            assert _same(g[k]["pose"]["rotation"], oh[k]["rotation"]), (what, i, k, g[k], oh[k])
            assert (int(g[k]["support"]), int(g[k]["n_patches"]), int(g[k]["seed_cell"])) == \
                (int(oh[k]["support"]), int(oh[k]["n_patches"]), int(oh[k]["seed_cell"])), (what, i, k, g[k], oh[k])
        assert not g[on:].tobytes().strip(b"\0"), (what, i)
        # tries whose centre ended more than the cube's 6 cells of margin from its seed had to rebuild their cube
        moved += sum(int(np.abs(t["centre"] - t["seed"]).max() > 6) for t in tries[1:])
    return moved


@pytest.mark.parametrize("forest", ["synthetic", "trained"])
@pytest.mark.parametrize("n", [12, 70])  # one-kernel patch gate below 64 frames a pass, the gated-patch lists from 64
def test_every_head_matches_the_oracle(ctx, request, forest, n):
    js, hp = request.getfixturevalue(forest)
    frames, _, _ = synth.make_person_frames(n, seed=11 + n)
    Ks = _matrices(n)
    mid, rot, hm, hr = _seeds(n, np.random.default_rng(n))
    votes = 1 if forest == "synthetic" else DEFAULT_MIN_CELL_VOTES // 4
    heads, n_heads = hp.predict_frames_heads(frames, Ks, mid, rot, hm, hr, max_heads=4, min_cell_votes=votes, ctx=ctx)
    want = _oracle_heads(js, frames, Ks, mid, rot, hm, hr, 4, votes, 150.0)
    moved = _compare(heads, n_heads, want, "%s, %d frames" % (forest, n))
    assert (n_heads > 1).any()
    if forest == "synthetic" and n == 70:
        assert moved > 0, "no try left its cube"


def test_radius_and_max_heads_against_the_oracle(ctx, synthetic):
    js, hp = synthetic
    frames, _, _ = synth.make_person_frames(20, seed=77, persons=3)
    Ks = np.tile(synth.KINECT_K, (20, 1, 1))
    none = np.zeros(20, bool)
    z3, z = np.zeros((20, 3), np.float32), np.zeros((20, 3))
    for max_heads, radius in ((8, 80.0), (3, 260.5), (2, 1000.0)):
        heads, n_heads = hp.predict_frames_heads(frames, Ks, max_heads=max_heads, radius_mm=radius, min_cell_votes=1, ctx=ctx)
        _compare(heads, n_heads, _oracle_heads(js, frames, Ks, z3, z, none, none, max_heads, 1, radius), (max_heads, radius))


def test_heads_are_found(ctx, trained):
    """the trained forest with the defaults: one head on one-person frames, two heads near the two true
    centres on two-person frames (lateral within 80 mm, depth between 150 mm in front of the centre and
    30 mm behind it: the reference's seed lies on the surface, DESIGN.md §7) in at least 20 of 24 frames"""
    _, hp = trained
    one = synth.make_frames(24, seed=999)
    _, n1 = hp.predict_frames_heads(one, K, ctx=ctx)
    assert np.all(n1 == 1), n1
    two, centres, _ = synth.make_person_frames(24, seed=5, persons=2)
    heads, n2 = hp.predict_frames_heads(two, K, ctx=ctx)
    good = 0
    for i in range(24):
        got = heads[i, :n2[i]]["pose"]["mid_point"].astype(np.float64)
        ok = 0
        for c in centres[i, :2]:
            d = got - c
            ok += bool(np.any((np.hypot(d[:, 0], d[:, 1]) < 80.0) & (d[:, 2] > -150.0) & (d[:, 2] < 30.0)))
        good += int(n2[i] == 2 and ok == 2)
    assert good >= 20, (good, n2, heads[:, :2]["pose"]["mid_point"], centres[:, :2])


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


def test_input_path_and_chunking_do_not_change_results(ctx, synthetic):
    import torch
    _, hp = synthetic
    n = 600  # more than one chunk of device frames (512)
    frames, _, _ = synth.make_person_frames(n, seed=21)
    Ks = _matrices(n)
    mid, rot, hm, hr = _seeds(n, np.random.default_rng(4))
    want, wn = hp.predict_frames_heads(frames, Ks, mid, rot, hm, hr, max_heads=4, min_cell_votes=1, ctx=ctx)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    got, gn = hp.predict_frames_heads(None, Ks, mid, rot, hm, hr, max_heads=4, min_cell_votes=1, ctx=ctx, device_ptr=dev.data_ptr(),
                                      n=n, w=640, h=480)
    assert _same(got, want) and np.array_equal(gn, wn), "device frames"
    enc = _encode_context()
    try:
        for c, chunk in ((ctx, 7), (ctx, 64), (enc, 0), (enc, 50)):
            c.set_chunk_frames(chunk)
            try:
                got, gn = hp.predict_frames_heads(frames[:130], Ks[:130], mid[:130], rot[:130], hm[:130], hr[:130], max_heads=4,
                                                  min_cell_votes=1, ctx=c)
            finally:
                c.set_chunk_frames(0)
            assert _same(got, want[:130]) and np.array_equal(gn, wn[:130]), ("chunk", chunk)
        assert enc.transfer_info()["encoded_chunks"] > 0
    finally:
        enc.close()
    # n = 0 is a no-op
    h0, n0 = hp.predict_frames_heads(np.zeros((0, 480, 640), np.uint16), np.zeros((0, 3, 3), np.float32), ctx=ctx)
    assert h0.shape == (0, 4) and n0.shape == (0,)


def test_argument_errors_on_a_live_context(ctx, synthetic):
    _, hp = synthetic
    frames = synth.make_frames(2, seed=1)
    for kw, msg in ((dict(max_heads=9), "max_heads"), (dict(radius_mm=float("nan")), "radius_mm"), (dict(min_cell_votes=0), "min_cell_votes")):
        with pytest.raises(capi.DhError, match=msg):
            hp.predict_frames_heads(frames, K, ctx=ctx, **kw)
    heads, n_heads = hp.predict_frames_heads(frames, K, ctx=ctx)  # the context still works
    assert _same(heads[:, 0]["pose"], hp.predict_frames(frames, K, ctx=ctx))
