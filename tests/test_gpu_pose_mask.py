"""GPU tests of the pose-and-mask calls (dh_predict_frames_mask, dh_predict_tracks_mask and their Biwi forms).
Every case runs the fused call and, on the same context, the two existing calls it stands for: the
dh_result bytes must equal the pose call's, the mask bytes dh_predict_mask_batch's, the counters the pose
call's but for one more launch per pass (which pins the chunking), and the transfer info the pose call's.
Output buffers, host and device, start as 0xA5 so that an unwritten byte shows.  A few frames per case are
also checked against the CPU oracle."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth
from depthhead_b200.api import _track_offsets, frame_args

pytestmark = pytest.mark.gpu

K = IntrinsicMatrix.default_kinect_intrinsic()
P = capi.ptr
H, D = capi.DH_DEPTH_HOST, capi.DH_DEPTH_DEVICE


def _context(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def ctx():
    c = _context(DH_HOST_ENCODE=0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def enc_ctx():
    c = _context(DH_HOST_ENCODE=1)
    yield c
    c.close()


def _forest(kind, stride=10):
    if kind == "box":      # one rectangle size: box-sum image, leaf words carry probability codes
        arr = synth.make_forest(seed=3, n_trees=4, max_depth=6)
    elif kind == "sat":    # ragged rectangles: summed-area table, no codes
        arr = synth.make_forest(seed=52, n_trees=3, max_depth=7, ragged_rects=True)
    else:                  # leaf probabilities 1.5 and -0.25: codes off
        arr = synth.make_forest(seed=93, n_trees=5, max_depth=6)
        rng = np.random.default_rng(5)
        prob = np.array([1.5, -0.25, 0.0, 0.7, 0.9, 1.0])[rng.integers(0, 6, len(arr["prob"]))]
        nv = np.diff(arr["vote_off"])
        arr["prob"] = np.where((nv == 0) & (prob > 0), 0.0, prob).astype(np.float64)
    js = synth.forest_to_json(arr, stepwidth=stride)
    return js, HoughPrediction.from_json(js)


@pytest.fixture(scope="module")
def box():
    return _forest("box")


def _matrices(n):
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 480.0 + 7.5 * i
        Ks[i] = [[f, 0.0, 300.0 + 2.0 * i], [0.0, f * 1.01, 230.0 + 1.5 * i], [0.0, 0.0, 1.0]]
    Ks[n // 2] = [[561.5, 3.25, 318.0], [-2.5, 557.0, 243.5], [1.0e-4, -2.0e-4, 1.0]]
    return Ks


def _frame_args(n, n_k=24, seed=1):
    """n frames over n_k matrices, with centre seeds, rotation seeds, both and none"""
    rng = np.random.default_rng(seed)
    Ks = _matrices(n_k)[np.arange(n) % n_k]
    mid = rng.uniform(-150.0, 150.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    rot = rng.uniform(-1.0, 1.0, (n, 3))
    kind = np.arange(n) % 4
    return frame_args(n, Ks, mid, rot, (kind & 1) == 1, (kind & 2) == 2)


def _cuda(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    return t


def _results_a5(n):
    return np.frombuffer(np.full(n * capi.RESULT_DTYPE.itemsize, 0xA5, np.uint8).tobytes(), capi.RESULT_DTYPE).copy()


class _Masks:
    """a [n,h,w] u8 destination prefilled with 0xA5, on the host or on the device"""

    def __init__(self, n, h, w, on_device):
        self.dev = None
        if on_device:
            import torch
            self.dev = torch.full((max(n, 1), h, w), 0xA5, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            self.ptr, self.loc = C.c_void_p(self.dev.data_ptr()), D
        else:
            self.host = np.full((n, h, w), 0xA5, np.uint8)
            self.ptr, self.loc = P(self.host), H
        self.n = n

    def get(self):
        if self.dev is not None:
            import torch
            torch.cuda.synchronize()
            return self.dev.cpu().numpy()[:self.n]
        return self.host


def _snap(ctx):
    return ctx.counters(), ctx.transfer_info()


def _check(what, pose, fused, mask_want, passes, transfer=True):
    (out_p, (cnt_p, tr_p)), (out_f, masks, (cnt_f, tr_f)) = pose, fused
    assert out_f.tobytes() == out_p.tobytes(), "%s: results differ at frames %s" % (
        what, np.argwhere((out_f.view(np.uint8).reshape(len(out_f), -1) != out_p.view(np.uint8).reshape(len(out_p), -1)).any(1)).ravel()[:8])
    bad = np.argwhere(masks != mask_want)
    assert len(bad) == 0, "%s: masks differ at %d pixels, first %s" % (what, len(bad), bad[0].tolist())
    for k in cnt_p:
        want = cnt_p[k] + (passes if k == "launches" else 0)
        got = cnt_f[k]
        if k == "launches" and not transfer:
            # the hybrid host path splits chunks between rewritten and raw by timing, and a rewritten chunk
            # has one decode launch more: compare the launches of the pipeline itself
            want -= tr_p["encoded_chunks"]
            got -= tr_f["encoded_chunks"]
        assert got == want, (what, k, cnt_p[k], cnt_f[k], passes, tr_p, tr_f)
    if transfer:
        assert tr_f == tr_p, (what, tr_p, tr_f)
    else:  # (the split also decides the bytes copied: only the workers are fixed)
        assert tr_f["encode_threads"] == tr_p["encode_threads"], (what, tr_p, tr_f)


# ------------------------------------------------------------------------------------------------ frames
def _frames_calls(hp, ctx, src, n, w, h, args, mask_dev):
    """(pose call: results, counters) and (fused call: results, masks, counters) on the same input.
    src: ("host", array) / ("device", tensor) / ("biwi", (blob, offsets))"""
    L = capi.load()
    kind, data = src
    out_p, out_f = _results_a5(n), _results_a5(n)
    masks = _Masks(n, h, w, mask_dev)
    if kind == "biwi":
        blob, off = data
        capi.check(L.dh_predict_frames_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(out_p)))
        pose = (out_p, _snap(ctx))
        capi.check(L.dh_predict_frames_mask_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(out_f), masks.ptr, masks.loc))
    else:
        p, loc = (P(data), H) if kind == "host" else (C.c_void_p(data), D)
        capi.check(L.dh_predict_frames(ctx._h, hp._h, p, n, w, h, loc, P(args), P(out_p)))
        pose = (out_p, _snap(ctx))
        capi.check(L.dh_predict_frames_mask(ctx._h, hp._h, p, n, w, h, loc, P(args), P(out_f), masks.ptr, masks.loc))
    return pose, (out_f, masks.get(), _snap(ctx))


def _passes(n, chunk, kind):
    c = chunk or (512 if kind in ("device", "biwi") else 128)
    return math.ceil(n / min(c, max(n, 1))) if n else 0


def _run_frames(hp, ctx, frames, args, sources, mask_locs, chunk, mask_want=None, what="", transfer=True, offset=0, per_pass=1):
    """per_pass: mask launches per pass (0 for frames that hold no patch: the masks are a memset)"""
    n, h, w = frames.shape
    if mask_want is None:
        mask_want = hp.predict_mask_batch(frames, ctx=ctx)
    for kind in sources:
        if kind == "host":
            src = ("host", frames)
        elif kind == "device":
            # at an odd frame offset inside a larger allocation
            buf = _cuda(np.concatenate([np.zeros((offset, h, w), np.uint16), frames]).view(np.int16))
            src = ("device", buf.data_ptr() + offset * h * w * 2)
        else:
            src = ("biwi", biwi.pack_files([biwi.encode_depth(f) for f in frames]))
        for mdev in mask_locs:
            ctx.set_chunk_frames(chunk)
            try:
                pose, fused = _frames_calls(hp, ctx, src, n, w, h, args, mdev)
            finally:
                ctx.set_chunk_frames(0)
            _check("%s: %s input, masks to %s, chunk %d" % (what, kind, "device" if mdev else "host", chunk), pose, fused,
                   mask_want, per_pass * _passes(n, chunk, kind), transfer)
    return mask_want


@pytest.fixture(scope="module")
def vga200(box):
    _, hp = box
    frames = synth.make_frames(200, seed=31)
    frames[17] = 0
    return frames, _frame_args(200)


@pytest.mark.parametrize("chunk", [0, 1, 7, 64, 130])
def test_200_frames_24_matrices(ctx, enc_ctx, box, vga200, chunk):
    """200 VGA frames, 24 matrices, mixed seeds: host input (raw and run-length), device input at an odd
    frame offset, Biwi files; masks to the host and to the device"""
    _, hp = box
    frames, args = vga200
    want = _run_frames(hp, ctx, frames, args, ("host", "device", "biwi"), (False, True), chunk, what="raw", offset=3)
    assert want.max() > 0 and (want == 0).any()
    _run_frames(hp, enc_ctx, frames, args, ("host",), (False, True), chunk, mask_want=want, what="encoded", transfer=False)
    assert enc_ctx.transfer_info()["encoded_chunks"] > 0


@pytest.mark.parametrize("n", [0, 1, 63, 64, 65])
def test_batch_sizes(ctx, box, vga200, n):
    _, hp = box
    frames, args = vga200
    fr = np.ascontiguousarray(frames[:n])
    a = np.ascontiguousarray(args[:n])
    if n == 0:
        out, masks = hp.predict_frames_with_mask(fr, a["K"].reshape(0, 3, 3), ctx=ctx)
        assert len(out) == 0 and masks.shape == (0, 480, 640) and ctx.counters()["frames"] == 0
        return
    _run_frames(hp, ctx, fr, a, ("host", "device"), (False, True), 0, what="n = %d" % n, offset=1)


@pytest.mark.parametrize("kind,env", [("box", {}), ("sat", {}), ("box", {"DH_PROB_CODES": 0}), ("odd", {})])
def test_forests_and_the_oracle(kind, env):
    """a box-image forest (leaf words with codes), a summed-area-table forest with ragged rectangles (no
    codes), DH_PROB_CODES=0, and leaf probabilities 1.5 and -0.25; two frames against the oracle"""
    js, hp = _forest(kind)
    c = _context(DH_HOST_ENCODE=0, **env)
    try:
        frames = synth.make_frames(24, seed=41)
        args = _frame_args(24, n_k=6, seed=2)
        want = _run_frames(hp, c, frames, args, ("host", "device"), (False, True), 0, what=kind + str(env))
        _run_frames(hp, c, frames, args, ("device",), (True,), 5, mask_want=want, what=kind + str(env))
        out, masks = hp.predict_frames_with_mask(frames, args["K"].reshape(-1, 3, 3), args["midp_guess"], args["rot_guess"],
                                                 (args["has_guess"] & 1) == 1, (args["has_guess"] & 2) == 2, ctx=c)
        of = oracle.OracleForest.from_json(js)
        for i in (0, 7):
            assert np.array_equal(masks[i], of.predict_mask(frames[i])), (kind, i)
            a = args[i]
            tr = of.predict(frames[i], a["K"].reshape(3, 3), a["midp_guess"] if a["has_guess"] & 1 else None,
                            a["rot_guess"] if a["has_guess"] & 2 else None, mode=oracle.MODE_SAT, keep=False)
            assert np.array_equal(out[i]["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32)), (kind, i)
            assert np.array_equal(out[i]["rotation"].view(np.uint64), tr.rotation.view(np.uint64)), (kind, i)
    finally:
        c.close()


@pytest.mark.parametrize("env", [{"DH_GATE_SPLIT_MIN": 1}, {"DH_GATE_SPLIT_MIN": 64}, {"DH_LANES": 1}, {"DH_LANES": 2}, {"timing": 1}])
def test_context_switches(box, vga200, env):
    """gate split at 1 and 64 (80 frames in one pass take the gated lists, in passes of 7 the folded gate),
    one and two lanes, stage timing (single-lane; the mask is booked under DH_STAGE_VOTE)"""
    _, hp = box
    frames, args = vga200
    fr, a = np.ascontiguousarray(frames[:80]), np.ascontiguousarray(args[:80])
    env = dict(env)
    timing = env.pop("timing", 0)
    c = _context(DH_HOST_ENCODE=0, **env)
    try:
        c.enable_stage_timing(bool(timing))
        want = None
        for chunk in (0, 7):
            want = _run_frames(hp, c, fr, a, ("host", "device"), (False, True), chunk, mask_want=want, what=str(env))
        if timing:
            ms = c.stage_ms()
            assert ms["vote"] > 0 and ms["traverse"] > 0, ms
    finally:
        c.close()


@pytest.mark.parametrize("stride", [5, 10, 7])
def test_strides_and_stepwidth_changes(ctx, stride):
    js, hp = _forest("box", stride=10)
    frames = synth.make_frames(12, seed=43)
    args = _frame_args(12, n_k=4)
    hp.stepwidth = stride
    _run_frames(hp, ctx, frames, args, ("host", "device"), (False, True), 5, what="stride %d" % stride)
    if stride == 7:
        of = oracle.OracleForest.from_json(js)
        of.stepwidth = 7
        _, masks = hp.predict_frames_with_mask(frames[:1], K, ctx=ctx)
        assert np.array_equal(masks[0], of.predict_mask(frames[0]))
    hp.stepwidth = 10  # and back, on the same context
    _run_frames(hp, ctx, frames, args, ("device",), (True,), 0, what="stride back to 10")


@pytest.mark.parametrize("w,h,n", [(80, 80, 9), (1280, 720, 12), (1920, 1080, 20)])
def test_frame_sizes(ctx, box, w, h, n):
    """80x80 frames (one sub-image, no patch), 720p, and 1080p x 20, where the 2-D calls cap chunks at 16
    frames and the fused call keeps one pass of 20"""
    _, hp = box
    big = synth.make_frames(n, seed=47, w=max(w, 640), h=max(h, 480))
    y0, x0 = (big.shape[1] - h) // 2, (big.shape[2] - w) // 2
    frames = np.ascontiguousarray(big[:, y0:y0 + h, x0:x0 + w])
    args = _frame_args(n, n_k=3)
    want = _run_frames(hp, ctx, frames, args, ("host", "device", "biwi"), (False, True), 0, what="%dx%d" % (w, h),
                       per_pass=0 if w == 80 else 1)
    assert (want.max() == 0) == (w == 80)


# ------------------------------------------------------------------------------------------------ tracks
LENGTHS = [0, 1, 2, 63, 64, 65, 300, 5]


def _n_passes(lengths, chunk):
    """passes of the slot plan of predict_tracks (dh_ctx.cu, plan_tracks)"""
    live = [s for s in range(len(lengths)) if lengths[s]]
    F = min(chunk, len(live)) if chunk else min(len(live), 512)
    order = sorted(live, key=lambda s: -lengths[s])
    slots = [[order[i], 0] for i in range(min(F, len(order)))]
    nxt, passes = len(slots), 0
    while any(s[0] is not None for s in slots):
        passes += 1
        for s in slots:
            if s[0] is None:
                continue
            s[1] += 1
            if s[1] >= lengths[s[0]]:
                s[0], s[1] = (order[nxt], 0) if nxt < len(order) else (None, 0)
                nxt += 1
    return passes


def _tracks_calls(hp, ctx, src, lengths, w, h, args, mask_dev, min_z=500.0):
    L = capi.load()
    seq_off, n_seq, total = _track_offsets(lengths)
    kind, data = src
    out_p, out_f = _results_a5(total), _results_a5(total)
    masks = _Masks(total, h, w, mask_dev)
    if kind == "biwi":
        blob, off = data
        capi.check(L.dh_predict_tracks_biwi(ctx._h, hp._h, P(blob), P(off), n_seq, P(seq_off), w, h, P(args), min_z, P(out_p)))
        pose = (out_p, _snap(ctx))
        capi.check(L.dh_predict_tracks_mask_biwi(ctx._h, hp._h, P(blob), P(off), n_seq, P(seq_off), w, h, P(args), min_z, P(out_f),
                                                 masks.ptr, masks.loc))
    else:
        p, loc = (P(data), H) if kind == "host" else (C.c_void_p(data), D)
        capi.check(L.dh_predict_tracks(ctx._h, hp._h, p, n_seq, P(seq_off), w, h, loc, P(args), min_z, P(out_p)))
        pose = (out_p, _snap(ctx))
        capi.check(L.dh_predict_tracks_mask(ctx._h, hp._h, p, n_seq, P(seq_off), w, h, loc, P(args), min_z, P(out_f), masks.ptr, masks.loc))
    return pose, (out_f, masks.get(), _snap(ctx))


def _track_frames(lengths, seed):
    parts = [synth.make_frames(n, seed=seed + s, sequence=True, start_index=700 * s) for s, n in enumerate(lengths) if n]
    frames = np.ascontiguousarray(np.concatenate(parts))
    off = np.concatenate([[0], np.cumsum(lengths)])
    longest = int(np.argmax(lengths))
    frames[off[longest] + 1] = 0
    return frames


@pytest.fixture(scope="module")
def tracks(ctx, box):
    _, hp = box
    n = len(LENGTHS)
    frames = _track_frames(LENGTHS, 800)
    rng = np.random.default_rng(3)
    mid = rng.uniform(-200.0, 200.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    kind = np.array([3, 1, 2, 0, 2, 1, 3, 0])[np.arange(n) % 8]
    args = frame_args(n, _matrices(n), mid, rng.uniform(-1.0, 1.0, (n, 3)), (kind & 1) == 1, (kind & 2) == 2)
    masks = hp.predict_mask_batch(frames, ctx=ctx)
    dev = _cuda(frames.view(np.int16))
    files = biwi.pack_files([biwi.encode_depth(f) for f in frames])
    return frames, args, masks, dev, files


@pytest.mark.parametrize("chunk", [0, 1, 2, 4, 64])
def test_tracks_of_any_length(ctx, box, tracks, chunk):
    """tracks of 0 .. 300 frames, each with its own K and first seeds; host, device and Biwi input; masks
    to the host (several windows of the mask staging at every chunk) and to the device"""
    _, hp = box
    frames, args, want, dev, files = tracks
    for kind, data in (("host", frames), ("device", dev.data_ptr()), ("biwi", files)):
        for mdev in (False, True):
            ctx.set_chunk_frames(chunk)
            try:
                pose, fused = _tracks_calls(hp, ctx, (kind, data), LENGTHS, 640, 480, args, mdev)
            finally:
                ctx.set_chunk_frames(0)
            _check("tracks: %s input, masks to %s, chunk %d" % (kind, "device" if mdev else "host", chunk), pose, fused, want,
                   _n_passes(LENGTHS, chunk))


def test_track_frames_against_the_oracle(ctx, box, tracks):
    js, hp = box
    frames, args, _, _, _ = tracks
    out, masks = hp.predict_tracks_with_mask(frames, LENGTHS, args["K"].reshape(-1, 3, 3), args["midp_guess"], args["rot_guess"],
                                             (args["has_guess"] & 1) == 1, (args["has_guess"] & 2) == 2, ctx=ctx)
    of = oracle.OracleForest.from_json(js)
    for i in (0, 200, len(frames) - 1):
        assert np.array_equal(masks[i], of.predict_mask(frames[i])), i
    # the first frame of a seeded track: the oracle with the track's seeds
    s = 3
    f0 = int(np.sum(LENGTHS[:s]))
    a = args[s]
    tr = of.predict(frames[f0], a["K"].reshape(3, 3), a["midp_guess"] if a["has_guess"] & 1 else None,
                    a["rot_guess"] if a["has_guess"] & 2 else None, mode=oracle.MODE_SAT, keep=False)
    assert np.array_equal(out[f0]["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32))
    assert np.array_equal(out[f0]["rotation"].view(np.uint64), tr.rotation.view(np.uint64))


@pytest.mark.parametrize("chunk", [0, 3])
def test_uniform_tracks_equal_predict_sequences(ctx, box, chunk):
    """equal lengths, one K, no seeds: the operations of dh_predict_sequences plus one mask launch per pass"""
    _, hp = box
    n_seq, T = 5, 6
    frames = np.ascontiguousarray(_track_frames([T] * n_seq, 500))
    want_masks = hp.predict_mask_batch(frames, ctx=ctx)
    dev = _cuda(frames.view(np.int16))
    ctx.set_chunk_frames(chunk)
    try:
        for where in ("host", "device"):
            seq_src = dict(device_ptr=dev.data_ptr(), n_seq=n_seq, frames_per_seq=T, w=640, h=480) if where == "device" else {}
            seq = hp.predict_sequences(None if seq_src else frames.reshape(n_seq, T, 480, 640), K, ctx=ctx, **seq_src)
            cnt_seq = ctx.counters()
            data = dev.data_ptr() if where == "device" else frames
            for mdev in (False, True):
                pose, fused = _tracks_calls(hp, ctx, (where, data), [T] * n_seq, 640, 480, frame_args(n_seq, K), mdev)
                assert pose[1][0] == cnt_seq
                assert fused[0].tobytes() == np.ascontiguousarray(seq.reshape(-1)).tobytes()
                passes = T * math.ceil(n_seq / (chunk or n_seq))
                _check("uniform, %s, chunk %d" % (where, chunk), pose, fused, want_masks, passes)
    finally:
        ctx.set_chunk_frames(0)


@pytest.mark.parametrize("chunk", [0, 1])
def test_damaged_files_give_the_pose_calls_error(ctx, box, chunk):
    _, hp = box
    lengths = [3, 9, 2]
    frames = _track_frames(lengths, 950)
    files = [biwi.encode_depth(f) for f in frames]
    args = frame_args(3, _matrices(3))
    ctx.set_chunk_frames(chunk)
    try:
        for short, longest in ((1, 3 + 6), (12 + 1, 3 + 1)):
            bad = list(files)
            bad[short] = bad[short][:len(bad[short]) // 2]
            bad[longest] = bad[longest][:len(bad[longest]) // 3]
            blob, off = biwi.pack_files(bad)
            msgs = []
            for fn in (biwi.predict_track_files, biwi.predict_track_files_with_mask):
                with pytest.raises(capi.DhError) as e:
                    fn(hp, blob, off, lengths, 640, 480, args["K"].reshape(-1, 3, 3), ctx=ctx)
                assert e.value.code == capi.DH_E_ARG
                msgs.append(str(e.value))
            assert msgs[0] == msgs[1] and "Biwi frame %d " % min(short, longest) in msgs[0], msgs
            # the frames form
            with pytest.raises(capi.DhError) as e:
                biwi.predict_files_with_mask(hp, blob, off, 640, 480, K, ctx=ctx)
            with pytest.raises(capi.DhError) as e2:
                biwi.predict_files(hp, blob, off, 640, 480, np.tile(K.mat, (len(frames), 1, 1)), ctx=ctx)
            assert str(e.value) == str(e2.value)
        blob, off = biwi.pack_files(files)
        out, masks = biwi.predict_track_files_with_mask(hp, blob, off, lengths, 640, 480, args["K"].reshape(-1, 3, 3), ctx=ctx)
        assert out.tobytes() == hp.predict_tracks(frames, lengths, args["K"].reshape(-1, 3, 3), ctx=ctx).tobytes()
        assert np.array_equal(masks, hp.predict_mask_batch(frames, ctx=ctx))
    finally:
        ctx.set_chunk_frames(0)


def test_empty_calls(ctx, box):
    _, hp = box
    out, masks = hp.predict_tracks_with_mask(np.zeros((0, 480, 640), np.uint16), [0, 0], K, ctx=ctx)
    assert len(out) == 0 and masks.shape == (0, 480, 640) and ctx.counters()["frames"] == 0
    out, masks = biwi.predict_files_with_mask(hp, np.zeros(16, np.uint8), np.zeros(1, np.uint64), 640, 480, K, ctx=ctx)
    assert len(out) == 0 and ctx.counters()["frames"] == 0
