"""GPU tests of the pose-and-Hough calls (dh_predict_frames_hough and its Biwi form).  Every case runs the
fused call and, on the same context, the two existing calls it stands for: the dh_result bytes must equal
the pose call's (run at the fused call's chunks), the image and from2d bytes dh_build_hough_image_frames'
with K[i] = args[i].K, the counters the pose call's but for the 2-D back end's launches per chunk (which
pins the chunking), and the transfer info the pose call's.  Output buffers, host and device, start as
0xA5 so that an unwritten byte shows.  A few frames per case are also checked against the CPU oracle."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import oracle
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth
from depthhead_b200.api import frame_args

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


class _Images:
    """a [n,h,w] u16 destination prefilled with 0xA5 bytes, on the host or on the device"""

    def __init__(self, n, h, w, on_device):
        self.dev = None
        if on_device:
            import torch
            self.dev = torch.full((max(n, 1), h, w), 0xA5A5 - 0x10000, dtype=torch.int16, device="cuda")
            torch.cuda.synchronize()
            self.ptr, self.loc = C.c_void_p(self.dev.data_ptr()), D
        else:
            self.host = np.full((n, h, w), 0xA5A5, np.uint16)
            self.ptr, self.loc = P(self.host), H
        self.n = n

    def get(self):
        if self.dev is not None:
            import torch
            torch.cuda.synchronize()
            return self.dev.cpu().numpy().view(np.uint16)[:self.n]
        return self.host


# what the 2-D side of a case asks for: (blur, image: None / "host" / "device", from2d)
MODES = [(1, "host", True), (1, "device", True), (1, None, True), (1, "device", False), (0, "host", False), (0, "device", False)]


def _snap(ctx):
    return ctx.counters(), ctx.transfer_info()


def _default_chunk(kind):
    return 512 if kind in ("device", "biwi") else 128


def _image_cap(w, h):
    """frames per chunk of the 2-D calls (dh_ctx.cu, image_chunk_cap)"""
    return max(1, min(1 << 30, (256 << 20) // (8 * w * h + 8)))


def _calls(hp, ctx, src, n, w, h, args, chunk, mode):
    """pose call at the fused call's chunks, 2-D call and fused call at `chunk`, on the same context:
    (pose results, snap), (2-D image, from2d, snap), (fused results, image, from2d, snap)"""
    L = capi.load()
    kind, data = src
    blur, iloc, f2d = mode
    eff = min(chunk or _default_chunk(kind), _image_cap(w, h))
    Ks = np.ascontiguousarray(args["K"])
    out_p, out_f = _results_a5(n), _results_a5(n)
    img_2d = np.full((n, h, w), 0xA5A5, np.uint16) if iloc else None
    f2d_2d = _results_a5(n) if f2d else None
    img_f = _Images(n, h, w, iloc == "device") if iloc else None
    f2d_f = _results_a5(n) if f2d else None
    ip, il = (img_f.ptr, img_f.loc) if img_f else (None, H)
    if kind == "biwi":
        blob, off = data
        ctx.set_chunk_frames(eff)
        capi.check(L.dh_predict_frames_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(out_p)))
        pose = (out_p, _snap(ctx))
        ctx.set_chunk_frames(chunk)
        capi.check(L.dh_build_hough_image_frames_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(Ks), blur, P(img_2d), H, P(f2d_2d)))
        two = (img_2d, f2d_2d, _snap(ctx))
        capi.check(L.dh_predict_frames_hough_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(out_f), blur, ip, il, P(f2d_f)))
    else:
        p, loc = (P(data), H) if kind == "host" else (C.c_void_p(data), D)
        ctx.set_chunk_frames(eff)
        capi.check(L.dh_predict_frames(ctx._h, hp._h, p, n, w, h, loc, P(args), P(out_p)))
        pose = (out_p, _snap(ctx))
        ctx.set_chunk_frames(chunk)
        capi.check(L.dh_build_hough_image_frames(ctx._h, hp._h, p, n, w, h, loc, P(Ks), blur, P(img_2d), H, P(f2d_2d)))
        two = (img_2d, f2d_2d, _snap(ctx))
        capi.check(L.dh_predict_frames_hough(ctx._h, hp._h, p, n, w, h, loc, P(args), P(out_f), blur, ip, il, P(f2d_f)))
    fused = (out_f, img_f.get() if img_f else None, f2d_f, _snap(ctx))
    passes = math.ceil(n / min(eff, n)) if n else 0
    return pose, two, fused, passes


def _check(what, pose, two, fused, passes, mode, votes=1, transfer=True):
    """votes: vote launches per pass (0 for frames that hold no patch)"""
    (out_p, (cnt_p, tr_p)), (img_2d, f2d_2d, (cnt_2d, _)), (out_f, img_f, f2d_f, (cnt_f, tr_f)) = pose, two, fused
    blur, iloc, f2d = mode
    assert out_f.tobytes() == out_p.tobytes(), "%s: results differ at frames %s" % (
        what, np.argwhere((out_f.view(np.uint8).reshape(len(out_f), -1) != out_p.view(np.uint8).reshape(len(out_p), -1)).any(1)).ravel()[:8])
    if iloc:
        bad = np.argwhere(img_f != img_2d)
        assert len(bad) == 0, "%s: images differ at %d pixels, first %s" % (what, len(bad), bad[0].tolist())
        assert not (img_2d == 0xA5A5).all(axis=(1, 2)).any(), what  # (and the 2-D call wrote every frame)
    if f2d:
        assert f2d_f.tobytes() == f2d_2d.tobytes(), "%s: from2d results differ" % what
    for k in ("frames", "patches", "valid_patches", "evals", "node_visits"):  # the front end ran on the same frames
        assert cnt_2d[k] == cnt_p[k], (what, k, cnt_2d[k], cnt_p[k])
    back = votes + (2 if blur else 1) + (1 if f2d else 0)  # 2-D launches of one chunk
    for k in cnt_p:
        want = cnt_p[k] + (passes * back if k == "launches" else 0)
        got = cnt_f[k]
        if k == "launches" and not transfer:
            # the hybrid host path splits chunks between rewritten and raw by timing, and a rewritten chunk
            # has one decode launch more: compare the launches of the pipeline itself
            want -= tr_p["encoded_chunks"]
            got -= tr_f["encoded_chunks"]
        assert got == want, (what, k, cnt_p[k], cnt_f[k], passes, back, tr_p, tr_f)
    if transfer:
        assert tr_f == tr_p, (what, tr_p, tr_f)
    else:  # (the split also decides the bytes copied: only the workers are fixed)
        assert tr_f["encode_threads"] == tr_p["encode_threads"], (what, tr_p, tr_f)


def _sources(frames, kinds, offset=0, files=None):
    n, h, w = frames.shape
    keep = []
    for kind in kinds:
        if kind == "host":
            yield ("host", frames), keep
        elif kind == "device":
            # at an odd frame offset inside a larger allocation
            buf = _cuda(np.concatenate([np.zeros((offset, h, w), np.uint16), frames]).view(np.int16))
            keep.append(buf)
            yield ("device", buf.data_ptr() + offset * h * w * 2), keep
        else:
            yield ("biwi", files or biwi.pack_files([biwi.encode_depth(f) for f in frames])), keep


def _run(hp, ctx, frames, args, kinds, chunk, modes=MODES, what="", transfer=True, offset=0, votes=1, files=None):
    n, h, w = frames.shape
    for src, _keep in _sources(frames, kinds, offset, files):
        for mode in modes:
            try:
                pose, two, fused, passes = _calls(hp, ctx, src, n, w, h, args, chunk, mode)
            finally:
                ctx.set_chunk_frames(0)
            _check("%s: %s input, mode %s, chunk %d" % (what, src[0], mode, chunk), pose, two, fused, passes, mode, votes, transfer)


@pytest.fixture(scope="module")
def vga200(box):
    frames = synth.make_frames(200, seed=31)
    frames[17] = 0
    return frames, _frame_args(200), biwi.pack_files([biwi.encode_depth(f) for f in frames])


@pytest.mark.parametrize("chunk", [0, 1, 7])
def test_200_frames_24_matrices(ctx, enc_ctx, box, vga200, chunk):
    """200 VGA frames, 24 matrices, mixed seeds: host input (raw and run-length), device input at an odd
    frame offset, Biwi files; raw and blurred images to the host and to the device, with and without from2d"""
    _, hp = box
    frames, args, files = vga200
    _run(hp, ctx, frames, args, ("host", "device", "biwi"), chunk, what="raw", offset=3, files=files)
    _run(hp, enc_ctx, frames, args, ("host",), chunk, modes=MODES[:1] + MODES[4:5], what="encoded", transfer=False)
    assert enc_ctx.transfer_info()["encoded_chunks"] > 0


@pytest.mark.parametrize("n", [0, 1])
def test_batch_sizes(ctx, box, vga200, n):
    _, hp = box
    frames, args, _ = vga200
    fr = np.ascontiguousarray(frames[:n])
    a = np.ascontiguousarray(args[:n])
    if n == 0:
        out, img, f2d = hp.predict_frames_with_hough(fr, a["K"].reshape(0, 3, 3), ctx=ctx)
        assert len(out) == 0 and img.shape == (0, 480, 640) and len(f2d) == 0 and ctx.counters()["frames"] == 0
        out, img, f2d = biwi.predict_files_with_hough(hp, np.zeros(16, np.uint8), np.zeros(1, np.uint64), 640, 480, K, ctx=ctx)
        assert len(out) == 0 and ctx.counters()["frames"] == 0
        return
    _run(hp, ctx, fr, a, ("host", "device", "biwi"), 0, what="n = 1", offset=1)


@pytest.mark.parametrize("kind", ["box", "sat", "odd"])
def test_forests_and_the_oracle(kind):
    """a box-image forest (leaf words with codes), a summed-area-table forest with ragged rectangles (no
    codes), and leaf probabilities outside [0, 1]; two frames against the oracle"""
    js, hp = _forest(kind)
    c = _context(DH_HOST_ENCODE=0)
    try:
        frames = synth.make_frames(24, seed=41)
        args = _frame_args(24, n_k=6, seed=2)
        _run(hp, c, frames, args, ("host", "device"), 0, what=kind)
        _run(hp, c, frames, args, ("device",), 5, modes=MODES[1:2] + MODES[5:], what=kind)
        kw = dict(midp_guess=args["midp_guess"], rot_guess=args["rot_guess"], has_midp=(args["has_guess"] & 1) == 1,
                  has_rot=(args["has_guess"] & 2) == 2, ctx=c)
        Ks = args["K"].reshape(-1, 3, 3)
        out, img, f2d = hp.predict_frames_with_hough(frames, Ks, **kw)
        _, raw, none = hp.predict_frames_with_hough(frames, Ks, blur=False, from2d=False, **kw)
        assert none is None
        of = oracle.OracleForest.from_json(js)
        for i in (0, 7):
            assert np.array_equal(img[i], of.build_hough_image(frames[i], Ks[i])), (kind, i)
            assert np.array_equal(raw[i], of.hough_image_raw(frames[i], Ks[i])), (kind, i)
            mid, _ = of.predict_parameter_from2dhough(frames[i], Ks[i])
            assert np.array_equal(f2d[i]["mid_point"].view(np.uint32), mid.view(np.uint32)), (kind, i)
            a = args[i]
            tr = of.predict(frames[i], Ks[i], a["midp_guess"] if a["has_guess"] & 1 else None,
                            a["rot_guess"] if a["has_guess"] & 2 else None, mode=oracle.MODE_SAT, keep=False)
            assert np.array_equal(out[i]["mid_point"].view(np.uint32), tr.mid_point.view(np.uint32)), (kind, i)
            assert np.array_equal(out[i]["rotation"].view(np.uint64), tr.rotation.view(np.uint64)), (kind, i)
        assert img[:8].max() > 0 and raw[:8].max() > 0, kind
    finally:
        c.close()


@pytest.mark.parametrize("env", [{"DH_LANES": 1}, {"timing": 1}])
def test_context_switches(box, vga200, env):
    """one lane; stage timing (single-lane; the 2-D back end is booked under DH_STAGE_VOTE)"""
    _, hp = box
    frames, args, _ = vga200
    fr, a = np.ascontiguousarray(frames[:80]), np.ascontiguousarray(args[:80])
    env = dict(env)
    timing = env.pop("timing", 0)
    c = _context(DH_HOST_ENCODE=0, **env)
    try:
        c.enable_stage_timing(bool(timing))
        for chunk in (0, 7):
            _run(hp, c, fr, a, ("host", "device"), chunk, modes=MODES[:1] + MODES[4:5], what=str(env))
        if timing:
            ms = c.stage_ms()
            assert ms["vote"] > 0 and ms["traverse"] > 0, ms
    finally:
        c.close()


@pytest.mark.parametrize("w,h,n", [(80, 80, 9), (1920, 1080, 20)])
def test_frame_sizes(ctx, box, w, h, n):
    """80x80 frames (one sub-image, no patch: no vote launch), and 1080p x 20, where the image scratch caps
    chunks at 16 frames, so the call takes two"""
    _, hp = box
    big = synth.make_frames(n, seed=47, w=max(w, 640), h=max(h, 480))
    y0, x0 = (big.shape[1] - h) // 2, (big.shape[2] - w) // 2
    frames = np.ascontiguousarray(big[:, y0:y0 + h, x0:x0 + w])
    args = _frame_args(n, n_k=3)
    _run(hp, ctx, frames, args, ("host", "device", "biwi"), 0, modes=MODES[:2] + MODES[4:5], what="%dx%d" % (w, h),
         votes=0 if w == 80 else 1)
    if w == 1920:
        assert _image_cap(w, h) == 16


def test_damaged_files_give_the_pose_calls_error(ctx, box):
    _, hp = box
    frames = synth.make_frames(12, seed=950)
    files = [biwi.encode_depth(f) for f in frames]
    Ks = _matrices(12)
    for chunk in (0, 1):
        ctx.set_chunk_frames(chunk)
        try:
            for a, b in ((3, 9), (10, 2)):
                bad = list(files)
                bad[a] = bad[a][:len(bad[a]) // 2]
                bad[b] = bad[b][:len(bad[b]) // 3]
                blob, off = biwi.pack_files(bad)
                msgs = []
                for fn in (biwi.predict_files, biwi.predict_files_with_hough):
                    with pytest.raises(capi.DhError) as e:
                        fn(hp, blob, off, 640, 480, Ks, ctx=ctx)
                    assert e.value.code == capi.DH_E_ARG
                    msgs.append(str(e.value))
                assert msgs[0] == msgs[1] and "Biwi frame %d " % min(a, b) in msgs[0], msgs
        finally:
            ctx.set_chunk_frames(0)
    blob, off = biwi.pack_files(files)
    out, img, f2d = biwi.predict_files_with_hough(hp, blob, off, 640, 480, Ks, ctx=ctx)
    assert out.tobytes() == hp.predict_frames(frames, Ks, ctx=ctx).tobytes()
    want_img, want_f2d = hp.build_hough_image_frames(frames, Ks, ctx=ctx, from2d=True)
    assert np.array_equal(img, want_img) and f2d.tobytes() == want_f2d.tobytes()


def test_argument_errors_leave_the_context_alone(ctx, box, vga200):
    """each DH_E_ARG rule on a live context: the error comes before any device work, so the counters and
    the transfer info of the call before it stay"""
    _, hp = box
    L = capi.load()
    frames, args, _ = vga200
    fr, a = np.ascontiguousarray(frames[:4]), np.ascontiguousarray(args[:4])
    blob, off = biwi.pack_files([biwi.encode_depth(f) for f in fr])
    out, img, f2d = _results_a5(4), np.zeros((4, 480, 640), np.uint16), _results_a5(4)
    hp.predict_frames(fr, a["K"].reshape(-1, 3, 3), ctx=ctx)
    before = _snap(ctx)

    def both(r=out, blur=1, i=img, iloc=H, fr2=f2d, aa=a):
        rc = (L.dh_predict_frames_hough(ctx._h, hp._h, P(fr), 4, 640, 480, H, P(aa), P(r), blur, P(i), iloc, P(fr2)),
              L.dh_predict_frames_hough_biwi(ctx._h, hp._h, P(blob), P(off), 4, 640, 480, P(aa), P(r), blur, P(i), iloc, P(fr2)))
        assert rc == (capi.DH_E_ARG, capi.DH_E_ARG), rc
        assert _snap(ctx) == before

    both(r=None)
    both(i=None, fr2=None)
    both(blur=0)
    both(blur=2)
    both(iloc=2)
    bad = a.copy()
    bad["has_guess"][2] = 4
    both(aa=bad)
    assert L.dh_predict_frames_hough(ctx._h, hp._h, P(fr), 4, 640, 480, 2, P(a), P(out), 1, P(img), H, P(f2d)) == capi.DH_E_ARG
    assert L.dh_predict_frames_hough_biwi(ctx._h, hp._h, P(blob), P(np.array([0, 8, 4, 12, 16], np.uint64)), 4, 640, 480, P(a),
                                          P(out), 1, P(img), H, P(f2d)) == capi.DH_E_ARG
    assert _snap(ctx) == before
