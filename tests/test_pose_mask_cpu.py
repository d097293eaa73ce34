"""CPU tests of the pose-and-mask calls (dh_predict_frames_mask, dh_predict_tracks_mask and their Biwi
forms): the signatures, the argument errors returned before any device work, and the dtype / shape /
length checks of the Python wrappers."""
import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi
from depthhead_b200.api import frame_args

K = IntrinsicMatrix.default_kinect_intrinsic()
H, D = capi.DH_DEPTH_HOST, capi.DH_DEPTH_DEVICE


def test_signatures():
    L = capi.load()
    for name, n_args in (("dh_predict_frames_mask", 11), ("dh_predict_frames_mask_biwi", 11),
                         ("dh_predict_tracks_mask", 13), ("dh_predict_tracks_mask_biwi", 13)):
        assert hasattr(L, name) and len(capi.SIGNATURES[name][1]) == n_args, name
    # the pose calls' arguments, then mask and mask_loc
    assert capi.SIGNATURES["dh_predict_frames_mask"][1][:9] == capi.SIGNATURES["dh_predict_frames"][1]
    assert capi.SIGNATURES["dh_predict_frames_mask_biwi"][1][:9] == capi.SIGNATURES["dh_predict_frames_biwi"][1]
    assert capi.SIGNATURES["dh_predict_tracks_mask"][1][:11] == capi.SIGNATURES["dh_predict_tracks"][1]
    assert capi.SIGNATURES["dh_predict_tracks_mask_biwi"][1][:11] == capi.SIGNATURES["dh_predict_tracks_biwi"][1]


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_frames_argument_errors(small_case):
    """every error below is returned with a NULL context: nothing reached a device"""
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    P = capi.ptr
    depth = np.zeros((3, 80, 80), np.uint16)
    res = np.zeros(3, capi.RESULT_DTYPE)
    mask = np.zeros((3, 80, 80), np.uint8)
    args = frame_args(3, K)
    blob, boff = np.zeros(64, np.uint8), np.array([0, 16, 32, 48], np.uint64)
    call, cbiwi = L.dh_predict_frames_mask, L.dh_predict_frames_mask_biwi

    def both(a=args, r=res, m=mask, mloc=H, ctx=None, f=hp._h, d=depth, b=blob, bo=boff, n=3):
        return (_err(call(ctx, f, P(d), n, 80, 80, H, P(a), P(r), P(m), mloc)),
                _err(cbiwi(ctx, f, P(b), P(bo), n, 80, 80, P(a), P(r), P(m), mloc)))

    for msg in both():
        assert "NULL argument" in msg, msg
    for msg in both(f=None):
        assert "NULL argument" in msg, msg
    for msg in both(a=None):
        assert "NULL argument" in msg, msg
    for msg in both(d=None, b=None):
        assert "NULL argument" in msg, msg
    assert "NULL argument" in _err(cbiwi(None, hp._h, P(blob), None, 3, 80, 80, P(args), P(res), P(mask), H))
    for msg in both(m=None):
        assert "NULL mask" in msg, msg
    for msg in both(r=None):
        assert "NULL out" in msg, msg
    for bad in (2, -1):
        for msg in both(mloc=bad):
            assert "mask_loc" in msg, msg
        assert "depth_loc" in _err(call(None, hp._h, P(depth), 3, 80, 80, bad, P(args), P(res), P(mask), H))
    for bad in (4, 0x80000000):
        a = frame_args(3, K)
        a["has_guess"][1] = bad
        for msg in both(a=a):
            assert "frame 1" in msg and "has_guess" in msg, msg
    # the Biwi offset checks of dh_predict_batch_biwi, before any device work
    bo = np.array([0, 8, 4, 12], np.uint64)
    assert "Biwi offsets are not monotone at frame 1" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, 80, 80, P(args), P(res),
                                                                      P(mask), H))
    bo = np.array([0, 8, 10, 12], np.uint64)
    assert "Biwi frame 2" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, 80, 80, P(args), P(res), P(mask), H))
    # n = 0 needs no outputs, but still a context and a forest
    for msg in both(r=None, m=None, d=None, b=None, n=0):
        assert "NULL argument" in msg, msg


def test_tracks_argument_errors(small_case):
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    P = capi.ptr
    depth = np.zeros((6, 80, 80), np.uint16)
    res = np.zeros(6, capi.RESULT_DTYPE)
    mask = np.zeros((6, 80, 80), np.uint8)
    off = np.array([0, 2, 2, 6], np.uint64)
    args = frame_args(3, K)
    blob, boff = np.zeros(128, np.uint8), np.arange(7, dtype=np.uint64) * 16
    call, cbiwi = L.dh_predict_tracks_mask, L.dh_predict_tracks_mask_biwi

    def both(seq_off=off, a=args, r=res, m=mask, mloc=H, ctx=None, f=hp._h, d=depth, b=blob, bo=boff):
        return (_err(call(ctx, f, P(d), 3, P(seq_off), 80, 80, H, P(a), 500.0, P(r), P(m), mloc)),
                _err(cbiwi(ctx, f, P(b), P(bo), 3, P(seq_off), 80, 80, P(a), 500.0, P(r), P(m), mloc)))

    for kw in (dict(), dict(f=None), dict(seq_off=None), dict(a=None), dict(d=None, b=None)):
        for msg in both(**kw):
            assert "NULL argument" in msg, (kw, msg)
    for msg in both(m=None):
        assert "NULL mask" in msg, msg
    for msg in both(r=None):
        assert "NULL out" in msg, msg
    for bad in (2, -1):
        for msg in both(mloc=bad):
            assert "mask_loc" in msg, msg
        assert "depth_loc" in _err(call(None, hp._h, P(depth), 3, P(off), 80, 80, bad, P(args), 500.0, P(res), P(mask), D))
    for bad, what in ((np.array([1, 2, 2, 6], np.uint64), "seq_off[0]"), (np.array([0, 3, 2, 6], np.uint64), "track 1"),
                      (np.array([0, 2, 2, 1 << 31], np.uint64), "2^31")):
        for msg in both(seq_off=bad):
            assert what in msg, msg
    a = frame_args(3, K)
    a["has_guess"][2] = 8
    for msg in both(a=a):
        assert "track 2" in msg and "has_guess" in msg, msg
    bo = np.array([0, 16, 8, 48, 64, 80, 96], np.uint64)
    assert "Biwi offsets are not monotone at frame 1" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, P(off), 80, 80, P(args), 500.0,
                                                                      P(res), P(mask), H))
    bo = np.array([0, 16, 32, 48, 66, 80, 96], np.uint64)
    assert "Biwi frame 4" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, P(off), 80, 80, P(args), 500.0, P(res), P(mask), H))
    # total = 0 needs no outputs
    zero = np.zeros(4, np.uint64)
    for msg in both(seq_off=zero, r=None, m=None, d=None, b=None):
        assert "NULL argument" in msg, msg


@pytest.mark.parametrize("kw", [
    dict(intrinsics=np.zeros((2, 3, 3), np.float32)),                     # 3 frames, 2 matrices
    dict(intrinsics=np.zeros((3, 3, 3), np.float64)),
    dict(midp_guess=np.zeros((3, 3), np.float64)),
    dict(rot_guess=np.zeros((2, 3), np.float64)),
    dict(has_midp=np.ones(3, bool)),                                      # a mask without its guesses
])
def test_frames_wrappers_reject_shapes_and_dtypes(small_case, kw):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    kw = dict(kw)
    intr = kw.pop("intrinsics", K)
    with pytest.raises(ValueError):
        hp.predict_frames_with_mask(np.zeros((3, 80, 80), np.uint16), intr, **kw)
    blob, off = np.zeros(64, np.uint8), np.zeros(4, np.uint64)
    with pytest.raises(ValueError):
        biwi.predict_files_with_mask(hp, blob, off, 80, 80, intr, **kw)


@pytest.mark.parametrize("kw", [
    dict(lengths=[2, 2]),                                                 # 4 frames for 6
    dict(lengths=[3, 4]),
    dict(lengths=[3, -3, 6]),
    dict(intrinsics=np.zeros((3, 3, 3), np.float32)),                     # 2 tracks, 3 matrices
    dict(rot_guess=np.zeros((6, 3), np.float64)),                         # one seed per frame, not per track
    dict(has_midp=np.ones(2, bool)),
])
def test_tracks_wrappers_reject_shapes_and_dtypes(small_case, kw):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    kw = dict(kw)
    lengths = kw.pop("lengths", [2, 4])
    intr = kw.pop("intrinsics", K)
    with pytest.raises(ValueError):
        hp.predict_tracks_with_mask(np.zeros((6, 80, 80), np.uint16), lengths, intr, **kw)
    blob, off = np.zeros(64, np.uint8), np.zeros(7, np.uint64)
    with pytest.raises(ValueError):
        biwi.predict_track_files_with_mask(hp, blob, off, lengths, 80, 80, intr, **kw)


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((80, 80), np.uint16)])
def test_wrappers_reject_frames(small_case, bad):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_frames_with_mask(bad, K)
    with pytest.raises(ValueError):
        hp.predict_tracks_with_mask(bad, [2], K)
    with pytest.raises(ValueError):
        hp.predict_frames_with_mask(None, K, device_ptr=1 << 40, w=640)
    with pytest.raises(ValueError):
        hp.predict_tracks_with_mask(None, [2], K, device_ptr=1 << 40, w=640)
