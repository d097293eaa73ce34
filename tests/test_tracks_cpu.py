"""CPU tests of dh_predict_tracks / dh_predict_tracks_biwi: the signatures, the argument errors that are
returned before any device work, and the dtype / rank / length checks of the Python wrappers."""
import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi
from depthhead_b200.api import _track_offsets, frame_args

K = IntrinsicMatrix.default_kinect_intrinsic()
H = capi.DH_DEPTH_HOST


def test_signatures():
    L = capi.load()
    for name, n_args in (("dh_predict_tracks", 11), ("dh_predict_tracks_biwi", 11)):
        assert hasattr(L, name) and len(capi.SIGNATURES[name][1]) == n_args


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_argument_errors(small_case):
    """every error below is returned with a NULL context: nothing reached a device"""
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    depth = np.zeros((6, 80, 80), np.uint16)
    res = np.zeros(6, capi.RESULT_DTYPE)
    off = np.array([0, 2, 2, 6], np.uint64)
    args = frame_args(3, K)
    blob, boff = np.zeros(64, np.uint8), np.zeros(7, np.uint64)
    call, cbiwi = L.dh_predict_tracks, L.dh_predict_tracks_biwi
    P = capi.ptr

    def both(seq_off, a, loc=H, ctx=None, f=hp._h, d=depth, r=res, b=blob, bo=boff):
        return (_err(call(ctx, f, P(d), 3, P(seq_off), 80, 80, loc, P(a), 500.0, P(r))),
                _err(cbiwi(ctx, f, P(b), P(bo), 3, P(seq_off), 80, 80, P(a), 500.0, P(r))))

    # NULL context, forest, seq_off, seq_args, frames, results
    for msg in both(off, args):
        assert "NULL" in msg, msg
    for msg in both(off, args, ctx=None, f=None):
        assert "NULL" in msg, msg
    for msg in both(None, args):
        assert "NULL" in msg, msg
    for msg in both(off, None):
        assert "NULL" in msg, msg
    for msg in both(off, args, d=None, b=None, r=None):
        assert "NULL" in msg, msg
    assert "NULL" in _err(cbiwi(None, hp._h, P(blob), None, 3, P(off), 80, 80, P(args), 500.0, P(res)))
    # bad depth_loc
    for loc in (2, -1):
        assert "depth_loc" in _err(call(None, hp._h, P(depth), 3, P(off), 80, 80, loc, P(args), 500.0, P(res)))
    # seq_off not starting at 0, not monotone, more than 2^31 - 1 frames
    for bad, what in ((np.array([1, 2, 2, 6], np.uint64), "seq_off[0]"), (np.array([0, 3, 2, 6], np.uint64), "track 1"),
                      (np.array([0, 2, 2, 1 << 31], np.uint64), "2^31")):
        for msg in both(bad, args):
            assert what in msg, msg
    # has_guess bits beyond 0-1, naming the track
    for bad in (4, 7, 0x80000000):
        a = frame_args(3, K)
        a["has_guess"][2] = bad
        for msg in both(off, a):
            assert "track 2" in msg and "has_guess" in msg, msg
    # the Biwi offset checks of dh_predict_batch_biwi
    bo = np.array([0, 8, 4, 12, 16, 20, 24], np.uint64)
    assert "not monotone at frame 1" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, P(off), 80, 80, P(args), 500.0, P(res)))
    bo = np.array([0, 8, 10, 12, 16, 20, 24], np.uint64)
    assert "Biwi frame 2" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, P(off), 80, 80, P(args), 500.0, P(res)))


def test_track_offsets():
    seq_off, n_seq, total = _track_offsets([7, 1, 0, 12, 3, 5])
    assert seq_off.dtype == np.uint64 and seq_off.tolist() == [0, 7, 8, 8, 20, 23, 28] and (n_seq, total) == (6, 28)
    assert _track_offsets([])[1:] == (0, 0)
    for bad in ([3, -1], [[1, 2]], [1.5, 2.0], [1 << 31]):
        with pytest.raises(ValueError):
            _track_offsets(np.array(bad))


@pytest.mark.parametrize("kw", [
    dict(lengths=[2, 2]),                                                 # 4 frames for 6
    dict(lengths=[3, 4]),                                                 # 7 frames for 6
    dict(lengths=[[3, 3]]),
    dict(lengths=[3, -3, 6]),
    dict(intrinsics=np.zeros((3, 3, 3), np.float32)),                     # 2 tracks, 3 matrices
    dict(intrinsics=np.zeros((2, 3, 3), np.float64)),
    dict(midp_guess=np.zeros((2, 3), np.float64)),
    dict(rot_guess=np.zeros((6, 3), np.float64)),                         # one seed per frame, not per track
    dict(rot_guess=np.zeros((2, 3), np.float64), has_rot=np.ones(2, np.uint8)),
    dict(has_midp=np.ones(2, bool)),                                      # a mask without its guesses
])
def test_wrappers_reject_shapes_and_dtypes(small_case, kw):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    frames = np.zeros((6, 80, 80), np.uint16)
    kw = dict(kw)
    lengths = kw.pop("lengths", [2, 4])
    intr = kw.pop("intrinsics", K)
    with pytest.raises(ValueError):
        hp.predict_tracks(frames, lengths, intr, **kw)
    blob, off = np.zeros(64, np.uint8), np.zeros(7, np.uint64)
    with pytest.raises(ValueError):
        biwi.predict_track_files(hp, blob, off, lengths, 80, 80, intr, **kw)


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((80, 80), np.uint16), np.zeros((1, 2, 80, 80), np.uint16)])
def test_wrapper_rejects_frames(small_case, bad):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_tracks(bad, [2], K)
    with pytest.raises(ValueError):
        hp.predict_tracks(None, [2], K, device_ptr=1 << 40, w=640)
