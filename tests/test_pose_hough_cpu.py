"""CPU tests of the pose-and-Hough calls (dh_predict_frames_hough and its Biwi form): the signatures, the
argument errors returned before any device work, and the dtype / shape checks of the Python wrappers."""
import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi
from depthhead_b200.api import frame_args

K = IntrinsicMatrix.default_kinect_intrinsic()
H, D = capi.DH_DEPTH_HOST, capi.DH_DEPTH_DEVICE


def test_signatures():
    L = capi.load()
    for name in ("dh_predict_frames_hough", "dh_predict_frames_hough_biwi"):
        assert hasattr(L, name) and len(capi.SIGNATURES[name][1]) == 13, name
    # the pose calls' arguments, then blur, hough, hough_loc and from2d as the 2-D calls have them
    assert capi.SIGNATURES["dh_predict_frames_hough"][1][:9] == capi.SIGNATURES["dh_predict_frames"][1]
    assert capi.SIGNATURES["dh_predict_frames_hough_biwi"][1][:9] == capi.SIGNATURES["dh_predict_frames_biwi"][1]
    assert capi.SIGNATURES["dh_predict_frames_hough"][1][9:] == capi.SIGNATURES["dh_build_hough_image_frames"][1][8:]
    assert capi.SIGNATURES["dh_predict_frames_hough_biwi"][1][9:] == capi.SIGNATURES["dh_build_hough_image_frames_biwi"][1][8:]


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_argument_errors(small_case):
    """every error below is returned with a NULL context: nothing reached a device"""
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    P = capi.ptr
    depth = np.zeros((3, 80, 80), np.uint16)
    res = np.zeros(3, capi.RESULT_DTYPE)
    img = np.zeros((3, 80, 80), np.uint16)
    f2d = np.zeros(3, capi.RESULT_DTYPE)
    args = frame_args(3, K)
    blob, boff = np.zeros(64, np.uint8), np.array([0, 16, 32, 48], np.uint64)
    call, cbiwi = L.dh_predict_frames_hough, L.dh_predict_frames_hough_biwi

    def both(a=args, r=res, blur=1, i=img, iloc=H, fr=f2d, ctx=None, f=hp._h, d=depth, b=blob, bo=boff, n=3):
        return (_err(call(ctx, f, P(d), n, 80, 80, H, P(a), P(r), blur, P(i), iloc, P(fr))),
                _err(cbiwi(ctx, f, P(b), P(bo), n, 80, 80, P(a), P(r), blur, P(i), iloc, P(fr))))

    for kw in (dict(), dict(f=None), dict(a=None), dict(d=None, b=None), dict(i=None), dict(fr=None), dict(blur=0, fr=None)):
        for msg in both(**kw):
            assert "NULL argument" in msg, (kw, msg)
    assert "NULL argument" in _err(cbiwi(None, hp._h, P(blob), None, 3, 80, 80, P(args), P(res), 1, P(img), H, P(f2d)))
    for msg in both(r=None):
        assert "NULL out" in msg, msg
    for kw in (dict(), dict(n=0, r=None, d=None, b=None)):  # with or without frames
        for msg in both(i=None, fr=None, **kw):
            assert "hough and from2d are both NULL" in msg, msg
        for msg in both(blur=0, **kw):
            assert "from2d needs blur = 1" in msg, msg
    for bad in (2, -1):
        for msg in both(blur=bad):
            assert "blur must be 0 or 1" in msg, msg
        for msg in both(iloc=bad):
            assert "hough_loc" in msg, msg
        assert "depth_loc" in _err(call(None, hp._h, P(depth), 3, 80, 80, bad, P(args), P(res), 1, P(img), H, P(f2d)))
    for bad in (4, 0x80000000):
        a = frame_args(3, K)
        a["has_guess"][1] = bad
        for msg in both(a=a):
            assert "frame 1" in msg and "has_guess" in msg, msg
    # the Biwi offset checks of dh_predict_batch_biwi, before any device work
    bo = np.array([0, 8, 4, 12], np.uint64)
    assert "Biwi offsets are not monotone at frame 1" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, 80, 80, P(args), P(res), 1,
                                                                      P(img), H, P(f2d)))
    bo = np.array([0, 8, 10, 12], np.uint64)
    assert "Biwi frame 2" in _err(cbiwi(None, hp._h, P(blob), P(bo), 3, 80, 80, P(args), P(res), 1, P(img), H, P(f2d)))
    # n = 0 needs no frames and no out, but still a context and a forest
    for msg in both(r=None, d=None, b=None, n=0):
        assert "NULL argument" in msg, msg


@pytest.mark.parametrize("kw", [
    dict(intrinsics=np.zeros((2, 3, 3), np.float32)),                     # 3 frames, 2 matrices
    dict(intrinsics=np.zeros((3, 3, 3), np.float64)),
    dict(midp_guess=np.zeros((3, 3), np.float64)),
    dict(rot_guess=np.zeros((2, 3), np.float64)),
    dict(has_midp=np.ones(3, bool)),                                      # a mask without its guesses
    dict(image=False, hough_device_ptr=1 << 40),                          # a device image nobody asked for
])
def test_wrappers_reject_shapes_and_dtypes(small_case, kw):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    kw = dict(kw)
    intr = kw.pop("intrinsics", K)
    with pytest.raises(ValueError):
        hp.predict_frames_with_hough(np.zeros((3, 80, 80), np.uint16), intr, **kw)
    blob, off = np.zeros(64, np.uint8), np.zeros(4, np.uint64)
    with pytest.raises(ValueError):
        biwi.predict_files_with_hough(hp, blob, off, 80, 80, intr, **kw)


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((80, 80), np.uint16)])
def test_wrappers_reject_frames(small_case, bad):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_frames_with_hough(bad, K)
    with pytest.raises(ValueError):
        hp.predict_frames_with_hough(None, K, device_ptr=1 << 40, w=640)


@pytest.mark.parametrize("kw,what", [(dict(image=False, from2d=False), "both NULL"), (dict(blur=False), "needs blur = 1")])
def test_wrappers_pass_the_c_rules_on(small_case, kw, what):
    """the wrappers leave the output rules to the C call, which refuses them before any device work"""
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(capi.DhError) as e:
        hp.predict_frames_with_hough(np.zeros((3, 80, 80), np.uint16), K, ctx=_NoContext(), **kw)
    assert e.value.code == capi.DH_E_ARG and what in str(e.value)
    with pytest.raises(capi.DhError) as e:
        biwi.predict_files_with_hough(hp, np.zeros(64, np.uint8), np.array([0, 16, 32, 48], np.uint64), 80, 80, K,
                                      ctx=_NoContext(), **kw)
    assert e.value.code == capi.DH_E_ARG and what in str(e.value)


class _NoContext:
    """stands in for a Context: a NULL handle, so that nothing can reach a device"""
    _h = None
