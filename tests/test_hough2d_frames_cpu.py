"""CPU tests of the 2-D entry points with a K per frame and from Biwi files (dh_build_hough_image_frames,
dh_build_hough_image_frames_biwi, dh_predict_mask_batch_biwi): their signatures in capi.py and the
header, the argument errors that need no device, and the checks of the Python wrappers."""
import os
import re

import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = IntrinsicMatrix.default_kinect_intrinsic()
NAMES = {"dh_build_hough_image_frames": 12, "dh_build_hough_image_frames_biwi": 12, "dh_predict_mask_batch_biwi": 9}


def test_signatures_in_capi_and_header():
    L = capi.load()
    text = open(os.path.join(ROOT, "include", "depthhead_cuda.h")).read()
    for name, n_args in NAMES.items():
        assert hasattr(L, name) and len(capi.SIGNATURES[name][1]) == n_args, name
        decl = re.search(r"\bint %s\((.*?)\);" % name, text, re.S).group(1)
        decl = re.sub(r"/\*.*?\*/", "", decl)
        assert len(decl.split(",")) == n_args, name
        assert name in text.split("*/")[0], "%s is missing from the table of replaced interfaces" % name


def _err(rc, fn):
    assert rc == capi.DH_E_ARG, rc
    msg = capi.load().dh_last_error().decode()
    assert fn in msg, msg
    return msg


@pytest.fixture
def hp(small_case):
    return HoughPrediction.from_json(small_case[1])  # a real forest: the context is the only missing piece


def test_frames_argument_errors(hp):
    L = capi.load()
    fn = "dh_build_hough_image_frames"
    call = L.dh_build_hough_image_frames
    depth = np.zeros((2, 80, 80), np.uint16)
    img = np.zeros((2, 80, 80), np.uint16)
    res = np.zeros(2, capi.RESULT_DTYPE)
    Ks = np.tile(K.mat.reshape(9), (2, 1))
    H, D = capi.DH_DEPTH_HOST, capi.DH_DEPTH_DEVICE
    d, k, i, r = capi.ptr(depth), capi.ptr(Ks), capi.ptr(img), capi.ptr(res)
    assert "NULL" in _err(call(None, hp._h, d, 2, 80, 80, H, k, 1, i, H, r), fn)
    assert "NULL" in _err(call(None, None, d, 0, 80, 80, H, k, 1, i, H, None), fn)
    assert "depth_loc" in _err(call(None, hp._h, d, 2, 80, 80, 2, k, 1, i, H, r), fn)
    assert "depth_loc" in _err(call(None, hp._h, d, 2, 80, 80, -1, k, 1, i, H, r), fn)
    assert "hough_loc" in _err(call(None, hp._h, d, 2, 80, 80, D, k, 1, i, 3, r), fn)
    assert "blur" in _err(call(None, hp._h, d, 2, 80, 80, H, k, 2, i, H, None), fn)
    assert "blur" in _err(call(None, hp._h, d, 2, 80, 80, H, k, -1, i, H, None), fn)
    assert "from2d needs blur" in _err(call(None, hp._h, d, 2, 80, 80, H, k, 0, i, H, r), fn)
    assert "both NULL" in _err(call(None, hp._h, d, 2, 80, 80, H, k, 1, None, H, None), fn)
    assert "both NULL" in _err(call(None, hp._h, d, 0, 80, 80, H, k, 0, None, H, None), fn)


def test_biwi_argument_errors(hp):
    L = capi.load()
    blob, off = np.zeros(64, np.uint8), np.array([0, 16, 32], np.uint64)
    img = np.zeros((2, 80, 80), np.uint16)
    mask = np.zeros((2, 80, 80), np.uint8)
    res = np.zeros(2, capi.RESULT_DTYPE)
    Ks = np.tile(K.mat.reshape(9), (2, 1))
    H = capi.DH_DEPTH_HOST
    b, o, k, i, r = capi.ptr(blob), capi.ptr(off), capi.ptr(Ks), capi.ptr(img), capi.ptr(res)
    fn, call = "dh_build_hough_image_frames_biwi", L.dh_build_hough_image_frames_biwi
    assert "NULL" in _err(call(None, hp._h, b, o, 2, 80, 80, k, 1, i, H, r), fn)
    assert "NULL" in _err(call(None, hp._h, b, None, 2, 80, 80, k, 1, i, H, r), fn)
    assert "hough_loc" in _err(call(None, hp._h, b, o, 2, 80, 80, k, 1, i, 5, r), fn)
    assert "blur" in _err(call(None, hp._h, b, o, 2, 80, 80, k, 3, i, H, r), fn)
    assert "from2d needs blur" in _err(call(None, hp._h, b, o, 2, 80, 80, k, 0, i, H, r), fn)
    assert "both NULL" in _err(call(None, hp._h, b, o, 2, 80, 80, k, 1, None, H, None), fn)
    mfn, mcall = "dh_predict_mask_batch_biwi", L.dh_predict_mask_batch_biwi
    assert "NULL" in _err(mcall(None, hp._h, b, o, 2, 80, 80, capi.ptr(mask), H), mfn)
    assert "NULL" in _err(mcall(None, None, b, o, 0, 80, 80, None, H), mfn)
    assert "NULL" in _err(mcall(None, hp._h, b, o, 2, 80, 80, None, H), mfn)
    assert "mask_loc" in _err(mcall(None, hp._h, b, o, 2, 80, 80, capi.ptr(mask), 2), mfn)


@pytest.mark.parametrize("off,what", [([0, 32, 16], "not monotone at frame 1"), ([0, 18, 32], "frame 1 does not start at a multiple of 4"),
                                      ([0, 16, 16 + (1 << 32)], "frame 1 is larger than 4 GB")])
def test_bad_biwi_offsets_are_rejected(hp, off, what):
    """before anything else that needs the context: the context here is NULL"""
    L = capi.load()
    blob = np.zeros(64, np.uint8)
    o = np.array(off, np.uint64)
    Ks = np.tile(K.mat.reshape(9), (2, 1))
    img = np.zeros((2, 80, 80), np.uint16)
    assert what in _err(L.dh_build_hough_image_frames_biwi(None, hp._h, capi.ptr(blob), capi.ptr(o), 2, 80, 80, capi.ptr(Ks), 1,
                                                           capi.ptr(img), capi.DH_DEPTH_HOST, None), "dh_build_hough_image_frames_biwi: Biwi")
    assert what in _err(L.dh_predict_mask_batch_biwi(None, hp._h, capi.ptr(blob), capi.ptr(o), 2, 80, 80, capi.ptr(img),
                                                     capi.DH_DEPTH_HOST), "dh_predict_mask_batch_biwi: Biwi")


@pytest.mark.parametrize("intr", [np.zeros((2, 3, 3), np.float32), np.zeros((3, 3, 3), np.float64), np.zeros((3, 9), np.float32),
                                  np.zeros((4, 3, 3), np.float32), K.mat])
def test_wrappers_reject_intrinsics(hp, intr):
    frames = np.zeros((3, 80, 80), np.uint16)
    for call in (hp.hough_image_raw_frames, hp.build_hough_image_frames, hp.predict_parameter_from2dhough_frames):
        with pytest.raises(ValueError):
            call(frames, intr)
    blob, off = np.zeros(64, np.uint8), np.array([0, 16, 32, 48], np.uint64)
    with pytest.raises(ValueError):
        biwi.build_hough_image_files(hp, blob, off, 80, 80, intr)


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((2, 80, 80), np.float32),
                                 np.zeros((80, 80), np.uint16), np.zeros((1, 2, 80, 80), np.uint16)])
def test_wrappers_reject_frames(hp, bad):
    for call in (hp.hough_image_raw_frames, hp.build_hough_image_frames, hp.predict_parameter_from2dhough_frames):
        with pytest.raises(ValueError):
            call(bad, K)


def test_device_pointer_needs_sizes(hp):
    with pytest.raises(ValueError):
        hp.build_hough_image_frames(None, K, device_ptr=1 << 40, n=2, w=640)
    with pytest.raises(ValueError):
        hp.predict_parameter_from2dhough_frames(None, K, device_ptr=1 << 40, w=640, h=480)
    with pytest.raises(ValueError):
        hp.hough_image_raw_frames(None, K, device_ptr=1 << 40, n=2, h=480)
