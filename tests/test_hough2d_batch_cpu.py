"""CPU tests of the batched 2-D entry points (dh_predict_mask_batch, dh_build_hough_image_batch):
their signatures, the argument errors that need no device, and the dtype / rank checks of the
Python wrappers."""
import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, capi

K = IntrinsicMatrix.default_kinect_intrinsic()


def test_signatures():
    L = capi.load()
    for name in ("dh_predict_mask_batch", "dh_build_hough_image_batch"):
        assert hasattr(L, name) and name in capi.SIGNATURES
    assert len(capi.SIGNATURES["dh_predict_mask_batch"][1]) == 9
    assert len(capi.SIGNATURES["dh_build_hough_image_batch"][1]) == 12


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_mask_batch_argument_errors():
    L = capi.load()
    depth = np.zeros((1, 80, 80), np.uint16)
    mask = np.zeros((1, 80, 80), np.uint8)
    H, D = capi.DH_DEPTH_HOST, capi.DH_DEPTH_DEVICE
    assert "NULL" in _err(L.dh_predict_mask_batch(None, None, capi.ptr(depth), 1, 80, 80, H, capi.ptr(mask), H))
    assert "depth_loc" in _err(L.dh_predict_mask_batch(None, None, capi.ptr(depth), 1, 80, 80, 2, capi.ptr(mask), H))
    assert "mask_loc" in _err(L.dh_predict_mask_batch(None, None, capi.ptr(depth), 1, 80, 80, D, capi.ptr(mask), -1))


def test_hough_batch_argument_errors(small_case):
    L = capi.load()
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)  # a real forest: the context is the only missing piece
    depth = np.zeros((1, 80, 80), np.uint16)
    img = np.zeros((1, 80, 80), np.uint16)
    res = np.zeros(1, capi.RESULT_DTYPE)
    H = capi.DH_DEPTH_HOST
    call = L.dh_build_hough_image_batch
    assert "NULL" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 1, capi.ptr(img), H, None))
    assert "NULL" in _err(call(None, None, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 1, capi.ptr(img), H, None))
    assert "depth_loc" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), 7, 1, capi.ptr(img), H, None))
    assert "hough_loc" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 1, capi.ptr(img), 3, None))
    assert "blur" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 2, capi.ptr(img), H, None))
    assert "from2d needs blur" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 0, capi.ptr(img), H,
                                            capi.ptr(res)))
    assert "both NULL" in _err(call(None, hp._h, capi.ptr(depth), 1, 80, 80, K._ptr(), H, 1, None, H, None))
    assert "both NULL" in _err(call(None, hp._h, capi.ptr(depth), 0, 80, 80, K._ptr(), H, 1, None, H, None))


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((2, 80, 80), np.float32),
                                 np.zeros((80, 80), np.uint16), np.zeros((1, 2, 80, 80), np.uint16)])
def test_wrappers_reject_dtype_and_rank(small_case, bad):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_mask_batch(bad)
    with pytest.raises(ValueError):
        hp.hough_image_raw_batch(bad, K)
    with pytest.raises(ValueError):
        hp.build_hough_image_batch(bad, K, from2d=True)
    with pytest.raises(ValueError):
        hp.predict_parameter_from2dhough_batch(bad, K)


def test_device_pointer_needs_sizes(small_case):
    arr, js, frames = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_mask_batch(None, device_ptr=1 << 40, n=2, w=640)
    with pytest.raises(ValueError):
        hp.predict_parameter_from2dhough_batch(None, K, device_ptr=1 << 40, w=640, h=480)
