"""CPU tests of dh_predict_frames / dh_predict_frames_biwi: the layout of dh_frame_args in the header,
capi.FRAME_ARGS_DTYPE and the library's static_assert, the argument errors that need no device, and
the shape / dtype checks of the Python wrappers."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from depthhead_b200 import HoughPrediction, IntrinsicMatrix, biwi, capi
from depthhead_b200.api import frame_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = IntrinsicMatrix.default_kinect_intrinsic()
_CTYPES = {"float": C.c_float, "double": C.c_double, "uint32_t": C.c_uint32}


def _header_struct():
    text = open(os.path.join(ROOT, "include", "depthhead_cuda.h")).read()
    body = re.search(r"typedef struct dh_frame_args \{(.*?)\} dh_frame_args;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for typ, name, n in re.findall(r"(\w+)\s+(\w+)(?:\[(\d+)\])?;", body):
        fields.append((name, _CTYPES[typ] * int(n) if n else _CTYPES[typ]))
    return type("dh_frame_args", (C.Structure,), {"_fields_": fields})


def test_layout_agrees_between_header_capi_and_library():
    S = _header_struct()
    dt = capi.FRAME_ARGS_DTYPE
    assert C.sizeof(S) == dt.itemsize == 80
    assert [f[0] for f in S._fields_] == list(dt.names)
    src = open(os.path.join(ROOT, "depthhead_b200", "csrc", "dh_capi.cu")).read()
    asserted = dict(re.findall(r"offsetof\(dh_frame_args, (\w+)\) == (\d+)", src))
    assert "sizeof(dh_frame_args) == 80" in src
    for name in dt.names:
        assert getattr(S, name).offset == dt.fields[name][1] == int(asserted[name]), name


def test_signatures():
    L = capi.load()
    for name, n_args in (("dh_predict_frames", 9), ("dh_predict_frames_biwi", 9)):
        assert hasattr(L, name) and len(capi.SIGNATURES[name][1]) == n_args


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_argument_errors(small_case):
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    depth = np.zeros((3, 80, 80), np.uint16)
    res = np.zeros(3, capi.RESULT_DTYPE)
    args = frame_args(3, K)
    H = capi.DH_DEPTH_HOST
    blob, off = np.zeros(64, np.uint8), np.zeros(4, np.uint64)
    call, cbiwi = L.dh_predict_frames, L.dh_predict_frames_biwi
    assert "NULL" in _err(call(None, hp._h, capi.ptr(depth), 3, 80, 80, H, capi.ptr(args), capi.ptr(res)))
    assert "NULL" in _err(call(None, None, capi.ptr(depth), 0, 80, 80, H, None, None))
    assert "depth_loc" in _err(call(None, hp._h, capi.ptr(depth), 3, 80, 80, 2, capi.ptr(args), capi.ptr(res)))
    assert "depth_loc" in _err(call(None, hp._h, capi.ptr(depth), 3, 80, 80, -1, capi.ptr(args), capi.ptr(res)))
    assert "NULL" in _err(cbiwi(None, hp._h, capi.ptr(blob), capi.ptr(off), 3, 80, 80, capi.ptr(args), capi.ptr(res)))
    assert "NULL" in _err(cbiwi(None, hp._h, capi.ptr(blob), None, 3, 80, 80, capi.ptr(args), capi.ptr(res)))
    for bad in (4, 7, 0x80000000):
        args["has_guess"][:] = 0
        args["has_guess"][2] = bad
        for msg in (_err(call(None, hp._h, capi.ptr(depth), 3, 80, 80, H, capi.ptr(args), capi.ptr(res))),
                    _err(cbiwi(None, hp._h, capi.ptr(blob), capi.ptr(off), 3, 80, 80, capi.ptr(args), capi.ptr(res)))):
            assert "frame 2" in msg and "has_guess" in msg, msg


def test_frame_args_packing():
    n = 4
    Ks = np.stack([K.mat * (1 + i) for i in range(n)]).astype(np.float32)
    mid = np.arange(12, dtype=np.float32).reshape(n, 3)
    rot = -np.arange(12, dtype=np.float64).reshape(n, 3)
    a = frame_args(n, Ks, mid, rot, has_midp=np.array([True, False, True, False]), has_rot=np.array([False, False, True, True]))
    assert a["has_guess"].tolist() == [1, 0, 3, 2]
    assert np.array_equal(a["K"], Ks.reshape(n, 9))
    assert np.array_equal(a["midp_guess"][[0, 2]], mid[[0, 2]]) and not a["midp_guess"][[1, 3]].any()
    assert np.array_equal(a["rot_guess"][[2, 3]], rot[[2, 3]]) and not a["rot_guess"][[0, 1]].any()
    b = frame_args(n, K, None, rot)
    assert b["has_guess"].tolist() == [2] * n and np.array_equal(b["K"], np.tile(K.mat.reshape(9), (n, 1)))


@pytest.mark.parametrize("kw", [
    dict(intrinsics=np.zeros((2, 3, 3), np.float32)),                    # n = 3 frames, 2 matrices
    dict(intrinsics=np.zeros((3, 3, 3), np.float64)),
    dict(intrinsics=np.zeros((3, 9), np.float32)),
    dict(midp_guess=np.zeros((3, 3), np.float64)),
    dict(midp_guess=np.zeros((3, 2), np.float32)),
    dict(rot_guess=np.zeros((3, 3), np.float32)),
    dict(rot_guess=np.zeros((4, 3), np.float64)),
    dict(midp_guess=np.zeros((3, 3), np.float32), has_midp=np.ones(3, np.uint8)),
    dict(rot_guess=np.zeros((3, 3), np.float64), has_rot=np.ones(2, bool)),
    dict(has_midp=np.ones(3, bool)),                                      # a mask without its guesses
])
def test_wrappers_reject_shapes_and_dtypes(small_case, kw):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    frames = np.zeros((3, 80, 80), np.uint16)
    kw = dict(kw)
    intr = kw.pop("intrinsics", K)
    with pytest.raises(ValueError):
        hp.predict_frames(frames, intr, **kw)
    blob, off = np.zeros(64, np.uint8), np.zeros(4, np.uint64)
    with pytest.raises(ValueError):
        biwi.predict_files(hp, blob, off, 80, 80, intr if not isinstance(intr, IntrinsicMatrix) else np.zeros((1, 3, 3), np.float32),
                           **kw)


@pytest.mark.parametrize("bad", [np.zeros((2, 80, 80), np.int16), np.zeros((80, 80), np.uint16), np.zeros((1, 2, 80, 80), np.uint16)])
def test_wrapper_rejects_frames(small_case, bad):
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    with pytest.raises(ValueError):
        hp.predict_frames(bad, K)
    with pytest.raises(ValueError):
        hp.predict_frames(None, K, device_ptr=1 << 40, n=2, w=640)
