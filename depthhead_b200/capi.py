"""ctypes binding of include/depthhead_cuda.h (libdepthhead_cuda.so).

This is the same surface the Rust shim in INTEGRATION.md binds; nothing here computes anything.
The library must exist (built in-tree by ``depthhead_b200._build``); there is no fallback of any
kind — a missing library or a missing GPU is an error, loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

DH_OK, DH_E_JSON, DH_E_SHAPE, DH_E_CUDA, DH_E_ARG, DH_E_STATE = 0, -1, -2, -3, -4, -5
DH_DEPTH_HOST, DH_DEPTH_DEVICE = 0, 1
DH_N_STAGES, DH_N_COUNTERS = 7, 12
STAGES = ("h2d", "sat", "traverse", "gate", "vote", "meanshift", "d2h")
COUNTERS = ("frames", "patches", "valid_patches", "evals", "node_visits", "gate_patches", "hits",
            "centre_votes", "rot_votes", "launches", "meanshift_iters", "cube_rebuilds")


class DhError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("%s (code %d)" % (msg, code))
        self.code = code


class dh_result(C.Structure):
    _fields_ = [("mid_point", C.c_float * 3), ("_pad", C.c_uint32), ("rotation", C.c_double * 3),
                ("bounding_box", C.c_uint32 * 4)]


RESULT_DTYPE = np.dtype([("mid_point", np.float32, 3), ("_pad", np.uint32), ("rotation", np.float64, 3),
                         ("bounding_box", np.uint32, 4)], align=True)
assert RESULT_DTYPE.itemsize == C.sizeof(dh_result) == 56


# dh_frame_args: the arguments of dh_predict for one frame of dh_predict_frames (80 bytes)
FRAME_ARGS_DTYPE = np.dtype([("K", np.float32, 9), ("midp_guess", np.float32, 3), ("rot_guess", np.float64, 3),
                             ("has_guess", np.uint32), ("_pad", np.uint32)], align=True)
assert FRAME_ARGS_DTYPE.itemsize == 80


# dh_heads_params / dh_head: dh_predict_frames_heads (16 and 72 bytes)
HEADS_PARAMS_DTYPE = np.dtype([("max_heads", np.uint32), ("min_cell_votes", np.uint32), ("radius_mm", np.float32),
                               ("_pad", np.uint32)], align=True)
assert HEADS_PARAMS_DTYPE.itemsize == 16
HEAD_DTYPE = np.dtype([("pose", RESULT_DTYPE), ("support", np.uint64), ("n_patches", np.uint32), ("seed_cell", np.uint32)],
                      align=True)
assert HEAD_DTYPE.itemsize == 72


class dh_split_stats(C.Structure):
    _fields_ = [("n", C.c_uint32 * 2), ("n_pos", C.c_uint32 * 2), ("det_off", C.c_double * 2), ("det_rot", C.c_double * 2),
                ("impurity", C.c_double)]


SPLIT_DTYPE = np.dtype([("n", np.uint32, 2), ("n_pos", np.uint32, 2), ("det_off", np.float64, 2), ("det_rot", np.float64, 2),
                        ("impurity", np.float64)], align=True)
assert SPLIT_DTYPE.itemsize == C.sizeof(dh_split_stats) == 56


class dh_train_params(C.Structure):
    _fields_ = [("stepwidth", C.c_uint32), ("subimage_width", C.c_uint32), ("subimage_height", C.c_uint32),
                ("max_depth", C.c_uint32), ("n_trees", C.c_uint32), ("subset_per_tree", C.c_uint32),
                ("subrect_feature_scale", C.c_double), ("features_per_node", C.c_uint32), ("min_subset_size", C.c_uint32),
                ("steepness", C.c_double), ("gaussian_sigma", C.c_float), ("_pad", C.c_uint32), ("seed", C.c_uint64)]


class dh_forest_arrays(C.Structure):
    _fields_ = [("stepwidth", C.c_uint32), ("subimage_width", C.c_uint32), ("subimage_height", C.c_uint32),
                ("meanshift_iterations", C.c_uint32), ("gaussian_sigma", C.c_float), ("n_trees", C.c_int32),
                ("tree_node_off", C.c_void_p), ("tree_leaf_off", C.c_void_p), ("rects", C.c_void_p),
                ("threshold", C.c_void_p), ("child", C.c_void_p), ("prob", C.c_void_p), ("vote_off", C.c_void_p),
                ("offsets", C.c_void_p), ("rotations", C.c_void_p)]


# name -> (restype, argtypes); the CPU test-suite checks this table against the header.
_vp, _u32, _i32, _u64, _f32 = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64, C.c_float
SIGNATURES = {
    "dh_last_error": (C.c_char_p, []),
    "dh_abi_version": (C.c_int, []),
    "dh_forest_from_json": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(_vp)]),
    "dh_forest_from_arrays": (C.c_int, [C.POINTER(dh_forest_arrays), C.POINTER(_vp)]),
    "dh_forest_free": (None, [_vp]),
    "dh_forest_get_stepwidth": (_u32, [_vp]),
    "dh_forest_set_stepwidth": (C.c_int, [_vp, _u32]),
    "dh_forest_get_meanshift_iterations": (_u32, [_vp]),
    "dh_forest_set_meanshift_iterations": (C.c_int, [_vp, _u32]),
    "dh_forest_get_sigma": (_f32, [_vp]),
    "dh_forest_set_sigma": (C.c_int, [_vp, _f32]),
    "dh_forest_get_subimage_width": (_u32, [_vp]),
    "dh_forest_get_subimage_height": (_u32, [_vp]),
    "dh_forest_n_trees": (_i32, [_vp]),
    "dh_forest_n_nodes": (C.c_int64, [_vp]),
    "dh_forest_n_leaves": (C.c_int64, [_vp]),
    "dh_forest_n_votes": (C.c_int64, [_vp]),
    "dh_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "dh_ctx_free": (None, [_vp]),
    "dh_ctx_set_stream": (C.c_int, [_vp, _vp]),
    "dh_ctx_set_chunk_frames": (C.c_int, [_vp, _u32]),
    "dh_ctx_synchronize": (C.c_int, [_vp]),
    "dh_ctx_set_encode_threads": (C.c_int, [_vp, _u32]),
    "dh_ctx_transfer_info": (C.c_int, [_vp, _vp]),
    "dh_build_id": (C.c_char_p, []),
    "dh_biwi_encode_bound": (C.c_size_t, [_u32, _u32]),
    "dh_biwi_encode_depth": (C.c_int, [_vp, _u32, _u32, _u32, _u32, _vp, C.c_size_t, _vp, C.POINTER(C.c_size_t)]),
    "dh_predict": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, C.POINTER(dh_result)]),
    "dh_predict_batch": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, _vp, C.c_int, _vp]),
    "dh_biwi_depth_dims": (C.c_int, [_vp, C.c_size_t, C.POINTER(_u32), C.POINTER(_u32)]),
    "dh_biwi_decode_depth": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, _vp, C.c_int]),
    "dh_predict_batch_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp]),
    "dh_biwi_parse_cal": (C.c_int, [C.c_char_p, C.c_size_t, _vp]),
    "dh_biwi_parse_pose": (C.c_int, [_vp, C.c_size_t, _vp, _vp, _vp, _vp]),
    "dh_trainset_create": (C.c_int, [_vp, _vp, _u64, _u32, _u32, _u32, _u32, _vp, _vp, _vp, C.POINTER(_vp)]),
    "dh_trainset_free": (None, [_vp]),
    "dh_train_score_level": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp, _vp, _u32, _u64, C.c_double, _vp]),
    "dh_train_split_level": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp, _vp, _vp]),
    "dh_train_forest": (C.c_int, [_vp, C.POINTER(dh_train_params), _vp, _u64, _vp, _vp, _vp, C.POINTER(_vp)]),
    "dh_train_learn": (C.c_int, [_vp, C.POINTER(dh_train_params), _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "dh_forest_to_json": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "dh_predict_mask": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp]),
    "dh_predict_sequences": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, _u32, _vp, C.c_int, _f32, _vp]),
    "dh_predict_frames": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, _vp]),
    "dh_predict_frames_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp]),
    "dh_predict_tracks": (C.c_int, [_vp, _vp, _vp, _u32, _vp, _u32, _u32, C.c_int, _vp, _f32, _vp]),
    "dh_predict_tracks_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp, _u32, _u32, _vp, _f32, _vp]),
    "dh_predict_frames_mask": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, _vp, _vp, C.c_int]),
    "dh_predict_frames_mask_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp, C.c_int]),
    "dh_predict_tracks_mask": (C.c_int, [_vp, _vp, _vp, _u32, _vp, _u32, _u32, C.c_int, _vp, _f32, _vp, _vp, C.c_int]),
    "dh_predict_tracks_mask_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _vp, _u32, _u32, _vp, _f32, _vp, _vp, C.c_int]),
    "dh_predict_frames_heads": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, _vp, _vp, _vp]),
    "dh_predict_frames_hough": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "dh_predict_frames_hough_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp, C.c_int, _vp, C.c_int, _vp]),
    "dh_hough_image_raw": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "dh_build_hough_image": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "dh_predict_from2dhough": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _vp, C.POINTER(dh_result)]),
    "dh_predict_mask_batch": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, C.c_int]),
    "dh_build_hough_image_batch": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "dh_build_hough_image_frames": (C.c_int, [_vp, _vp, _vp, _u32, _u32, _u32, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp]),
    "dh_build_hough_image_frames_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, C.c_int, _vp, C.c_int, _vp]),
    "dh_predict_mask_batch_biwi": (C.c_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, C.c_int]),
    "dh_ctx_enable_stage_timing": (C.c_int, [_vp, C.c_int]),
    "dh_ctx_stage_ms": (C.c_int, [_vp, _vp]),
    "dh_ctx_counters": (C.c_int, [_vp, _vp]),
    "dh_ctx_enable_debug": (C.c_int, [_vp, C.c_int]),
    "dh_debug_dims": (C.c_int, [_vp, C.POINTER(_u32), C.POINTER(_u32), C.POINTER(_u32)]),
    "dh_debug_leaf_indices": (C.c_int, [_vp, _vp]),
    "dh_debug_patches": (C.c_int, [_vp, _vp, _vp]),
    "dh_debug_seeds": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "dh_debug_votes": (C.c_int, [_vp, C.c_int, _vp, _vp, C.POINTER(_u64), _vp, C.POINTER(_i32)]),
    "dh_debug_meanshift": (C.c_int, [_vp, C.c_int, _vp, C.POINTER(_u32)]),
    "dh_debug_meanshift_flags": (C.c_int, [_vp, _vp]),
    "dh_debug_tile_plan": (C.c_int, [_vp, _vp]),
    "dh_debug_leaf_static": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load libdepthhead_cuda.so (building it first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    if os.environ.get("DH_NO_BUILD") != "1":
        _build.build()
    if not os.path.exists(_build.LIB):
        raise RuntimeError("libdepthhead_cuda.so is missing: run `python -m depthhead_b200._build` "
                           "(there is no CPU or PyTorch fallback)")
    L = C.CDLL(_build.LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int):
    if rc != DH_OK:
        raise DhError(rc, load().dh_last_error().decode("utf-8", "replace"))


def ptr(a):
    """Pointer for a numpy array / int device pointer / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)
