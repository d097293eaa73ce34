"""Host-side mirror of the reference's prediction API, on top of the C ABI.

Names, arguments and error behaviour follow the reference so the parity tests read like the
reference's own usage (Readme.md:76-100, examples/live_prediction.rs:76-88):

    reference (Rust)                                          here
    ---------------------------------------------------------------------------------------------
    serde_json::from_str::<HoughPrediction>(&s)               HoughPrediction.from_json(s)
    IntrinsicMatrix::default_kinect_intrinsic()               IntrinsicMatrix.default_kinect_intrinsic()
    forest.predict_parameter_parallel(img, &K, None, None)    forest.predict_parameter_parallel(img, K)
    forest.predict_parameter(img, &K, mid, rot)               forest.predict_parameter(img, K, mid, rot)
    forest.predict_mask(img)                                  forest.predict_mask(img)
    forest.update_sigma(v) / forest.sigma()                   same
    forest.stepwidth / forest.meanshift_iterations (pub)      properties with setters
    PredictionResult {mid_point, rotation, bounding_box}      PredictionResult dataclass

Every compute call goes to libdepthhead_cuda.so on a CUDA device; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi


class IntrinsicMatrix:
    """types.rs:405-446.  Row-major 3x3 f32; the inverse is computed inside the library with the
    adjugate formula of meancov_estimation.rs:344-352."""

    def __init__(self, mat):
        m = np.asarray(mat, np.float32)
        if m.size != 9:
            raise ValueError("IntrinsicMatrix needs 9 values")
        self.mat = np.ascontiguousarray(m.reshape(3, 3))

    @staticmethod
    def default_kinect_intrinsic() -> "IntrinsicMatrix":  # types.rs:418-420
        return IntrinsicMatrix([[560.0, 0.0, 320.0], [0.0, 560.0, 240.0], [0.0, 0.0, 1.0]])

    def _ptr(self):
        return capi.ptr(self.mat)


@dataclass
class PredictionResult:  # prediction.rs:259-267
    mid_point: np.ndarray      # [3] f32, whole millimetres
    rotation: np.ndarray       # [3] f64, radians
    bounding_box: tuple        # always (0, 0, 0, 0): the reference never predicts it


class Context:
    """One per GPU per host thread (the reference's HoughPrediction is !Sync for the same reason)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        capi.check(capi.load().dh_ctx_create(int(device), C.byref(self._h)))
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            capi.load().dh_ctx_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int | None):
        capi.check(capi.load().dh_ctx_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def set_chunk_frames(self, frames: int):
        capi.check(capi.load().dh_ctx_set_chunk_frames(self._h, int(frames)))

    def set_encode_threads(self, n: int):
        """worker threads of the compressed host->device path of predict_batch (0 = default)"""
        capi.check(capi.load().dh_ctx_set_encode_threads(self._h, int(n)))

    def transfer_info(self) -> dict:
        a = np.zeros(4, np.uint64)
        capi.check(capi.load().dh_ctx_transfer_info(self._h, capi.ptr(a)))
        return {"h2d_bytes": int(a[0]), "encoded_chunks": int(a[1]), "encode_threads": int(a[2])}

    def synchronize(self):
        capi.check(capi.load().dh_ctx_synchronize(self._h))

    def enable_stage_timing(self, on: bool = True):
        capi.check(capi.load().dh_ctx_enable_stage_timing(self._h, int(on)))

    def enable_debug(self, on: bool = True):
        capi.check(capi.load().dh_ctx_enable_debug(self._h, int(on)))

    def stage_ms(self) -> dict:
        a = np.zeros(capi.DH_N_STAGES, np.float32)
        capi.check(capi.load().dh_ctx_stage_ms(self._h, capi.ptr(a)))
        return dict(zip(capi.STAGES, a.tolist()))

    def counters(self) -> dict:
        a = np.zeros(capi.DH_N_COUNTERS, np.uint64)
        capi.check(capi.load().dh_ctx_counters(self._h, capi.ptr(a)))
        return dict(zip(capi.COUNTERS, (int(x) for x in a)))

    # ---- debug exports (parity tests)
    def tile_plan(self) -> dict:
        v = np.zeros(8, np.uint32)
        capi.check(capi.load().dh_debug_tile_plan(self._h, capi.ptr(v)))
        keys = ("patches_x", "patches_y", "tiles_x", "tiles_y", "tile_w", "tile_h", "smem_bytes", "threads")
        return {k: int(x) for k, x in zip(keys, v)}

    def debug_dims(self):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        capi.check(capi.load().dh_debug_dims(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def debug_leaf_indices(self) -> np.ndarray:
        npx, npy, T = self.debug_dims()
        out = np.zeros((npx * npy, T), np.int32)
        capi.check(capi.load().dh_debug_leaf_indices(self._h, capi.ptr(out)))
        return out

    def debug_patches(self):
        npx, npy, _ = self.debug_dims()
        p3 = np.zeros((npx * npy, 3), np.float32)
        gate = np.zeros(npx * npy, np.uint8)
        capi.check(capi.load().dh_debug_patches(self._h, capi.ptr(p3), capi.ptr(gate)))
        return p3, gate

    def debug_seeds(self):
        gp, gr = np.zeros(400, np.uint32), np.zeros(8000, np.uint32)
        sm, sr = np.zeros(3, np.int32), np.zeros(3, np.int32)
        capi.check(capi.load().dh_debug_seeds(self._h, capi.ptr(gp), capi.ptr(gr), capi.ptr(sm), capi.ptr(sr)))
        return gp, gr, sm, sr

    def debug_votes(self, which: int):
        """(keys[n,3] i32, vals[n] u32, box_origin[3], box_dim) sorted by key: the non-zero cells of the
        dense accumulator cube around the last mean-shift position."""
        L = capi.load()
        n, dim = C.c_uint64(), C.c_int32()
        org = np.zeros(3, np.int32)
        capi.check(L.dh_debug_votes(self._h, int(which), None, None, C.byref(n), capi.ptr(org), C.byref(dim)))
        keys = np.zeros((n.value, 3), np.int32)
        vals = np.zeros(n.value, np.uint32)
        if n.value:
            capi.check(L.dh_debug_votes(self._h, int(which), capi.ptr(keys), capi.ptr(vals), C.byref(n), capi.ptr(org),
                                        C.byref(dim)))
            order = np.lexsort((keys[:, 2], keys[:, 1], keys[:, 0]))
            keys, vals = keys[order], vals[order]
        return keys, vals, org, dim.value

    def debug_meanshift(self, which: int, max_iter: int = 65535):
        L = capi.load()
        n = C.c_uint32(0)
        capi.check(L.dh_debug_meanshift(self._h, int(which), None, C.byref(n)))
        cnt = min(n.value, max_iter)
        pos = np.zeros((cnt, 3), np.int32)
        n2 = C.c_uint32(cnt)
        if cnt:
            capi.check(L.dh_debug_meanshift(self._h, int(which), capi.ptr(pos), C.byref(n2)))
        return pos

    def debug_meanshift_flags(self):
        a = np.zeros(2, np.uint32)
        capi.check(capi.load().dh_debug_meanshift_flags(self._h, capi.ptr(a)))
        return int(a[0]), int(a[1])


_default_ctx: dict = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


def _as_depth(img) -> np.ndarray:
    a = np.asarray(img)
    if a.dtype != np.uint16 or a.ndim != 2:
        raise ValueError("DepthImage must be a 2-D uint16 array [h, w] (types.rs:10)")
    return np.ascontiguousarray(a)


def _as_frames(frames, device_ptr, n, w, h):
    """(keep-alive array, pointer, location, n, w, h) of a [n,h,w] uint16 host batch or a device pointer."""
    if device_ptr is None:
        a = np.asarray(frames)
        if a.dtype != np.uint16 or a.ndim != 3:
            raise ValueError("frames must be [n,h,w] uint16")
        a = np.ascontiguousarray(a)
        n, h, w = a.shape
        return a, capi.ptr(a), capi.DH_DEPTH_HOST, int(n), int(w), int(h)
    if n is None or w is None or h is None:
        raise ValueError("device_ptr needs n, w and h")
    return None, C.c_void_p(int(device_ptr)), capi.DH_DEPTH_DEVICE, int(n), int(w), int(h)


def frame_args(n: int, intrinsics, midp_guess=None, rot_guess=None, has_midp=None, has_rot=None) -> np.ndarray:
    """capi.FRAME_ARGS_DTYPE[n] for dh_predict_frames.  intrinsics: one IntrinsicMatrix for every frame
    or a float32 [n,3,3] array; midp_guess: float32 [n,3] mm, rot_guess: float64 [n,3] radians, or None;
    has_midp / has_rot: bool [n] masks of the frames whose guess is used (None = every frame)."""
    n = int(n)
    args = np.zeros(n, capi.FRAME_ARGS_DTYPE)
    if isinstance(intrinsics, IntrinsicMatrix):
        args["K"] = intrinsics.mat.reshape(9)
    else:
        k = np.asarray(intrinsics)
        if k.dtype != np.float32 or k.shape != (n, 3, 3):
            raise ValueError("intrinsics must be an IntrinsicMatrix or a float32 [n,3,3] array (n = %d)" % n)
        args["K"] = k.reshape(n, 9)
    for bit, name, guess, dtype, has in ((1, "midp_guess", midp_guess, np.float32, has_midp),
                                         (2, "rot_guess", rot_guess, np.float64, has_rot)):
        if guess is None:
            if has is not None:
                raise ValueError("a mask for %s needs %s" % (name, name))
            continue
        g = np.asarray(guess)
        if g.dtype != dtype or g.shape != (n, 3):
            raise ValueError("%s must be a %s [n,3] array (n = %d)" % (name, np.dtype(dtype).name, n))
        if has is None:
            use = np.ones(n, bool)
        else:
            use = np.asarray(has)
            if use.dtype != np.bool_ or use.shape != (n,):
                raise ValueError("the mask of %s must be a bool [n] array (n = %d)" % (name, n))
        args[name][use] = g[use]
        args["has_guess"][use] |= bit
    return args


def _image_out(out_device_ptr, shape, dtype):
    """(host array or None, pointer, location) of a batch of images: a new host array, or the caller's device memory."""
    if out_device_ptr is None:
        out = np.zeros(shape, dtype)
        return out, capi.ptr(out), capi.DH_DEPTH_HOST
    return None, C.c_void_p(int(out_device_ptr)), capi.DH_DEPTH_DEVICE


class HoughPrediction:
    """prediction.rs:239-256 — the model plus the prediction entry points."""

    def __init__(self, handle: C.c_void_p):
        self._h = handle

    # ---- construction
    @classmethod
    def from_json(cls, text: str | bytes) -> "HoughPrediction":
        """serde_json::from_str::<HoughPrediction> (Readme.md:82-86).  Raises DhError(DH_E_JSON)."""
        data = text.encode("utf-8") if isinstance(text, str) else bytes(text)
        h = C.c_void_p()
        capi.check(capi.load().dh_forest_from_json(data, len(data), C.byref(h)))
        return cls(h)

    @classmethod
    def from_arrays(cls, arr: dict, stepwidth: int, gaussian_sigma: float = 8.0, meanshift_iterations: int = 20,
                    subimage_width: int | None = None, subimage_height: int | None = None) -> "HoughPrediction":
        """Binary structure-of-arrays form (same layout as synth.make_forest) — skips JSON."""
        keep = dict(
            tree_node_off=np.ascontiguousarray(arr["tree_node_off"], np.int64),
            tree_leaf_off=np.ascontiguousarray(arr["tree_leaf_off"], np.int64),
            rects=np.ascontiguousarray(arr["rects"], np.int32),
            threshold=np.ascontiguousarray(arr["threshold"], np.float64),
            child=np.ascontiguousarray(arr["child"], np.int32),
            prob=np.ascontiguousarray(arr["prob"], np.float64),
            vote_off=np.ascontiguousarray(arr["vote_off"], np.int64),
            offsets=np.ascontiguousarray(arr["offsets"], np.float32),
            rotations=np.ascontiguousarray(arr["rotations"], np.float64),
        )
        a = capi.dh_forest_arrays()
        a.stepwidth = int(stepwidth)
        a.subimage_width = int(subimage_width if subimage_width is not None else arr.get("sub_w", 80))
        a.subimage_height = int(subimage_height if subimage_height is not None else arr.get("sub_h", 80))
        a.meanshift_iterations = int(meanshift_iterations)
        a.gaussian_sigma = float(gaussian_sigma)
        a.n_trees = int(arr["n_trees"])
        for k, v in keep.items():
            setattr(a, k, v.ctypes.data)
        h = C.c_void_p()
        capi.check(capi.load().dh_forest_from_arrays(C.byref(a), C.byref(h)))
        return cls(h)

    def to_json(self) -> str:
        """serde_json::to_string(&HoughPrediction) (what hough_tree_trainer.rs:182 writes)."""
        need = C.c_size_t(0)
        capi.check(capi.load().dh_forest_to_json(self._h, None, 0, C.byref(need)))
        buf = C.create_string_buffer(need.value)
        capi.check(capi.load().dh_forest_to_json(self._h, buf, need.value, C.byref(need)))
        return buf.raw[:need.value].decode("utf-8")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            capi.load().dh_forest_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- public fields / accessors of the reference
    @property
    def stepwidth(self) -> int:
        return capi.load().dh_forest_get_stepwidth(self._h)

    @stepwidth.setter
    def stepwidth(self, v: int):
        capi.check(capi.load().dh_forest_set_stepwidth(self._h, int(v)))

    @property
    def meanshift_iterations(self) -> int:
        return capi.load().dh_forest_get_meanshift_iterations(self._h)

    @meanshift_iterations.setter
    def meanshift_iterations(self, v: int):
        capi.check(capi.load().dh_forest_set_meanshift_iterations(self._h, int(v)))

    def sigma(self) -> float:  # prediction.rs:329-331
        return float(capi.load().dh_forest_get_sigma(self._h))

    def update_sigma(self, val: float):  # prediction.rs:320-326
        capi.check(capi.load().dh_forest_set_sigma(self._h, float(val)))

    @property
    def subimage_width(self) -> int:
        return capi.load().dh_forest_get_subimage_width(self._h)

    @property
    def subimage_height(self) -> int:
        return capi.load().dh_forest_get_subimage_height(self._h)

    @property
    def n_trees(self) -> int:
        return capi.load().dh_forest_n_trees(self._h)

    @property
    def n_nodes(self) -> int:
        return capi.load().dh_forest_n_nodes(self._h)

    @property
    def n_leaves(self) -> int:
        return capi.load().dh_forest_n_leaves(self._h)

    @property
    def n_votes(self) -> int:
        return capi.load().dh_forest_n_votes(self._h)

    # ---- prediction
    def predict_parameter_parallel(self, img, intrinsic: IntrinsicMatrix, midp_guess=None, rot_guess=None,
                                   ctx: Context | None = None) -> PredictionResult:
        """prediction.rs:397-409.  img: [h,w] uint16 mm; guesses: None or 3 values (mm / radians)."""
        ctx = ctx or default_context()
        depth = _as_depth(img)
        h, w = depth.shape
        mg = None if midp_guess is None else np.ascontiguousarray(np.asarray(midp_guess, np.float32).reshape(3))
        rg = None if rot_guess is None else np.ascontiguousarray(np.asarray(rot_guess, np.float64).reshape(3))
        res = capi.dh_result()
        capi.check(capi.load().dh_predict(ctx._h, self._h, capi.ptr(depth), w, h, intrinsic._ptr(), capi.ptr(mg),
                                          capi.ptr(rg), C.byref(res)))
        return PredictionResult(np.array(res.mid_point[:], np.float32), np.array(res.rotation[:], np.float64),
                                tuple(res.bounding_box[:]))

    # The single-core variant returns identical results (same leaves in tree order, all later
    # accumulation sequential — prediction.rs:376-388); on the GPU they are the same call.
    predict_parameter = predict_parameter_parallel

    def predict_batch(self, frames, intrinsic: IntrinsicMatrix, ctx: Context | None = None, device_ptr: int | None = None,
                      n: int | None = None, w: int | None = None, h: int | None = None) -> np.ndarray:
        """n independent frames with seeds None.  `frames`: [n,h,w] uint16 host array (pinned
        preferred), or pass device_ptr + (n, w, h) for frames already resident in HBM.
        Returns a structured array (capi.RESULT_DTYPE) with mid_point / rotation per frame."""
        ctx = ctx or default_context()
        if device_ptr is None:
            a = np.asarray(frames)
            if a.dtype != np.uint16 or a.ndim != 3:
                raise ValueError("frames must be [n,h,w] uint16")
            a = np.ascontiguousarray(a)
            n, h, w = a.shape
            p, loc = capi.ptr(a), capi.DH_DEPTH_HOST
        else:
            p, loc = C.c_void_p(int(device_ptr)), capi.DH_DEPTH_DEVICE
        out = np.zeros(int(n), capi.RESULT_DTYPE)
        capi.check(capi.load().dh_predict_batch(ctx._h, self._h, p, int(n), int(w), int(h), intrinsic._ptr(), loc,
                                                capi.ptr(out)))
        return out

    def predict_frames(self, frames, intrinsics, midp_guess=None, rot_guess=None, has_midp=None, has_rot=None,
                       ctx: Context | None = None, device_ptr: int | None = None, n: int | None = None, w: int | None = None,
                       h: int | None = None) -> np.ndarray:
        """predict_parameter_parallel(img_i, K_i, midp_i, rot_i) for n independent frames in one call, equal to
        predict_parameter_parallel frame by frame.  `frames`: [n,h,w] uint16 on the host, or device_ptr +
        (n, w, h).  intrinsics: one IntrinsicMatrix or a float32 [n,3,3] array; midp_guess (float32 [n,3] mm)
        and rot_guess (float64 [n,3] radians) may be None; has_midp / has_rot (bool [n]) pick the frames
        whose guess is used (None = all).  Returns capi.RESULT_DTYPE[n]."""
        _keep, p, loc, n, w, h = _as_frames(frames, device_ptr, n, w, h)
        args = frame_args(n, intrinsics, midp_guess, rot_guess, has_midp, has_rot)
        ctx = ctx or default_context()
        out = np.zeros(n, capi.RESULT_DTYPE)
        capi.check(capi.load().dh_predict_frames(ctx._h, self._h, p, n, w, h, loc, capi.ptr(args), capi.ptr(out)))
        return out

    def predict_sequences(self, frames, intrinsic: IntrinsicMatrix, min_seed_z: float = 500.0, ctx: Context | None = None,
                          device_ptr: int | None = None, n_seq: int | None = None, frames_per_seq: int | None = None,
                          w: int | None = None, h: int | None = None) -> np.ndarray:
        """n_seq independent sequences, every frame seeded with the pose of the frame before it as
        examples/live_prediction.rs:75-88 does (centre seed only if the previous z > min_seed_z).
        `frames`: [n_seq, frames_per_seq, h, w] uint16 on the host, or device_ptr + the four sizes.
        Returns capi.RESULT_DTYPE[n_seq, frames_per_seq]."""
        ctx = ctx or default_context()
        if device_ptr is None:
            a = np.asarray(frames)
            if a.dtype != np.uint16 or a.ndim != 4:
                raise ValueError("frames must be [n_seq, frames_per_seq, h, w] uint16")
            a = np.ascontiguousarray(a)
            n_seq, frames_per_seq, h, w = a.shape
            p, loc = capi.ptr(a), capi.DH_DEPTH_HOST
        else:
            p, loc = C.c_void_p(int(device_ptr)), capi.DH_DEPTH_DEVICE
        out = np.zeros((int(n_seq), int(frames_per_seq)), capi.RESULT_DTYPE)
        capi.check(capi.load().dh_predict_sequences(ctx._h, self._h, p, int(n_seq), int(frames_per_seq), int(w), int(h),
                                                    intrinsic._ptr(), loc, float(min_seed_z), capi.ptr(out)))
        return out

    def predict_mask(self, img, ctx: Context | None = None) -> np.ndarray:
        """prediction.rs:850-905."""
        ctx = ctx or default_context()
        depth = _as_depth(img)
        h, w = depth.shape
        out = np.zeros((h, w), np.uint8)
        capi.check(capi.load().dh_predict_mask(ctx._h, self._h, capi.ptr(depth), w, h, capi.ptr(out)))
        return out

    def hough_image_raw(self, img, intrinsic: IntrinsicMatrix, ctx: Context | None = None) -> np.ndarray:
        """build_hough_image before its gaussian blur (prediction.rs:760-841)."""
        ctx = ctx or default_context()
        depth = _as_depth(img)
        h, w = depth.shape
        out = np.zeros((h, w), np.uint16)
        capi.check(capi.load().dh_hough_image_raw(ctx._h, self._h, capi.ptr(depth), w, h, intrinsic._ptr(), capi.ptr(out)))
        return out

    def build_hough_image(self, img, intrinsic: IntrinsicMatrix, ctx: Context | None = None) -> np.ndarray:
        """prediction.rs:760-845: the 2-D vote image after its gaussian blur (sigma = the model's)."""
        ctx = ctx or default_context()
        depth = _as_depth(img)
        h, w = depth.shape
        out = np.zeros((h, w), np.uint16)
        capi.check(capi.load().dh_build_hough_image(ctx._h, self._h, capi.ptr(depth), w, h, intrinsic._ptr(), capi.ptr(out)))
        return out

    def predict_parameter_from2dhough(self, img, intrinsic: IntrinsicMatrix, ctx: Context | None = None) -> PredictionResult:
        """prediction.rs:343-367: arg-max of the blurred vote image mapped to 3-D; rotation is always 0."""
        ctx = ctx or default_context()
        depth = _as_depth(img)
        h, w = depth.shape
        res = capi.dh_result()
        capi.check(capi.load().dh_predict_from2dhough(ctx._h, self._h, capi.ptr(depth), w, h, intrinsic._ptr(), C.byref(res)))
        return PredictionResult(np.array(res.mid_point[:], np.float32), np.array(res.rotation[:], np.float64),
                                tuple(res.bounding_box[:]))

    # ---- the 2-D entry points over n frames.  Frames: a [n,h,w] uint16 host array, or device_ptr +
    # (n, w, h) for frames resident in HBM.  Images: returned as host arrays, or written to the
    # caller's device memory at out_device_ptr ([n,h,w], nothing returned on the host).
    def predict_mask_batch(self, frames, ctx: Context | None = None, device_ptr: int | None = None, n: int | None = None,
                           w: int | None = None, h: int | None = None, out_device_ptr: int | None = None) -> np.ndarray | None:
        """predict_mask (prediction.rs:850-905) per frame: uint8 [n,h,w]."""
        _keep, p, loc, n, w, h = _as_frames(frames, device_ptr, n, w, h)
        ctx = ctx or default_context()
        out, op, oloc = _image_out(out_device_ptr, (n, h, w), np.uint8)
        capi.check(capi.load().dh_predict_mask_batch(ctx._h, self._h, p, n, w, h, loc, op, oloc))
        return out

    def hough_image_raw_batch(self, frames, intrinsic: IntrinsicMatrix, ctx: Context | None = None, device_ptr: int | None = None,
                              n: int | None = None, w: int | None = None, h: int | None = None,
                              out_device_ptr: int | None = None) -> np.ndarray | None:
        """build_hough_image before its gaussian blur (prediction.rs:760-841) per frame: uint16 [n,h,w]."""
        _keep, p, loc, n, w, h = _as_frames(frames, device_ptr, n, w, h)
        ctx = ctx or default_context()
        out, op, oloc = _image_out(out_device_ptr, (n, h, w), np.uint16)
        capi.check(capi.load().dh_build_hough_image_batch(ctx._h, self._h, p, n, w, h, intrinsic._ptr(), loc, 0, op, oloc, None))
        return out

    def build_hough_image_batch(self, frames, intrinsic: IntrinsicMatrix, ctx: Context | None = None, device_ptr: int | None = None,
                                n: int | None = None, w: int | None = None, h: int | None = None, out_device_ptr: int | None = None,
                                from2d: bool = False):
        """build_hough_image (prediction.rs:760-845) per frame: uint16 [n,h,w] (None with out_device_ptr).
        from2d=True: returns (images, capi.RESULT_DTYPE[n] of predict_parameter_from2dhough) from the same pass."""
        _keep, p, loc, n, w, h = _as_frames(frames, device_ptr, n, w, h)
        ctx = ctx or default_context()
        out, op, oloc = _image_out(out_device_ptr, (n, h, w), np.uint16)
        res = np.zeros(n, capi.RESULT_DTYPE) if from2d else None
        capi.check(capi.load().dh_build_hough_image_batch(ctx._h, self._h, p, n, w, h, intrinsic._ptr(), loc, 1, op, oloc,
                                                          capi.ptr(res)))
        return (out, res) if from2d else out

    def predict_parameter_from2dhough_batch(self, frames, intrinsic: IntrinsicMatrix, ctx: Context | None = None,
                                            device_ptr: int | None = None, n: int | None = None, w: int | None = None,
                                            h: int | None = None) -> np.ndarray:
        """predict_parameter_from2dhough (prediction.rs:343-367) per frame, without copying any image out:
        capi.RESULT_DTYPE[n] (shards with shard.shard_range / gather_results like predict_batch)."""
        _keep, p, loc, n, w, h = _as_frames(frames, device_ptr, n, w, h)
        ctx = ctx or default_context()
        res = np.zeros(n, capi.RESULT_DTYPE)
        capi.check(capi.load().dh_build_hough_image_batch(ctx._h, self._h, p, n, w, h, intrinsic._ptr(), loc, 1, None,
                                                          capi.DH_DEPTH_HOST, capi.ptr(res)))
        return res

    def debug_leaf_static(self, ctx: Context | None = None):
        ctx = ctx or default_context()
        n = self.n_leaves
        v, r, o = np.zeros(n, np.uint32), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        capi.check(capi.load().dh_debug_leaf_static(ctx._h, self._h, capi.ptr(v), capi.ptr(r), capi.ptr(o)))
        return v, r, o
