"""CPU oracle for depthhead's Hough-forest prediction path — TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import this package.  The product (``depthhead_b200``) never does.

The arithmetic lives in ``depthhead_oracle.cpp`` (a C++ restatement citing the reference
file:line for every function).  This module is a ctypes wrapper plus a pure-Python
JSON -> arrays flattener, deliberately independent of the product's C++ JSON loader so a loader
bug cannot hide behind a shared parser.

Parity status: pinned to the reference's unit tests for the linear algebra / intrinsics / Rect
pieces; UNPINNED for the stamm 0.2.0 traversal and the end-to-end pose (the reference has no such
tests and stamm's source is not vendored) — see DESIGN.md.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libdepthhead_oracle.so")
_lib = None

MODE_NAIVE = 0  # faithful: O(area) rectangle sums like types.rs:317-339
MODE_SAT = 1    # summed-area table (same results, asserted in tests)


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (g++ only, a few seconds)."""
    src = os.path.join(_HERE, "depthhead_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH)
    vp, i32, u32, u64, f32, f64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_float, C.c_double
    L.orc_forest_new.restype = vp
    L.orc_forest_new.argtypes = [i32] + [vp] * 9
    L.orc_forest_free.argtypes = [vp]
    L.orc_trace_new.restype = vp
    L.orc_trace_free.argtypes = [vp]
    L.orc_predict.restype = C.c_int
    L.orc_predict.argtypes = [vp, u32, u32, u32, f32, u32, vp, u32, u32, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.orc_trace_error.restype = C.c_char_p
    L.orc_trace_error.argtypes = [vp]
    L.orc_trace_result.argtypes = [vp, vp, vp]
    L.orc_trace_seeds.argtypes = [vp, vp, vp, vp]
    L.orc_trace_dims.argtypes = [vp] + [vp] * 10
    L.orc_trace_patches.argtypes = [vp] + [vp] * 6
    L.orc_trace_grids.argtypes = [vp, vp, vp]
    L.orc_trace_accumulators.argtypes = [vp] + [vp] * 4
    L.orc_trace_meanshift.argtypes = [vp, vp, vp]
    L.orc_predict_batch.restype = C.c_int
    L.orc_predict_batch.argtypes = [vp, u32, u32, u32, f32, u32, vp, u32, u32, u32, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.orc_predict_mask.restype = C.c_int
    L.orc_predict_mask.argtypes = [vp, u32, u32, u32, vp, u32, u32, C.c_int, vp]
    L.orc_hough_image_raw.restype = C.c_int
    L.orc_hough_image_raw.argtypes = [vp, u32, u32, u32, vp, u32, u32, vp, C.c_int, vp]
    L.orc_rect_scale_and_replace.argtypes = [vp, f64, f64, f64, vp]
    L.orc_space_to_img.argtypes = [vp, vp, vp]
    L.orc_img_to_space.argtypes = [vp, vp, f32, vp]
    L.orc_mat3_inv_f32.argtypes = [vp, vp]
    L.orc_mat3_inv_f64.argtypes = [vp, vp]
    L.orc_mat3_det_f64.restype = f64
    L.orc_mat3_det_f64.argtypes = [vp]
    L.orc_mat3_trace_f64.restype = f64
    L.orc_mat3_trace_f64.argtypes = [vp]
    L.orc_mat2_det_f64.restype = f64
    L.orc_mat2_det_f64.argtypes = [vp]
    L.orc_mat2_trace_f64.restype = f64
    L.orc_mat2_trace_f64.argtypes = [vp]
    L.orc_mat2_inv_f64.argtypes = [vp, vp]
    L.orc_mat3_mul_vec3_f64.argtypes = [vp, vp, vp]
    L.orc_mat2_mul_vec2_f64.argtypes = [vp, vp, vp]
    L.orc_mean_cov3_f64.restype = C.c_int
    L.orc_mean_cov3_f64.argtypes = [vp, u64, vp, vp]
    L.orc_mean_cov3_f32.restype = C.c_int
    L.orc_mean_cov3_f32.argtypes = [vp, u64, vp, vp]
    L.orc_mean_cov2_f64.restype = C.c_int
    L.orc_mean_cov2_f64.argtypes = [vp, u64, vp, vp]
    L.orc_build_kernel.argtypes = [u32, f32, vp]
    L.orc_rect_average.restype = f64
    L.orc_rect_average.argtypes = [vp, u32, u32, vp, vp, C.c_int]
    L.orc_leaf_static.argtypes = [vp, C.c_int64, vp, vp, vp]
    L.orc_num_threads.restype = C.c_int
    L.orc_train_binarize.argtypes = [vp, u32, u32, vp, u64, vp, f64, vp]
    L.orc_train_impurity.restype = f64
    L.orc_train_impurity.argtypes = [vp, vp, vp, vp, u64, vp, u64, u64, f64, vp, vp]
    L.orc_train_impurity_from_stats.restype = f64
    L.orc_train_impurity_from_stats.argtypes = [vp, u64, f64, vp]
    L.orc_train_early_stop.restype = C.c_int
    L.orc_train_early_stop.argtypes = [vp, vp, u64, u64, u64, u64]
    L.orc_gaussian_kernel_f32.restype = C.c_int
    L.orc_gaussian_kernel_f32.argtypes = [C.c_float, vp, u32]
    L.orc_gaussian_blur_u16.restype = None
    L.orc_gaussian_blur_u16.argtypes = [vp, u32, u32, C.c_float, vp]
    L.orc_build_hough_image.restype = C.c_int
    L.orc_build_hough_image.argtypes = [vp, u32, u32, u32, C.c_float, vp, u32, u32, vp, C.c_int, vp]
    L.orc_predict_from2dhough.restype = C.c_int
    L.orc_predict_from2dhough.argtypes = [vp, u32, u32, u32, C.c_float, vp, u32, u32, vp, C.c_int, vp, vp]
    L.orc_biwi_read_depth.restype = C.c_int
    L.orc_biwi_read_depth.argtypes = [vp, u64, vp, u64, vp, vp]
    L.orc_biwi_read_gt.restype = C.c_int
    L.orc_biwi_read_gt.argtypes = [vp, u64, vp, vp, vp, vp]
    L.orc_biwi_read_cal.restype = C.c_int
    L.orc_biwi_read_cal.argtypes = [C.c_char_p, u64, vp]
    _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


# ----------------------------------------------------------------------------- JSON -> arrays
def forest_arrays_from_doc(doc: dict) -> dict:
    """Flatten the `forest` sub-object of a HoughPrediction JSON document (schema: DESIGN.md §3,
    the builder-defined stand-in for stamm's unknown serde layout) into flat numpy arrays.
    Leaf/NodeParam/Rect field names follow the reference serde derives
    (houghforest.rs:63-78, types.rs:33-37, meancov_estimation.rs:32-33)."""
    trees = doc["forest"]["trees"]
    node_off, leaf_off = [0], [0]
    rects, thr, child, prob, vote_off, offs, rots = [], [], [], [], [0], [], []
    for t in trees:
        for n in t["nodes"]:
            p = n["param"]
            rects.append(p["r1"]["topleft"] + p["r1"]["bottomright"] + p["r2"]["topleft"] + p["r2"]["bottomright"])
            thr.append(p["threshold"])
            child.append(n["children"])
        for lf in t["leaves"]:
            prob.append(lf["prob"])
            if len(lf["offsets"]) != len(lf["rotations"]):
                raise ValueError("offsets/rotations length mismatch")
            offs.extend(lf["offsets"])
            rots.extend(lf["rotations"])
            vote_off.append(vote_off[-1] + len(lf["offsets"]))
        node_off.append(node_off[-1] + len(t["nodes"]))
        leaf_off.append(leaf_off[-1] + len(t["leaves"]))
    # f32 fields: serde_json parses a number as f64 and narrows to f32 (`as f32`), so go through
    # float64 first.
    return dict(
        n_trees=len(trees),
        tree_node_off=np.asarray(node_off, np.int64),
        tree_leaf_off=np.asarray(leaf_off, np.int64),
        rects=np.asarray(rects, np.int64).reshape(-1, 8),
        threshold=np.asarray(thr, np.float64),
        child=np.asarray(child, np.int32).reshape(-1, 2),
        prob=np.asarray(prob, np.float64),
        vote_off=np.asarray(vote_off, np.int64),
        offsets=np.asarray(offs, np.float64).reshape(-1, 3).astype(np.float32),
        rotations=np.asarray(rots, np.float64).reshape(-1, 3),
    )


@dataclass
class Trace:
    mid_point: np.ndarray
    rotation: np.ndarray
    seed_mid: np.ndarray
    seed_rot: np.ndarray
    seed_rot_deg: np.ndarray
    npx: int = 0
    npy: int = 0
    n_mid_votes: int = 0
    n_rot_votes: int = 0
    valid: np.ndarray | None = None       # [P] u8
    leaf: np.ndarray | None = None        # [P, T] i32 (global leaf id, -1 background)
    visited: np.ndarray | None = None     # [P, T] i32
    p3: np.ndarray | None = None          # [P, 3] f32
    gate: np.ndarray | None = None        # [P] u8
    patch_prob: np.ndarray | None = None  # [P] f64
    guess_pos: np.ndarray | None = None   # [400] u32
    guess_rot: np.ndarray | None = None   # [8000] u32
    mid_keys: np.ndarray | None = None    # [n,3] i32 sorted
    mid_vals: np.ndarray | None = None
    rot_keys: np.ndarray | None = None
    rot_vals: np.ndarray | None = None
    ms_mid: np.ndarray | None = None      # [iters_run, 3]
    ms_rot: np.ndarray | None = None
    ms_mid_zero: bool = False
    ms_rot_zero: bool = False
    extra: dict = field(default_factory=dict)


class OracleForest:
    """Holds the flattened forest + the HoughPrediction scalar fields (prediction.rs:239-256)."""

    def __init__(self, arrays: dict, stepwidth: int, subimage_width: int, subimage_height: int,
                 gaussian_sigma: float, meanshift_iterations: int):
        self.a = {k: (np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v) for k, v in arrays.items()}
        self.stepwidth = int(stepwidth)
        self.subimage_width = int(subimage_width)
        self.subimage_height = int(subimage_height)
        self.gaussian_sigma = float(np.float32(gaussian_sigma))
        self.meanshift_iterations = int(meanshift_iterations)
        a = self.a
        self.n_trees = int(a["n_trees"])
        self._h = lib().orc_forest_new(
            self.n_trees, _p(a["tree_node_off"]), _p(a["tree_leaf_off"]), _p(a["rects"]), _p(a["threshold"]),
            _p(a["child"]), _p(a["prob"]), _p(a["vote_off"]), _p(a["offsets"]), _p(a["rotations"]))

    @classmethod
    def from_json(cls, text: str) -> "OracleForest":
        doc = json.loads(text)
        return cls(forest_arrays_from_doc(doc), doc["stepwidth"], doc["subimage_width"], doc["subimage_height"],
                   doc["gaussian_sigma"], doc["meanshift_iterations"])

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().orc_forest_free(self._h)
                self._h = None
        except Exception:
            pass

    # prediction.rs:320-326 update_sigma
    def update_sigma(self, val: float):
        val = float(np.float32(val))
        if val == self.gaussian_sigma or val <= 0.0:
            return
        self.gaussian_sigma = val

    def predict(self, depth: np.ndarray, K, midp_guess=None, rot_guess=None, mode=MODE_SAT,
                tree_threads=1, keep=True) -> Trace:
        """predict_parameter{,_parallel} (prediction.rs:376-409) with every intermediate."""
        L = lib()
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        mg = None if midp_guess is None else np.ascontiguousarray(np.asarray(midp_guess, np.float32))
        rg = None if rot_guess is None else np.ascontiguousarray(np.asarray(rot_guess, np.float64))
        th = L.orc_trace_new()
        try:
            rc = L.orc_predict(self._h, self.stepwidth, self.subimage_width, self.subimage_height,
                               self.gaussian_sigma, self.meanshift_iterations, _p(depth), w, h, _p(K), _p(mg),
                               _p(rg), int(mode), int(tree_threads), int(bool(keep)), th)
            if rc != 0:
                raise RuntimeError("oracle: %s (rc=%d)" % (L.orc_trace_error(th).decode(), rc))
            mid = np.zeros(3, np.float32)
            rot = np.zeros(3, np.float64)
            L.orc_trace_result(th, _p(mid), _p(rot))
            sm, sr, srd = np.zeros(3, np.int32), np.zeros(3, np.int32), np.zeros(3, np.float64)
            L.orc_trace_seeds(th, _p(sm), _p(sr), _p(srd))
            tr = Trace(mid, rot, sm, sr, srd)
            npx, npy = C.c_uint32(), C.c_uint32()
            nmv, nrv, nmc, nrc = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
            nmm, nmr = C.c_uint32(), C.c_uint32()
            zm, zr = C.c_int32(), C.c_int32()
            L.orc_trace_dims(th, *[C.addressof(x) for x in (npx, npy, nmv, nrv, nmc, nrc, nmm, nmr, zm, zr)])
            tr.npx, tr.npy = npx.value, npy.value
            tr.n_mid_votes, tr.n_rot_votes = nmv.value, nrv.value
            tr.ms_mid_zero, tr.ms_rot_zero = bool(zm.value), bool(zr.value)
            tr.ms_mid = np.zeros((nmm.value, 3), np.int32)
            tr.ms_rot = np.zeros((nmr.value, 3), np.int32)
            L.orc_trace_meanshift(th, _p(tr.ms_mid), _p(tr.ms_rot))
            tr.guess_pos = np.zeros(400, np.uint32)
            tr.guess_rot = np.zeros(8000, np.uint32)
            L.orc_trace_grids(th, _p(tr.guess_pos), _p(tr.guess_rot))
            if keep:
                P, T = tr.npx * tr.npy, self.n_trees
                tr.valid = np.zeros(P, np.uint8)
                tr.leaf = np.zeros((P, T), np.int32)
                tr.visited = np.zeros((P, T), np.int32)
                tr.p3 = np.zeros((P, 3), np.float32)
                tr.gate = np.zeros(P, np.uint8)
                tr.patch_prob = np.zeros(P, np.float64)
                L.orc_trace_patches(th, _p(tr.valid), _p(tr.leaf), _p(tr.visited), _p(tr.p3), _p(tr.gate),
                                    _p(tr.patch_prob))
                tr.mid_keys = np.zeros((nmc.value, 3), np.int32)
                tr.mid_vals = np.zeros(nmc.value, np.uint32)
                tr.rot_keys = np.zeros((nrc.value, 3), np.int32)
                tr.rot_vals = np.zeros(nrc.value, np.uint32)
                L.orc_trace_accumulators(th, _p(tr.mid_keys), _p(tr.mid_vals), _p(tr.rot_keys), _p(tr.rot_vals))
            return tr
        finally:
            L.orc_trace_free(th)

    def predict_batch(self, depth: np.ndarray, K, mode=MODE_NAIVE, tree_threads=1, frame_threads=1):
        """Results only, for the CPU baseline.  Returns (mid_points[n,3] f32, rotations[n,3] f64, evals)."""
        L = lib()
        depth = np.ascontiguousarray(depth, np.uint16)
        n, h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        mid = np.zeros((n, 3), np.float32)
        rot = np.zeros((n, 3), np.float64)
        ev = C.c_uint64()
        rc = L.orc_predict_batch(self._h, self.stepwidth, self.subimage_width, self.subimage_height,
                                 self.gaussian_sigma, self.meanshift_iterations, _p(depth), n, w, h, _p(K),
                                 int(mode), int(tree_threads), int(frame_threads), _p(mid), _p(rot),
                                 C.addressof(ev))
        if rc != 0:
            raise RuntimeError("oracle batch failed rc=%d" % rc)
        return mid, rot, ev.value

    def predict_mask(self, depth: np.ndarray, mode=MODE_SAT) -> np.ndarray:
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        out = np.zeros((h, w), np.uint8)
        rc = lib().orc_predict_mask(self._h, self.stepwidth, self.subimage_width, self.subimage_height, _p(depth),
                                    w, h, int(mode), _p(out))
        if rc != 0:
            raise RuntimeError("oracle predict_mask rc=%d" % rc)
        return out

    def hough_image_raw(self, depth: np.ndarray, K, mode=MODE_SAT) -> np.ndarray:
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        out = np.zeros((h, w), np.uint16)
        rc = lib().orc_hough_image_raw(self._h, self.stepwidth, self.subimage_width, self.subimage_height,
                                       _p(depth), w, h, _p(K), int(mode), _p(out))
        if rc != 0:
            raise RuntimeError("oracle hough_image_raw rc=%d" % rc)
        return out

    def build_hough_image(self, depth: np.ndarray, K, mode=MODE_SAT) -> np.ndarray:
        """build_hough_image (prediction.rs:760-845) including its gaussian blur (imageproc: unpinned)"""
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        out = np.zeros((h, w), np.uint16)
        rc = lib().orc_build_hough_image(self._h, self.stepwidth, self.subimage_width, self.subimage_height,
                                         self.gaussian_sigma, _p(depth), w, h, _p(K), int(mode), _p(out))
        if rc != 0:
            raise RuntimeError("oracle build_hough_image rc=%d" % rc)
        return out

    def predict_parameter_from2dhough(self, depth: np.ndarray, K, mode=MODE_SAT):
        """prediction.rs:343-367 -> (mid_point[3] f32, (x, y) of the winning pixel)"""
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        mid = np.zeros(3, np.float32)
        xy = np.zeros(2, np.uint32)
        rc = lib().orc_predict_from2dhough(self._h, self.stepwidth, self.subimage_width, self.subimage_height,
                                           self.gaussian_sigma, _p(depth), w, h, _p(K), int(mode), _p(mid), _p(xy))
        if rc != 0:
            raise RuntimeError("oracle predict_parameter_from2dhough rc=%d" % rc)
        return mid, (int(xy[0]), int(xy[1]))

    def leaf_static(self, leaf: int):
        v, tr, to = C.c_uint32(), C.c_double(), C.c_float()
        lib().orc_leaf_static(self._h, int(leaf), C.addressof(v), C.addressof(tr), C.addressof(to))
        return v.value, tr.value, to.value


def gaussian_kernel_f32(sigma: float) -> np.ndarray:
    """imageproc's gaussian_kernel_f32 as restated in the oracle (unpinned, see depthhead_oracle.cpp)"""
    n = lib().orc_gaussian_kernel_f32(float(sigma), None, 0)
    out = np.zeros(n, np.float32)
    lib().orc_gaussian_kernel_f32(float(sigma), _p(out), n)
    return out


def gaussian_blur_u16(img: np.ndarray, sigma: float) -> np.ndarray:
    a = np.ascontiguousarray(img, np.uint16)
    h, w = a.shape
    out = np.zeros((h, w), np.uint16)
    lib().orc_gaussian_blur_u16(_p(a), w, h, float(sigma), _p(out))
    return out


def num_threads() -> int:
    return lib().orc_num_threads()


# ----------------------------------------------------------------------------- Biwi wire formats
class BiwiError(RuntimeError):
    """code 1: UnexpectedEof / Unsupported Calibration-File, 2: panic or ParseFloatError, 3: see message"""

    def __init__(self, code: int, what: str):
        super().__init__("%s (code %d)" % (what, code))
        self.code = code


def biwi_read_depth(data: bytes) -> np.ndarray:
    """read_depth (src/db_reader/biwi.rs:81-103) -> [h, w] uint16."""
    buf = np.frombuffer(bytes(data), np.uint8)
    if buf.size < 8:
        raise BiwiError(1, "read_depth: UnexpectedEof in the header")
    w, h = (int(x) for x in np.frombuffer(buf[:8].tobytes(), "<u4"))
    npx = (w * h) & 0xFFFFFFFF
    if npx > (1 << 28):
        raise BiwiError(3, "read_depth: oracle refuses frames over 2^28 pixels")
    out = np.zeros(max(npx, 1), np.uint16)
    wo, ho = C.c_uint32(0), C.c_uint32(0)
    rc = lib().orc_biwi_read_depth(_p(buf), buf.size, _p(out), out.size, C.byref(wo), C.byref(ho))
    if rc:
        raise BiwiError(rc, "read_depth: " + {1: "UnexpectedEof", 2: "run past the last pixel (panic)", 3: "buffer"}[rc])
    return out[:npx].reshape(h, w)


def biwi_read_gt(data: bytes, K) -> tuple:
    """read_gt (biwi.rs:63-77) -> (pos3d[3], pos2d[2], rot[3]) float32."""
    buf = np.frombuffer(bytes(data), np.uint8)
    k = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
    p3, p2, rot = np.zeros(3, np.float32), np.zeros(2, np.float32), np.zeros(3, np.float32)
    rc = lib().orc_biwi_read_gt(_p(buf) if buf.size else None, buf.size, _p(k), _p(p3), _p(p2), _p(rot))
    if rc:
        raise BiwiError(rc, "read_gt: UnexpectedEof")
    return p3, p2, rot


def biwi_read_cal(text: str | bytes) -> np.ndarray:
    """read_cal (biwi.rs:27-60) -> 3x3 float32."""
    b = text.encode() if isinstance(text, str) else bytes(text)
    K = np.zeros(9, np.float32)
    rc = lib().orc_biwi_read_cal(b, len(b), _p(K))
    if rc:
        raise BiwiError(rc, "read_cal: " + {1: "Unsupported Calibration-File", 2: "ParseFloatError", 3: "fourth number on a line (panic)"}[rc])
    return K.reshape(3, 3)


# ----------------------------------------------------------------------------- training callbacks
SIDE_DTYPE = np.dtype([("n", np.uint64), ("n_pos", np.uint64), ("det_off", np.float64), ("det_rot", np.float64)])


def train_binarize(patches: np.ndarray, idx, rects8, threshold: float) -> np.ndarray:
    """binarize (houghforest.rs:185-193) of one NodeParam on the samples idx -> u8 bits."""
    p = np.ascontiguousarray(patches, np.uint16)
    i = np.ascontiguousarray(idx, np.uint32)
    r = np.ascontiguousarray(rects8, np.int32).reshape(8)
    bits = np.zeros(len(i), np.uint8)
    lib().orc_train_binarize(_p(p), p.shape[2], p.shape[1], _p(i), len(i), _p(r), float(threshold), _p(bits))
    return bits


def train_impurity(is_object, offsets, rotations, left, right, depth: int, steepness: float):
    """impurity (houghforest.rs:250-295) -> (value, per-side stats SIDE_DTYPE[2], hit_unreachable)."""
    o = np.ascontiguousarray(is_object, np.uint8)
    of = np.ascontiguousarray(offsets, np.float32)
    ro = np.ascontiguousarray(rotations, np.float64)
    le, ri = np.ascontiguousarray(left, np.uint32), np.ascontiguousarray(right, np.uint32)
    st = np.zeros(2, SIDE_DTYPE)
    bad = C.c_int(0)
    v = lib().orc_train_impurity(_p(o), _p(of), _p(ro), _p(le), len(le), _p(ri), len(ri), int(depth), float(steepness), _p(st),
                                 C.byref(bad))
    return float(v), st, bool(bad.value)


def train_impurity_from_stats(stats, depth: int, steepness: float) -> float:
    st = np.ascontiguousarray(stats, SIDE_DTYPE)
    return float(lib().orc_train_impurity_from_stats(_p(st), int(depth), float(steepness), None))


def train_early_stop(is_object, idx, depth: int, max_depth: int, min_subset_size: int) -> bool:
    o = np.ascontiguousarray(is_object, np.uint8)
    i = np.ascontiguousarray(idx, np.uint32)
    return bool(lib().orc_train_early_stop(_p(o), _p(i), len(i), int(depth), int(max_depth), int(min_subset_size)))


def train_feature(patch: np.ndarray, rects8) -> float:
    """avg1 - avg2 of binarize (houghforest.rs:185-193) on one patch [sh, sw]: the value a threshold
    ties with."""
    p = np.ascontiguousarray(patch, np.uint16)
    sh, sw = p.shape
    sub = np.array([0, 0, sw, sh], np.uint32)
    r = np.asarray(rects8, np.int64).reshape(8)
    a = [lib().orc_rect_average(_p(p), sw, sh, _p(sub), _p(np.ascontiguousarray(r[k:k + 4], np.uint32)), MODE_NAIVE) for k in (0, 4)]
    return a[0] - a[1]


# the layout of dh_split_stats (include/depthhead_cuda.h), restated so that the oracle does not import the product
TRAIN_STATS_DTYPE = np.dtype([("n", np.uint32, 2), ("n_pos", np.uint32, 2), ("det_off", np.float64, 2), ("det_rot", np.float64, 2),
                              ("impurity", np.float64)], align=True)


class OracleTrainSet:
    """A training set scored on the CPU, with the attributes `depthhead_b200.train.HoughLearning.train_tree`
    uses (`n`, `is_object`, `offsets`, `rotations`, `score_level`, `split_level`): every candidate is
    scored with `train_binarize` and `train_impurity`, and its impurity is NaN where a side is empty
    or the reference hits unreachable!() — the candidates the trainer skips (DESIGN.md §9).  So
    `HoughLearning(...).train_forest(OracleTrainSet(...), CounterRng(seed))` grows a forest without
    the GPU, with the same driver and random stream as the product.

    After each `score_level`, `last_bad` [n_nodes, m] flags the unreachable!() candidates and
    `last_value` holds the impurity the reference computes before its checks."""

    def __init__(self, patches, is_object, offsets, rotations):
        self.patches = np.ascontiguousarray(patches, np.uint16)
        if self.patches.ndim != 3:
            raise ValueError("patches must be [n, sub_h, sub_w] uint16")
        self.n = len(self.patches)
        self.is_object = np.ascontiguousarray(is_object, np.uint8).reshape(self.n)
        self.offsets = np.ascontiguousarray(offsets, np.float32).reshape(self.n, 3)
        self.rotations = np.ascontiguousarray(rotations, np.float64).reshape(self.n, 3)
        self.last_bad = self.last_value = None

    def close(self):
        pass

    def score_level(self, sample_idx, node_off, cand_rects, cand_thr, depth: int, steepness: float) -> np.ndarray:
        idx = np.asarray(sample_idx, np.uint32)
        off = np.asarray(node_off, np.int64)
        k = len(off) - 1
        thr = np.asarray(cand_thr, np.float64).reshape(k, -1)
        m = thr.shape[1]
        rects = np.asarray(cand_rects, np.int32).reshape(k, m, 8)
        out = np.zeros((k, m), TRAIN_STATS_DTYPE)
        self.last_bad = np.zeros((k, m), bool)
        self.last_value = np.zeros((k, m), np.float64)
        for a in range(k):
            s = idx[off[a]:off[a + 1]]
            for j in range(m):
                bits = train_binarize(self.patches, s, rects[a, j], thr[a, j])
                left, right = s[bits == 0], s[bits != 0]
                v, st, bad = train_impurity(self.is_object, self.offsets, self.rotations, left, right, depth, steepness)
                o = out[a, j]
                o["n"], o["n_pos"] = st["n"], st["n_pos"]
                o["det_off"], o["det_rot"] = st["det_off"], st["det_rot"]
                o["impurity"] = np.nan if (len(left) == 0 or len(right) == 0 or bad) else v
                self.last_bad[a, j], self.last_value[a, j] = bad, v
        return out

    def split_level(self, sample_idx, node_off, rects, thr) -> np.ndarray:
        idx = np.asarray(sample_idx, np.uint32)
        off = np.asarray(node_off, np.int64)
        r = np.asarray(rects, np.int32).reshape(-1, 8)
        t = np.asarray(thr, np.float64).reshape(-1)
        bits = np.zeros(int(off[-1]), np.uint8)
        for a in range(len(off) - 1):
            bits[off[a]:off[a + 1]] = train_binarize(self.patches, idx[off[a]:off[a + 1]], r[a], t[a])
        return bits
