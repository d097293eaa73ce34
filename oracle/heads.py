"""CPU oracle of several heads per frame (dh_predict_frames_heads, DESIGN.md §7) — TEST INFRASTRUCTURE ONLY.

The rules are restated in ``heads_oracle.cpp``, which includes ``depthhead_oracle.cpp``: the single-head
restatement (seeds, unbounded sparse accumulators, rotation voting, mean-shift) is used as it is.  The
file builds its own library with the flags of ``oracle/Makefile``; forests are created in that library.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from . import OracleForest, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "heads_oracle.cpp")
_DEPS = (_SRC, os.path.join(_HERE, "depthhead_oracle.cpp"))
_LIB_NAME = "libheads_oracle.so"
# the flags of oracle/Makefile: -ffp-contract=off (Rust never fuses mul+add), -fno-fast-math (IEEE semantics)
_CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-Wall", "-Wextra",
             "-Wno-unused-parameter", "-Wno-subobject-linkage"]
_lib = None

# a head as dh_head lays it out, a try as the oracle reports it (the dropped ones too)
HEAD_DTYPE = np.dtype([("mid_point", np.float32, 3), ("_pad", np.uint32), ("rotation", np.float64, 3),
                       ("bounding_box", np.uint32, 4), ("support", np.uint64), ("n_patches", np.uint32),
                       ("seed_cell", np.uint32)], align=True)
TRY_DTYPE = np.dtype([("seed", np.int32, 3), ("centre", np.int32, 3), ("seed_cell", np.uint32), ("support", np.uint64),
                      ("accepted", np.int32), ("cell_votes", np.uint32)], align=True)
assert HEAD_DTYPE.itemsize == 72 and TRY_DTYPE.itemsize == 48


def _stale(path: str) -> bool:
    return not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(d) for d in _DEPS)


def build(force: bool = False) -> str:
    """Compile the library next to its source, or in a temporary directory when the tree is read-only."""
    cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
    for d in (_HERE, os.path.join(tempfile.gettempdir(), "depthhead_heads_oracle_%d" % os.getuid())):
        path = os.path.join(d, _LIB_NAME)
        if not force and not _stale(path):
            return path
        try:
            os.makedirs(d, exist_ok=True)
            tmp = path + ".%d.tmp" % os.getpid()
            subprocess.check_call([cxx] + _CXXFLAGS + ["-shared", "-o", tmp, _SRC])
            os.replace(tmp, path)
            return path
        except (OSError, subprocess.CalledProcessError):
            if d != _HERE:
                raise
    raise RuntimeError("unreachable")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    vp, i32, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_float
    L.orc_forest_new.restype = vp
    L.orc_forest_new.argtypes = [i32] + [vp] * 9
    L.orc_forest_free.argtypes = [vp]
    L.orc_heads_search.restype = C.c_int
    L.orc_heads_search.argtypes = [vp, vp, vp, u64, vp, u32, u32, vp, vp, u32, u32, u32, f32, f32, u32, vp, vp]
    L.orc_predict_heads.restype = C.c_int
    L.orc_predict_heads.argtypes = [vp, u32, u32, u32, f32, u32, vp, u32, u32, vp, vp, vp, u32, u32, f32, C.c_int, vp, vp, vp, vp]
    _lib = L
    return L


def heads_search(guess_pos, mid_keys, mid_vals, depth, K, head0, head0_cell, max_heads, min_cell_votes, radius,
                 sigma=8.0, iterations=20):
    """Rules 2-5 of the head search on given inputs: the 20x20 grid, the centre accumulator as keys [n,3] /
    values [n], the frame (the seeds' depth), head 0's centre and seed cell.  Returns the tries, head 0
    first (TRY_DTYPE)."""
    g = np.ascontiguousarray(guess_pos, np.uint32).reshape(400)
    keys = np.ascontiguousarray(mid_keys, np.int32).reshape(-1, 3)
    vals = np.ascontiguousarray(mid_vals, np.uint32).reshape(-1)
    depth = np.ascontiguousarray(depth, np.uint16)
    h, w = depth.shape
    K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
    c0 = np.ascontiguousarray(head0, np.int32).reshape(3)
    tries = np.zeros(2 * max_heads - 1, TRY_DTYPE)
    n = C.c_uint32()
    lib().orc_heads_search(_p(g), _p(keys), _p(vals), len(vals), _p(depth), w, h, _p(K), _p(c0), int(head0_cell), int(max_heads),
                           int(min_cell_votes), float(radius), float(sigma), int(iterations), _p(tries), C.addressof(n))
    return tries[:n.value]


class HeadsForest:
    """An OracleForest's model in the heads library: predict_heads restates rules 1-7 on one frame."""

    def __init__(self, forest: OracleForest):
        self.f = forest
        a = forest.a
        self._h = lib().orc_forest_new(
            forest.n_trees, _p(a["tree_node_off"]), _p(a["tree_leaf_off"]), _p(a["rects"]), _p(a["threshold"]),
            _p(a["child"]), _p(a["prob"]), _p(a["vote_off"]), _p(a["offsets"]), _p(a["rotations"]))

    @classmethod
    def from_json(cls, text: str) -> "HeadsForest":
        return cls(OracleForest.from_json(text))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().orc_forest_free(self._h)
                self._h = None
        except Exception:
            pass

    def predict_heads(self, depth: np.ndarray, K, max_heads: int, min_cell_votes: int, radius: float, midp_guess=None,
                      rot_guess=None, mode: int = 1):
        """(heads HEAD_DTYPE[max_heads] with unused slots zero, n_heads, tries TRY_DTYPE[...] including the
        dropped ones).  mode: oracle.MODE_NAIVE or oracle.MODE_SAT (default)."""
        f = self.f
        depth = np.ascontiguousarray(depth, np.uint16)
        h, w = depth.shape
        K = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        mg = None if midp_guess is None else np.ascontiguousarray(np.asarray(midp_guess, np.float32))
        rg = None if rot_guess is None else np.ascontiguousarray(np.asarray(rot_guess, np.float64))
        heads = np.zeros(max_heads, HEAD_DTYPE)
        tries = np.zeros(2 * max_heads - 1, TRY_DTYPE)
        nh, nt = C.c_uint32(), C.c_uint32()
        rc = lib().orc_predict_heads(self._h, f.stepwidth, f.subimage_width, f.subimage_height, f.gaussian_sigma,
                                     f.meanshift_iterations, _p(depth), w, h, _p(K), _p(mg), _p(rg), int(max_heads),
                                     int(min_cell_votes), float(radius), int(mode), _p(heads), C.addressof(nh), _p(tries),
                                     C.addressof(nt))
        if rc != 0:
            raise RuntimeError("oracle: predict_heads failed (rc=%d)" % rc)
        return heads, nh.value, tries[:nt.value]
