"""Biwi Kinect Head Pose Database wire formats (reference: src/db_reader/biwi.rs).

Host-side mirror of the reference reader for the prediction path: `read_cal`, `read_gt` and
`read_depth` keep their names; `read_depth` and `predict_files` expand the run-length coded frames
on the GPU (the compressed bytes are what crosses PCIe).  `encode_depth` / `pack_files` exist
because the database itself is not available offline: they write synthetic frames in the same
format (the reference only reads it)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .api import (Context, HoughPrediction, IntrinsicMatrix, _image_out, _track_offsets, default_context, frame_args,
                  intrinsic_array)


def encode_depth(img: np.ndarray) -> bytes:
    """[h, w] uint16 -> the byte stream read_depth (biwi.rs:81-103) expects: u32 w, u32 h, then
    [u32 n_empty][u32 n_full][n_full x u16] until every pixel is covered (little endian).  Runs
    cross row boundaries, as in the database's files."""
    a = np.ascontiguousarray(img, dtype=np.uint16)
    h, w = a.shape
    flat = a.reshape(-1)
    nz = flat != 0
    # run boundaries of the zero / non-zero mask
    edges = np.flatnonzero(np.diff(nz.astype(np.int8))) + 1
    starts = np.concatenate(([0], edges))
    ends = np.concatenate((edges, [flat.size]))
    parts = [np.array([w, h], "<u4").tobytes()]
    i = 0
    n_runs = len(starts)
    while i < n_runs:
        if nz[starts[i]]:          # file starts with pixels: an empty run of length 0 first
            n_empty, full = 0, (starts[i], ends[i])
            i += 1
        else:
            n_empty = ends[i] - starts[i]
            if i + 1 < n_runs:
                full = (starts[i + 1], ends[i + 1])
                i += 2
            else:
                full = (ends[i], ends[i])
                i += 1
        parts.append(np.array([n_empty, full[1] - full[0]], "<u4").tobytes())
        parts.append(flat[full[0]:full[1]].astype("<u2").tobytes())
    return b"".join(parts)


def encode_frames(frames: np.ndarray, threads: int = 0) -> tuple:
    """[n, h, w] uint16 -> (blob, offsets) through the library's own multi-threaded writer
    (dh_biwi_encode_depth: the encoder dh_predict_batch runs for host frames; runs at a
    granularity of 16 pixels, so isolated zeros travel as literal zeros).  Host-only."""
    a = np.ascontiguousarray(frames, dtype=np.uint16)
    if a.ndim != 3:
        raise ValueError("frames must be [n, h, w] uint16")
    n, h, w = a.shape
    L = capi.load()
    offsets = np.zeros(n + 1, np.uint64)
    need = C.c_size_t(0)
    cap = int(L.dh_biwi_encode_bound(w, h)) * n + 16
    blob = np.zeros(cap, np.uint8)
    capi.check(L.dh_biwi_encode_depth(capi.ptr(a) if n else None, n, w, h, int(threads), capi.ptr(blob), cap, capi.ptr(offsets),
                                      C.byref(need)))
    return blob[:need.value].copy(), offsets


def pack_files(files) -> tuple:
    """Concatenate compressed depth files into the blob + offsets the C ABI takes (every file
    starts at a multiple of 16 bytes)."""
    offsets = np.zeros(len(files) + 1, np.uint64)
    chunks = []
    pos = 0
    for i, f in enumerate(files):
        offsets[i] = pos
        pad = (-len(f)) % 16
        chunks.append(bytes(f) + b"\0" * pad)
        pos += len(f) + pad
    offsets[len(files)] = pos
    blob = np.frombuffer(b"".join(chunks) + b"\0" * 16, np.uint8).copy()
    return blob, offsets


def depth_dims(data: bytes) -> tuple:
    buf = np.frombuffer(bytes(data), np.uint8)
    w, h = C.c_uint32(0), C.c_uint32(0)
    capi.check(capi.load().dh_biwi_depth_dims(capi.ptr(buf) if buf.size else None, buf.size, C.byref(w), C.byref(h)))
    return int(w.value), int(h.value)


def read_depth(files, ctx: Context | None = None) -> np.ndarray:
    """read_depth (biwi.rs:81-103) for one file (bytes -> [h, w]) or a list of files of one size
    (-> [n, h, w]), expanded on the GPU."""
    single = isinstance(files, (bytes, bytearray, memoryview))
    lst = [files] if single else list(files)
    ctx = ctx or default_context()
    if not lst:
        return np.zeros((0, 0, 0), np.uint16)
    w, h = depth_dims(lst[0])
    blob, offsets = pack_files(lst)
    out = np.zeros((len(lst), h, w), np.uint16)
    capi.check(capi.load().dh_biwi_decode_depth(ctx._h, capi.ptr(blob), capi.ptr(offsets), len(lst), w, h, capi.ptr(out),
                                                capi.DH_DEPTH_HOST))
    return out[0] if single else out


def read_cal(text) -> IntrinsicMatrix:
    """read_cal (biwi.rs:27-60): depth.cal -> IntrinsicMatrix."""
    b = text.encode() if isinstance(text, str) else bytes(text)
    K = np.zeros(9, np.float32)
    capi.check(capi.load().dh_biwi_parse_cal(b, len(b), capi.ptr(K)))
    return IntrinsicMatrix(K.reshape(3, 3))


def read_gt(data: bytes, intrinsic: IntrinsicMatrix) -> dict:
    """read_gt (biwi.rs:63-77): HeadTransformation {pos3d, pos2d, rot}."""
    buf = np.frombuffer(bytes(data), np.uint8)
    p3, p2, rot = np.zeros(3, np.float32), np.zeros(2, np.float32), np.zeros(3, np.float32)
    capi.check(capi.load().dh_biwi_parse_pose(capi.ptr(buf) if buf.size else None, buf.size, intrinsic._ptr(), capi.ptr(p3),
                                              capi.ptr(p2), capi.ptr(rot)))
    return {"pos3d": p3, "pos2d": p2, "rot": rot}


def predict_files(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, w: int, h: int, intrinsic,
                  ctx: Context | None = None, midp_guess=None, rot_guess=None, has_midp=None, has_rot=None) -> np.ndarray:
    """read_depth + predict_parameter_parallel(img, K, None, None) per file
    (examples/db_evaluate.rs:296), the decode on the GPU.  Returns capi.RESULT_DTYPE[n].
    intrinsic: one IntrinsicMatrix for every file, or a float32 [n,3,3] array with the K of every file
    (a database of several sequence folders, each with its own depth.cal); with such an array or with
    seeds (see HoughPrediction.predict_frames) every file is predicted with its own arguments."""
    n = len(offsets) - 1
    per_frame = not isinstance(intrinsic, IntrinsicMatrix) or midp_guess is not None or rot_guess is not None
    args = frame_args(n, intrinsic, midp_guess, rot_guess, has_midp, has_rot) if per_frame else None
    if not per_frame and (has_midp is not None or has_rot is not None):
        raise ValueError("a guess mask needs its guesses")
    ctx = ctx or default_context()
    out = np.zeros(n, capi.RESULT_DTYPE)
    offsets = np.ascontiguousarray(offsets, np.uint64)
    if per_frame:
        capi.check(capi.load().dh_predict_frames_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h),
                                                      capi.ptr(args), capi.ptr(out)))
        return out
    capi.check(capi.load().dh_predict_batch_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h),
                                                 intrinsic._ptr(), capi.ptr(out)))
    return out


def build_hough_image_files(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, w: int, h: int, intrinsics, blur: bool = True,
                            from2d: bool = False, images: bool = True, ctx: Context | None = None, out_device_ptr: int | None = None):
    """read_depth + build_hough_image (blur=True; blur=False: the vote image before its blur) per file,
    every file with its own K (examples/db_prediction.rs:154 over a database of several sequence folders),
    the decode on the GPU.  intrinsics: one IntrinsicMatrix or a float32 [n,3,3] array.  Returns uint16
    [n,h,w] (None with out_device_ptr or images=False); from2d=True (needs blur): (images,
    capi.RESULT_DTYPE[n] of predict_parameter_from2dhough)."""
    n = len(offsets) - 1
    Ks = intrinsic_array(n, intrinsics)
    ctx = ctx or default_context()
    out, op, oloc = _image_out(out_device_ptr, (n, int(h), int(w)), np.uint16) if images else (None, None, capi.DH_DEPTH_HOST)
    res = np.zeros(n, capi.RESULT_DTYPE) if from2d else None
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_build_hough_image_frames_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h),
                                                            capi.ptr(Ks), int(bool(blur)), op, oloc, capi.ptr(res)))
    return (out, res) if from2d else out


def predict_mask_files(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, w: int, h: int, ctx: Context | None = None,
                       out_device_ptr: int | None = None) -> np.ndarray | None:
    """read_depth + predict_mask per file, the decode on the GPU: uint8 [n,h,w] (None with out_device_ptr)."""
    n = len(offsets) - 1
    ctx = ctx or default_context()
    out, op, oloc = _image_out(out_device_ptr, (n, int(h), int(w)), np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_predict_mask_batch_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h), op, oloc))
    return out


def predict_track_files(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, lengths, w: int, h: int, intrinsics,
                        midp_guess=None, rot_guess=None, has_midp=None, has_rot=None, min_seed_z: float = 500.0,
                        ctx: Context | None = None) -> np.ndarray:
    """HoughPrediction.predict_tracks over Biwi files: track s is the next lengths[s] files (in time order),
    with intrinsics[s] (one IntrinsicMatrix or a float32 [n_seq,3,3] array, e.g. the depth.cal of every
    sequence folder) and optional seeds of its first frame.  The decode runs on the GPU.  Returns
    capi.RESULT_DTYPE[n] in file order; a damaged file is DH_E_ARG naming the lowest bad file."""
    seq_off, n_seq, total = _track_offsets(lengths)
    n = len(offsets) - 1
    if n != total:
        raise ValueError("sum(lengths) = %d but there are %d files" % (total, n))
    args = frame_args(n_seq, intrinsics, midp_guess, rot_guess, has_midp, has_rot)
    ctx = ctx or default_context()
    out = np.zeros(n, capi.RESULT_DTYPE)
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_predict_tracks_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n_seq, capi.ptr(seq_off),
                                                  int(w), int(h), capi.ptr(args), float(min_seed_z), capi.ptr(out)))
    return out


def predict_files_with_mask(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, w: int, h: int, intrinsic,
                            ctx: Context | None = None, midp_guess=None, rot_guess=None, has_midp=None, has_rot=None,
                            mask_device_ptr: int | None = None):
    """read_depth + pose and head mask per file from one traversal, the decode on the GPU: (capi.RESULT_DTYPE[n],
    uint8 [n,h,w] or None with mask_device_ptr), equal to predict_files and predict_mask_files.  intrinsic: one
    IntrinsicMatrix (repeated for every file) or a float32 [n,3,3] array; seeds as in predict_files."""
    n = len(offsets) - 1
    args = frame_args(n, intrinsic, midp_guess, rot_guess, has_midp, has_rot)
    ctx = ctx or default_context()
    out = np.zeros(n, capi.RESULT_DTYPE)
    masks, mp, mloc = _image_out(mask_device_ptr, (n, int(h), int(w)), np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_predict_frames_mask_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h),
                                                       capi.ptr(args), capi.ptr(out), mp, mloc))
    return out, masks


def predict_track_files_with_mask(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, lengths, w: int, h: int, intrinsics,
                                  midp_guess=None, rot_guess=None, has_midp=None, has_rot=None, min_seed_z: float = 500.0,
                                  ctx: Context | None = None, mask_device_ptr: int | None = None):
    """predict_track_files plus the head mask of every file from the same traversal: (capi.RESULT_DTYPE[n],
    uint8 [n,h,w] or None with mask_device_ptr), both in file order."""
    seq_off, n_seq, total = _track_offsets(lengths)
    n = len(offsets) - 1
    if n != total:
        raise ValueError("sum(lengths) = %d but there are %d files" % (total, n))
    args = frame_args(n_seq, intrinsics, midp_guess, rot_guess, has_midp, has_rot)
    ctx = ctx or default_context()
    out = np.zeros(n, capi.RESULT_DTYPE)
    masks, mp, mloc = _image_out(mask_device_ptr, (n, int(h), int(w)), np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_predict_tracks_mask_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n_seq, capi.ptr(seq_off),
                                                       int(w), int(h), capi.ptr(args), float(min_seed_z), capi.ptr(out), mp, mloc))
    return out, masks


def predict_files_with_hough(hp: HoughPrediction, blob: np.ndarray, offsets: np.ndarray, w: int, h: int, intrinsic,
                             ctx: Context | None = None, midp_guess=None, rot_guess=None, has_midp=None, has_rot=None,
                             blur: bool = True, image: bool = True, from2d: bool = True, hough_device_ptr: int | None = None):
    """read_depth + pose and 2-D Hough result per file from one traversal, the decode on the GPU
    (examples/db_prediction.rs:140,154): (capi.RESULT_DTYPE[n], uint16 [n,h,w] or None, capi.RESULT_DTYPE[n]
    or None), equal to predict_files and build_hough_image_files with every file's K.  intrinsic: one
    IntrinsicMatrix (repeated for every file) or a float32 [n,3,3] array; seeds as in predict_files (they act
    on the poses only); blur, image and from2d as in HoughPrediction.predict_frames_with_hough."""
    if hough_device_ptr is not None and not image:
        raise ValueError("hough_device_ptr needs image=True")
    n = len(offsets) - 1
    args = frame_args(n, intrinsic, midp_guess, rot_guess, has_midp, has_rot)
    ctx = ctx or default_context()
    out = np.zeros(n, capi.RESULT_DTYPE)
    images, ip, iloc = _image_out(hough_device_ptr, (n, int(h), int(w)), np.uint16) if image else (None, None, capi.DH_DEPTH_HOST)
    res = np.zeros(n, capi.RESULT_DTYPE) if from2d else None
    offsets = np.ascontiguousarray(offsets, np.uint64)
    capi.check(capi.load().dh_predict_frames_hough_biwi(ctx._h, hp._h, capi.ptr(blob), capi.ptr(offsets), n, int(w), int(h),
                                                        capi.ptr(args), capi.ptr(out), int(bool(blur)), ip, iloc, capi.ptr(res)))
    return out, images, res
