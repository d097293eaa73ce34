"""Pose and 2-D Hough result of the same frames from one traversal (dh_predict_frames_hough and its Biwi form)
against the two calls a caller makes without them, on the configs[1] forest (10 trees of depth 15, stride 5)
and synthetic 640x480 frames.

    python tools/bench_pose_hough.py [--repeats 3] [--out FILE.jsonl]

Prints (and appends to --out) the GPU name and power limit, then one JSON line per measurement.  The arms
of a comparison run alternately, --repeats times each; their outputs (dh_result bytes, from2d bytes, image
bytes) are asserted equal before anything is timed.
  frames_hbm_from2d   512 frames of 24 calibrations with mixed seeds, resident in HBM, from2d only:
                      dh_predict_frames_hough against dh_predict_frames + dh_build_hough_image_frames
  frames_hbm_images   the same with the blurred images to device memory as well
  biwi_files_from2d   the same frames as Biwi files in host memory, from2d only: dh_predict_frames_hough_biwi
                      against dh_predict_frames_biwi + dh_build_hough_image_frames_biwi
  pose_chunks         what the fused call's smaller chunks (the image scratch's 109 VGA frames instead of 512)
                      cost the pose part: dh_predict_frames on the HBM frames at the default chunk and at 109
  latency             one VGA frame from host memory: dh_predict + dh_predict_from2dhough against
                      dh_predict_frames_hough with n = 1 (dh_predict replays a CUDA graph; the fused call does not)
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_tracks import gpu_info, matrices  # noqa: E402
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth  # noqa: E402
from depthhead_b200.api import frame_args  # noqa: E402


def timed(fn, reps=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5, help="calls per timed sample of the 512-frame workloads")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = open(a.out, "a") if a.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    info = gpu_info()
    bid = capi.load().dh_build_id().decode()
    info["build_id"] = bid
    info["workload"] = "configs[1]: 10 trees depth 15, stride 5, synthetic 640x480 frames"
    emit(info)
    ctx = Context(0)
    hp = HoughPrediction.from_arrays(synth.make_forest(seed=1, n_trees=10, max_depth=15), stepwidth=5)
    L = capi.load()
    P = capi.ptr
    w, h = 640, 480
    D, H = capi.DH_DEPTH_DEVICE, capi.DH_DEPTH_HOST

    def compare(name, arms, outputs, n, reps=1, extra=None):
        """arms: {label: fn}; outputs(): the bytes the last call wrote.  Equal outputs (every destination
        overwritten with 0xFF before each arm), then alternating timings of the calls alone"""
        ref = None
        for k, fn in arms.items():
            res.view(np.uint8).fill(0xFF)
            f2d.view(np.uint8).fill(0xFF)
            if dimg is not None:
                dimg.fill_(-1)
            fn()
            got = outputs()
            assert ref is None or got == ref, (name, k)
            ref = got
        for fn in arms.values():  # (warm-up: every shape and chunk setting of the timed window)
            fn()
        times = {k: [] for k in arms}
        for _ in range(a.repeats):
            for k, fn in arms.items():
                times[k].append(timed(fn, reps))
        for k, ts in times.items():
            emit(dict(name=name, arm=k, frames=n, calls_per_sample=reps, ms_per_call=[1000.0 * t for t in ts],
                      frames_per_s=[n / t for t in ts], outputs_equal=True, build_id=bid, **(extra or {})))

    # ---- 512 frames of 24 calibrations, mixed seeds, in HBM
    n = 512
    frames = synth.make_frames(n, seed=77)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    rng = np.random.default_rng(4)
    Ks = matrices(24)[np.arange(n) % 24]
    mid = rng.uniform(-150.0, 150.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    kind = np.arange(n) % 4
    args = frame_args(n, Ks, mid, rng.uniform(-1.0, 1.0, (n, 3)), (kind & 1) == 1, (kind & 2) == 2)
    K9 = np.ascontiguousarray(args["K"])
    res, f2d = np.zeros(n, capi.RESULT_DTYPE), np.zeros(n, capi.RESULT_DTYPE)
    src = C.c_void_p(dev.data_ptr())
    dimg = torch.empty((n, h, w), dtype=torch.int16, device="cuda")
    for images in (False, True):
        ip = C.c_void_p(dimg.data_ptr()) if images else None

        def outputs():
            return (res.tobytes(), f2d.tobytes()) + ((dimg.cpu().numpy().tobytes(),) if images else ())

        def fused():
            capi.check(L.dh_predict_frames_hough(ctx._h, hp._h, src, n, w, h, D, P(args), P(res), 1, ip, D, P(f2d)))

        def two_calls():
            capi.check(L.dh_predict_frames(ctx._h, hp._h, src, n, w, h, D, P(args), P(res)))
            capi.check(L.dh_build_hough_image_frames(ctx._h, hp._h, src, n, w, h, D, P(K9), 1, ip, D, P(f2d)))

        compare("frames_hbm_images" if images else "frames_hbm_from2d", {"fused": fused, "pose_then_hough": two_calls}, outputs, n,
                a.calls)
    dimg = None

    # ---- the pose part alone at the pose call's chunks and at the fused call's
    def pose_at(chunk):
        def run():
            ctx.set_chunk_frames(chunk)
            try:
                capi.check(L.dh_predict_frames(ctx._h, hp._h, src, n, w, h, D, P(args), P(res)))
            finally:
                ctx.set_chunk_frames(0)
        return run

    compare("pose_chunks", {"chunk_512": pose_at(0), "chunk_109": pose_at(109)}, lambda: res.tobytes(), n, a.calls)

    # ---- the same frames as Biwi files in host memory
    blob, off = biwi.pack_files([biwi.encode_depth(f) for f in frames])

    def b_fused():
        capi.check(L.dh_predict_frames_hough_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(res), 1, None, H, P(f2d)))

    def b_two():
        capi.check(L.dh_predict_frames_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(args), P(res)))
        capi.check(L.dh_build_hough_image_frames_biwi(ctx._h, hp._h, P(blob), P(off), n, w, h, P(K9), 1, None, H, P(f2d)))

    compare("biwi_files_from2d", {"fused": b_fused, "pose_then_hough": b_two}, lambda: (res.tobytes(), f2d.tobytes()), n, a.calls,
            {"blob_bytes": int(off[-1])})
    del dev

    # ---- latency: one VGA host frame
    one = np.ascontiguousarray(frames[5])
    K = IntrinsicMatrix.default_kinect_intrinsic()
    a1 = frame_args(1, K)
    r1, f1 = capi.dh_result(), capi.dh_result()
    rr, ff = np.zeros(1, capi.RESULT_DTYPE), np.zeros(1, capi.RESULT_DTYPE)
    reps = 200

    def single():
        capi.check(L.dh_predict(ctx._h, hp._h, P(one), w, h, K._ptr(), None, None, C.byref(r1)))
        capi.check(L.dh_predict_from2dhough(ctx._h, hp._h, P(one), w, h, K._ptr(), C.byref(f1)))

    def fused1():
        capi.check(L.dh_predict_frames_hough(ctx._h, hp._h, P(one), 1, w, h, H, P(a1), P(rr), 1, None, H, P(ff)))

    single()
    fused1()
    for want, got in ((r1, rr), (f1, ff)):
        want = np.frombuffer(bytes(want), capi.RESULT_DTYPE)
        assert want["mid_point"].tobytes() == got["mid_point"].tobytes() and want["rotation"].tobytes() == got["rotation"].tobytes()
    for _ in range(20):
        single()
        fused1()
    times = {"predict_then_from2dhough": [], "fused_n1": []}
    for _ in range(a.repeats):
        times["predict_then_from2dhough"].append(timed(single, reps))
        times["fused_n1"].append(timed(fused1, reps))
    for k, ts in times.items():
        emit(dict(name="latency_one_vga_host_frame", arm=k, calls_per_sample=reps, ms_per_frame=[1000.0 * t for t in ts],
                  outputs_equal=True, build_id=bid))


if __name__ == "__main__":
    main()
