"""Pose and head mask of the same frames from one traversal (dh_predict_frames_mask, dh_predict_tracks_mask)
against the two calls a caller makes without them, on the configs[1] forest (10 trees of depth 15, stride 5)
and synthetic 640x480 frames.

    python tools/bench_pose_mask.py [--repeats 3] [--out FILE.jsonl]

Prints (and appends to --out) the GPU name and power limit, then one JSON line per measurement.  The two
arms of a comparison run alternately, --repeats times each; their outputs (dh_result bytes, mask bytes) are
asserted equal before anything is timed.
  frames    512 frames of 24 calibrations with mixed seeds, resident in HBM: dh_predict_frames_mask
            against dh_predict_frames + dh_predict_mask_batch, masks to device memory and to host memory
  tracks    24 Biwi-shaped tracks (the lengths of tools/bench_tracks.py divided by 4, 100-225 frames,
            ~3 900 in all), 24 matrices, in HBM and as Biwi files in host memory, masks to device memory:
            dh_predict_tracks_mask(_biwi) against dh_predict_tracks(_biwi) + dh_predict_mask_batch(_biwi)
  latency   one VGA frame from host memory, mask to host memory: dh_predict + dh_predict_mask against
            dh_predict_frames_mask with n = 1 (dh_predict replays a CUDA graph; the fused call does not)
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

from bench_tracks import gpu_info, make_frames, matrices  # noqa: E402
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth  # noqa: E402
from depthhead_b200.api import _track_offsets, frame_args  # noqa: E402


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
    w, h, px = 640, 480, 640 * 480

    def compare(name, arms, n, extra=None):
        """arms: {label: fn}, each returning (results, masks); equal outputs, then alternating timings"""
        outs = {k: fn() for k, fn in arms.items()}
        ref = next(iter(outs.values()))
        for k, (r, m) in outs.items():
            assert r.tobytes() == ref[0].tobytes(), (name, k, "results")
            assert torch.equal(torch.as_tensor(m), torch.as_tensor(ref[1])), (name, k, "masks")
        times = {k: [] for k in arms}
        for _ in range(a.repeats):
            for k, fn in arms.items():
                times[k].append(timed(fn))
        for k, ts in times.items():
            emit(dict(name=name, arm=k, frames=n, ms_per_call=[1000.0 * t for t in ts], frames_per_s=[n / t for t in ts],
                      outputs_equal=True, build_id=bid, **(extra or {})))

    # ---- frames: 512 frames of 24 calibrations, mixed seeds, in HBM
    n = 512
    frames = synth.make_frames(n, seed=77)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    rng = np.random.default_rng(4)
    Ks = matrices(24)[np.arange(n) % 24]
    mid = rng.uniform(-150.0, 150.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    kind = np.arange(n) % 4
    args = frame_args(n, Ks, mid, rng.uniform(-1.0, 1.0, (n, 3)), (kind & 1) == 1, (kind & 2) == 2)
    dmask = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    hmask = np.empty((n, h, w), np.uint8)
    res = np.zeros(n, capi.RESULT_DTYPE)
    src = C.c_void_p(dev.data_ptr())
    for where in ("device", "host"):
        mp, mloc = (C.c_void_p(dmask.data_ptr()), capi.DH_DEPTH_DEVICE) if where == "device" else (P(hmask), capi.DH_DEPTH_HOST)
        mview = dmask if where == "device" else hmask

        def fused():
            capi.check(L.dh_predict_frames_mask(ctx._h, hp._h, src, n, w, h, capi.DH_DEPTH_DEVICE, P(args), P(res), mp, mloc))
            return res.copy(), (mview.clone() if where == "device" else mview.copy())

        def two_calls():
            capi.check(L.dh_predict_frames(ctx._h, hp._h, src, n, w, h, capi.DH_DEPTH_DEVICE, P(args), P(res)))
            capi.check(L.dh_predict_mask_batch(ctx._h, hp._h, src, n, w, h, capi.DH_DEPTH_DEVICE, mp, mloc))
            return res.copy(), (mview.clone() if where == "device" else mview.copy())

        compare("frames_hbm_masks_to_" + where, {"fused": fused, "pose_then_mask": two_calls}, n)
    del dmask, hmask

    # ---- tracks: Biwi-shaped, in HBM and as Biwi files
    rng = np.random.default_rng(15)
    lengths = [int(x) // 4 for x in rng.integers(400, 901, 24)]
    seq_off, n_seq, total = _track_offsets(lengths)
    tframes = make_frames(total)
    tdev = torch.from_numpy(tframes.view(np.int16)).cuda()
    targs = frame_args(24, matrices(24))
    blob, off = biwi.pack_files([biwi.encode_depth(f) for f in tframes])
    tmask = torch.empty((total, h, w), dtype=torch.uint8, device="cuda")
    tres = np.zeros(total, capi.RESULT_DTYPE)
    mp = C.c_void_p(tmask.data_ptr())
    tsrc = C.c_void_p(tdev.data_ptr())
    D = capi.DH_DEPTH_DEVICE

    def t_fused():
        capi.check(L.dh_predict_tracks_mask(ctx._h, hp._h, tsrc, n_seq, P(seq_off), w, h, D, P(targs), 500.0, P(tres), mp, D))
        return tres.copy(), tmask.clone()

    def t_two():
        capi.check(L.dh_predict_tracks(ctx._h, hp._h, tsrc, n_seq, P(seq_off), w, h, D, P(targs), 500.0, P(tres)))
        capi.check(L.dh_predict_mask_batch(ctx._h, hp._h, tsrc, total, w, h, D, mp, D))
        return tres.copy(), tmask.clone()

    def b_fused():
        capi.check(L.dh_predict_tracks_mask_biwi(ctx._h, hp._h, P(blob), P(off), n_seq, P(seq_off), w, h, P(targs), 500.0, P(tres), mp, D))
        return tres.copy(), tmask.clone()

    def b_two():
        capi.check(L.dh_predict_tracks_biwi(ctx._h, hp._h, P(blob), P(off), n_seq, P(seq_off), w, h, P(targs), 500.0, P(tres)))
        capi.check(L.dh_predict_mask_batch_biwi(ctx._h, hp._h, P(blob), P(off), total, w, h, mp, D))
        return tres.copy(), tmask.clone()

    extra = {"lengths": lengths}
    compare("tracks_hbm", {"fused": t_fused, "tracks_then_mask": t_two}, total, extra)
    compare("tracks_biwi_files", {"fused": b_fused, "tracks_then_mask": b_two}, total, extra)
    del tmask, tdev

    # ---- latency: one VGA host frame
    one = np.ascontiguousarray(frames[5])
    K = IntrinsicMatrix.default_kinect_intrinsic()
    a1 = frame_args(1, K)
    m1 = np.empty((h, w), np.uint8)
    r1 = capi.dh_result()
    rr = np.zeros(1, capi.RESULT_DTYPE)
    reps = 200

    def single():
        capi.check(L.dh_predict(ctx._h, hp._h, P(one), w, h, K._ptr(), None, None, C.byref(r1)))
        capi.check(L.dh_predict_mask(ctx._h, hp._h, P(one), w, h, P(m1)))

    def fused1():
        capi.check(L.dh_predict_frames_mask(ctx._h, hp._h, P(one), 1, w, h, capi.DH_DEPTH_HOST, P(a1), P(rr), P(m1), capi.DH_DEPTH_HOST))

    single()
    want_m, want_r = m1.copy(), (np.array(r1.mid_point[:], np.float32), np.array(r1.rotation[:]))
    fused1()
    assert np.array_equal(m1, want_m) and np.array_equal(rr["mid_point"][0], want_r[0]) and np.array_equal(rr["rotation"][0], want_r[1])
    for _ in range(20):
        single()
        fused1()
    times = {"predict_then_mask": [], "fused_n1": []}
    for _ in range(a.repeats):
        times["predict_then_mask"].append(timed(single, reps))
        times["fused_n1"].append(timed(fused1, reps))
    for k, ts in times.items():
        emit(dict(name="latency_one_vga_host_frame", arm=k, calls_per_sample=reps, ms_per_frame=[1000.0 * t for t in ts],
                  outputs_equal=True, build_id=bid))


if __name__ == "__main__":
    main()
