"""Rates of dh_predict_frames (every frame with its own intrinsics and seeds) against the calls a
caller has to use without it, on the configs[1] forest (10 trees of depth 15, stride 5) and
synthetic 640x480 frames.

    python tools/bench_frame_args.py [--frames 1024] [--repeats 3] [--out FILE.jsonl]

Prints (and appends to --out) the GPU name and power limit, then one JSON line per measurement.
The variants of a comparison run alternately, --repeats times each:
  same_k      dh_predict_batch against dh_predict_frames with one K for every frame and no seeds
              (device-resident frames: both run the same kernels, the second copies the arguments)
  mixed       dh_predict_frames with 24 distinct matrices and a mix of seeds (device-resident frames)
  loop        dh_predict frame by frame with those matrices and seeds (host frames): what such a
              caller runs today
  biwi        Biwi run-length files of 24 calibrations (contiguous groups, as the sequence folders of
              the database): one dh_predict_frames_biwi call against 24 dh_predict_batch_biwi calls
Outputs of the variants that compute the same thing are asserted equal before anything is timed.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = "nvidia-smi unavailable"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": out}


def matrices(n):
    Ks = np.zeros((n, 3, 3), np.float32)
    for i in range(n):
        f = 500.0 + 5.0 * i
        Ks[i] = [[f, 0.0, 310.0 + i], [0.0, f, 235.0 + 0.5 * i], [0.0, 0.0, 1.0]]
    return Ks


def timed(fn, steps=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps


def same(a, b):
    return np.array_equal(np.ascontiguousarray(a["mid_point"]).view(np.uint32), np.ascontiguousarray(b["mid_point"]).view(np.uint32)) and \
        np.array_equal(np.ascontiguousarray(a["rotation"]).view(np.uint64), np.ascontiguousarray(b["rotation"]).view(np.uint64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5, help="calls per timed run of the batched variants")
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
    info["workload"] = "configs[1]: 10 trees depth 15, stride 5, %d synthetic 640x480 frames" % a.frames
    emit(info)
    ctx = Context(0)
    hp = HoughPrediction.from_arrays(synth.make_forest(seed=1, n_trees=10, max_depth=15), stepwidth=5)
    K = IntrinsicMatrix.default_kinect_intrinsic()
    frames = synth.make_frames(a.frames, seed=2024)
    n, h, w = frames.shape
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    src = dict(ctx=ctx, device_ptr=dev.data_ptr(), n=n, w=w, h=h)
    n_cal = 24
    group = np.arange(n) * n_cal // n  # contiguous groups of frames with one calibration each
    Ks = matrices(n_cal)[group]
    rng = np.random.default_rng(7)
    kind = np.arange(n) % 4
    has_mid, has_rot = (kind & 1) == 1, (kind & 2) == 2
    mid = rng.uniform(-200.0, 200.0, (n, 3)).astype(np.float32)
    mid[:, 2] += 1000.0
    rot = rng.uniform(-1.0, 1.0, (n, 3))

    # ---- outputs first
    batch = hp.predict_batch(None, K, **src)
    assert same(batch, hp.predict_frames(None, K, **src)), "same K: dh_predict_frames differs from dh_predict_batch"
    mixed = hp.predict_frames(None, Ks, mid, rot, has_mid, has_rot, **src)

    def loop():
        r = np.zeros(n, capi.RESULT_DTYPE)
        for i in range(n):
            p = hp.predict_parameter_parallel(frames[i], IntrinsicMatrix(Ks[i]), mid[i] if has_mid[i] else None,
                                              rot[i] if has_rot[i] else None, ctx=ctx)
            r[i]["mid_point"], r[i]["rotation"] = p.mid_point, p.rotation
        return r

    assert same(mixed, loop()), "mixed: dh_predict_frames differs from the dh_predict loop"
    blob, offsets = biwi.encode_frames(frames)
    bounds = np.searchsorted(group, np.arange(n_cal + 1))
    Kcal = matrices(n_cal)

    def biwi_groups():
        r = np.zeros(n, capi.RESULT_DTYPE)
        for g in range(n_cal):
            a0, a1 = int(bounds[g]), int(bounds[g + 1])
            r[a0:a1] = biwi.predict_files(hp, blob, offsets[a0:a1 + 1], w, h, IntrinsicMatrix(Kcal[g]), ctx=ctx)
        return r

    biwi_one = lambda: biwi.predict_files(hp, blob, offsets, w, h, Ks, ctx=ctx)
    assert same(biwi_one(), biwi_groups()), "Biwi: dh_predict_frames_biwi differs from dh_predict_batch_biwi per group"

    # ---- timing, variants alternating
    comparisons = {
        "same_k": {"predict_batch": lambda: hp.predict_batch(None, K, **src), "predict_frames": lambda: hp.predict_frames(None, K, **src)},
        "mixed": {"predict_frames_24k_seeds": lambda: hp.predict_frames(None, Ks, mid, rot, has_mid, has_rot, **src),
                  "predict_loop_24k_seeds": loop},
        "biwi": {"predict_frames_biwi_24k": biwi_one, "predict_batch_biwi_x24": biwi_groups},
    }
    for comp, variants in comparisons.items():
        for fn in variants.values():
            fn()  # warm-up
        for rep in range(a.repeats):
            for name, fn in variants.items():
                steps = 1 if name == "predict_loop_24k_seeds" else a.steps
                dt = timed(fn, steps)
                emit({"comparison": comp, "call": name, "repeat": rep, "frames": n,
                      "input": "biwi files (host)" if comp == "biwi" else ("host frames" if "loop" in name else "device-resident"),
                      "frames_per_s": n / dt, "ms_per_call": 1000.0 * dt, "build_id": bid})
    ctx.close()


if __name__ == "__main__":
    main()
