"""Rates of the batched 2-D entry points against the single-frame calls in a loop, on the
configs[1] forest (10 trees of depth 15) and synthetic 640x480 frames.

    python tools/bench_hough2d.py [--frames 512] [--strides 5 10] [--steps 3]

Prints the GPU name and power limit, then one JSON line per call: mask, raw vote image, blurred
vote image (all three written to device memory) and from2d-only batches on device-resident frames;
the same frames through dh_predict_mask / dh_hough_image_raw / dh_build_hough_image /
dh_predict_from2dhough frame by frame (host frames, host output); and from2d batches from host
frames end to end.  Batch and loop outputs are asserted equal before anything is timed.
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

from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = "nvidia-smi unavailable"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": out}


def timed(fn, steps):
    fn()  # warm-up: shapes, scratch, taps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--strides", type=int, nargs="+", default=[5, 10])
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    K = IntrinsicMatrix.default_kinect_intrinsic()
    info = gpu_info()
    info["build_id"] = capi.load().dh_build_id().decode()
    print(json.dumps(info), flush=True)
    ctx = Context(0)
    arr = synth.make_forest(seed=1, n_trees=10, max_depth=15)
    frames = synth.make_frames(a.frames, seed=2024)
    n, h, w = frames.shape
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    out8 = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    out16 = torch.empty((n, h, w), dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    src = dict(ctx=ctx, device_ptr=dev.data_ptr(), n=n, w=w, h=h)
    for stride in a.strides:
        hp = HoughPrediction.from_arrays(arr, stepwidth=stride)
        batch = {
            "mask_batch": (lambda: hp.predict_mask_batch(None, out_device_ptr=out8.data_ptr(), **src), out8, np.uint8),
            "raw_batch": (lambda: hp.hough_image_raw_batch(None, K, out_device_ptr=out16.data_ptr(), **src), out16, np.uint16),
            "blurred_batch": (lambda: hp.build_hough_image_batch(None, K, out_device_ptr=out16.data_ptr(), **src), out16, np.uint16),
            "from2d_batch": (lambda: hp.predict_parameter_from2dhough_batch(None, K, **src), None, None),
        }
        loop = {
            "mask_batch": ("mask_loop", lambda d: hp.predict_mask(d, ctx=ctx)),
            "raw_batch": ("raw_loop", lambda d: hp.hough_image_raw(d, K, ctx=ctx)),
            "blurred_batch": ("blurred_loop", lambda d: hp.build_hough_image(d, K, ctx=ctx)),
            "from2d_batch": ("from2d_loop", lambda d: hp.predict_parameter_from2dhough(d, K, ctx=ctx).mid_point),
        }
        for name, (fn, out, dtype) in batch.items():
            res = fn()
            got = res["mid_point"] if out is None else out.cpu().numpy().view(dtype)
            lname, single = loop[name]
            single(frames[0])  # warm-up
            t0 = time.perf_counter()
            ref = np.stack([single(d) for d in frames])
            t_loop = time.perf_counter() - t0
            assert np.array_equal(np.ascontiguousarray(got).view(np.uint8), np.ascontiguousarray(ref).view(np.uint8)), (name, stride)
            dt = timed(fn, a.steps)
            line = {"call": name, "stride": stride, "frames": n, "input": "device", "output": "device" if out is not None else "host results",
                    "frames_per_s": n / dt, "ms_per_call": 1000.0 * dt, "counters": ctx.counters(), "build_id": info["build_id"]}
            print(json.dumps(line), flush=True)
            print(json.dumps({"call": lname, "stride": stride, "frames": n, "input": "host", "output": "host",
                              "frames_per_s": n / t_loop, "ms_per_frame": 1000.0 * t_loop / n, "build_id": info["build_id"]}), flush=True)
        want = hp.predict_parameter_from2dhough_batch(None, K, **src)
        got = hp.predict_parameter_from2dhough_batch(frames, K, ctx=ctx)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8))
        dt = timed(lambda: hp.predict_parameter_from2dhough_batch(frames, K, ctx=ctx), a.steps)
        print(json.dumps({"call": "from2d_batch_host_frames", "stride": stride, "frames": n, "input": "host (end to end)",
                          "output": "host results", "frames_per_s": n / dt, "ms_per_call": 1000.0 * dt,
                          "transfer": ctx.transfer_info(), "build_id": info["build_id"]}), flush=True)
        ctx.enable_stage_timing(True)
        hp.build_hough_image_batch(None, K, out_device_ptr=out16.data_ptr(), **src)
        print(json.dumps({"call": "blurred_batch_stage_ms", "stride": stride, "frames": n, "stage_ms": ctx.stage_ms(),
                          "build_id": info["build_id"]}), flush=True)
        ctx.enable_stage_timing(False)
        hp.close()
    ctx.close()


if __name__ == "__main__":
    main()
