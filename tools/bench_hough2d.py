"""Rates of the batched 2-D entry points against the single-frame calls in a loop, on the
configs[1] forest (10 trees of depth 15) and synthetic 640x480 frames.

    python tools/bench_hough2d.py [--frames 512] [--strides 5 10] [--steps 3] [--sections batch frames]

Prints the GPU name and power limit, then one JSON line per call.
Section "batch": mask, raw vote image, blurred vote image (all three written to device memory) and
from2d-only batches on device-resident frames; the same frames through dh_predict_mask /
dh_hough_image_raw / dh_build_hough_image / dh_predict_from2dhough frame by frame (host frames, host
output); and from2d batches from host frames end to end.  Batch and loop outputs are asserted equal
before anything is timed.
Section "frames": a database of 24 calibrations (the frames in 24 consecutive folders of equal size,
each with its own K, as the Biwi database's sequence folders): one dh_build_hough_image_frames call
against one dh_build_hough_image_batch call per folder, on device-resident frames; the same frames
as Biwi files in host memory: one dh_build_hough_image_frames_biwi call against dh_biwi_decode_depth
to device memory plus one _batch call per folder; and one K for every frame through _frames against
_batch (the price of reading the matrices per frame).  Calls of a comparison alternate, --repeats
times; their outputs are asserted equal before anything is timed.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, biwi, capi, synth  # noqa: E402

N_CAL = 24


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
    ap.add_argument("--repeats", type=int, default=3, help="alternations of each comparison of the frames section")
    ap.add_argument("--sections", nargs="+", default=["batch", "frames"], choices=["batch", "frames"])
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
        if "frames" in a.sections:
            bench_frames(a, ctx, hp, stride, frames, dev, out16, info)
        if "batch" not in a.sections:
            hp.close()
            continue
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


def calibrations(n):
    """N_CAL Kinect-like matrices (other focal lengths and centres) and the folder of every frame:
    n frames in N_CAL consecutive folders of (nearly) equal size"""
    Ks = np.zeros((N_CAL, 3, 3), np.float32)
    for i in range(N_CAL):
        f = 540.0 + 2.5 * i
        Ks[i] = [[f, 0.0, 310.0 + 1.0 * i], [0.0, f, 235.0 + 0.5 * i], [0.0, 0.0, 1.0]]
    folder = (np.arange(n) * N_CAL) // n
    return Ks, folder


def bench_frames(a, ctx, hp, stride, frames, dev, out16, info):
    L = capi.load()
    n, h, w = frames.shape
    Ks, folder = calibrations(n)
    Kf = np.ascontiguousarray(Ks[folder])
    bounds = np.searchsorted(folder, np.arange(N_CAL + 1))
    src = dict(ctx=ctx, device_ptr=dev.data_ptr(), n=n, w=w, h=h)
    blob, offsets = biwi.encode_frames(frames)
    decoded = torch.empty_like(dev)
    torch.cuda.synchronize()

    def grouped(base_ptr, call):  # one _batch call per folder, on the folder's frames in device memory
        for g in range(N_CAL):
            f0, f1 = int(bounds[g]), int(bounds[g + 1])
            call(IntrinsicMatrix(Ks[g]), dict(ctx=ctx, device_ptr=base_ptr + f0 * h * w * 2, n=f1 - f0, w=w, h=h), f0)

    res = np.zeros(n, capi.RESULT_DTYPE)

    def from2d_grouped(base_ptr):
        def one(k, s, f0):
            res[f0:f0 + s["n"]] = hp.predict_parameter_from2dhough_batch(None, k, **s)
        grouped(base_ptr, one)
        return res

    def blurred_grouped(base_ptr):
        grouped(base_ptr, lambda k, s, f0: hp.build_hough_image_batch(None, k, out_device_ptr=out16.data_ptr() + f0 * h * w * 2, **s))

    def decode():
        capi.check(L.dh_biwi_decode_depth(ctx._h, capi.ptr(blob), capi.ptr(offsets), n, w, h, C.c_void_p(decoded.data_ptr()),
                                          capi.DH_DEPTH_DEVICE))

    one_k = np.tile(K_DEFAULT.mat, (n, 1, 1))
    comparisons = {
        "from2d_24_matrices": (
            ("predict_parameter_from2dhough_frames", lambda: hp.predict_parameter_from2dhough_frames(None, Kf, **src)),
            ("predict_parameter_from2dhough_batch x 24", lambda: from2d_grouped(dev.data_ptr()).copy()), "device-resident", "host results"),
        "blurred_24_matrices": (
            ("build_hough_image_frames", lambda: hp.build_hough_image_frames(None, Kf, out_device_ptr=out16.data_ptr(), **src)),
            ("build_hough_image_batch x 24", lambda: blurred_grouped(dev.data_ptr())), "device-resident", "device"),
        "biwi_from2d_24_matrices": (
            ("build_hough_image_frames_biwi", lambda: biwi.build_hough_image_files(hp, blob, offsets, w, h, Kf, from2d=True, images=False,
                                                                                 ctx=ctx)[1]),
            ("biwi_decode_depth + predict_parameter_from2dhough_batch x 24", lambda: (decode(), from2d_grouped(decoded.data_ptr()).copy())[1]),
            "Biwi files in host memory", "host results"),
        "biwi_blurred_24_matrices": (
            ("build_hough_image_frames_biwi", lambda: biwi.build_hough_image_files(hp, blob, offsets, w, h, Kf, ctx=ctx,
                                                                                 out_device_ptr=out16.data_ptr())),
            ("biwi_decode_depth + build_hough_image_batch x 24", lambda: (decode(), blurred_grouped(decoded.data_ptr()))),
            "Biwi files in host memory", "device"),
        "from2d_one_k": (
            ("predict_parameter_from2dhough_frames", lambda: hp.predict_parameter_from2dhough_frames(None, one_k, **src)),
            ("predict_parameter_from2dhough_batch", lambda: hp.predict_parameter_from2dhough_batch(None, K_DEFAULT, **src)),
            "device-resident", "host results"),
        "blurred_one_k": (
            ("build_hough_image_frames", lambda: hp.build_hough_image_frames(None, one_k, out_device_ptr=out16.data_ptr(), **src)),
            ("build_hough_image_batch", lambda: hp.build_hough_image_batch(None, K_DEFAULT, out_device_ptr=out16.data_ptr(), **src)),
            "device-resident", "device"),
        "raw_one_k": (
            ("hough_image_raw_frames", lambda: hp.hough_image_raw_frames(None, one_k, out_device_ptr=out16.data_ptr(), **src)),
            ("hough_image_raw_batch", lambda: hp.hough_image_raw_batch(None, K_DEFAULT, out_device_ptr=out16.data_ptr(), **src)),
            "device-resident", "device"),
    }
    for comp, (first, second, inp, outp) in comparisons.items():
        outs = []
        for _, fn in (first, second):  # equal outputs before anything is timed
            r = fn()
            torch.cuda.synchronize()
            outs.append(np.ascontiguousarray(r).view(np.uint8) if isinstance(r, np.ndarray) else out16.cpu().numpy())
        assert np.array_equal(outs[0], outs[1]), (comp, stride)
        for rep in range(a.repeats):
            for call, fn in (first, second):
                dt = timed(fn, a.steps)
                print(json.dumps({"comparison": comp, "call": call, "repeat": rep, "stride": stride, "frames": n, "calibrations":
                                  N_CAL if "24" in comp else 1, "input": inp, "output": outp, "frames_per_s": n / dt,
                                  "ms_per_call": 1000.0 * dt, "build_id": info["build_id"]}), flush=True)


K_DEFAULT = IntrinsicMatrix.default_kinect_intrinsic()


if __name__ == "__main__":
    main()
