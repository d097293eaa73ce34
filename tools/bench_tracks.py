"""Rates of dh_predict_tracks (tracks of any length, each with its own K and starting seeds, every later
frame seeded from the frame before it) against the calls a caller has to use without it, on the
configs[1] forest (10 trees of depth 15, stride 5) and synthetic Biwi-shaped 640x480 sequences.

    python tools/bench_tracks.py [--repeats 3] [--out FILE.jsonl]

Prints (and appends to --out) the GPU name and power limit, then one JSON line per measurement.
The variants of a comparison run alternately, --repeats times each; outputs of variants that compute
the same thing are asserted equal, bit for bit, before anything is timed.
  biwi_shaped   24 tracks of seeded ragged lengths (400-900 frames, about 15 000 in all), 24 matrices,
                frames in HBM: dh_predict_tracks against dh_predict_sequences once per track, and
                against the live rule applied on the host around dh_predict_frames, one call per step
  biwi_files    the same tracks as Biwi files in host memory: dh_predict_tracks_biwi against
                dh_biwi_decode_depth (to HBM) followed by dh_predict_sequences per track
  many_short    2 000 tracks of 1-60 frames, one K each of 24, frames in HBM, the default chunk:
                passes, frames per pass and rate of dh_predict_tracks
  equal         24 x 625 frames, one K: dh_predict_tracks against dh_predict_sequences
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

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


def _frames_part(args):
    n, start = args
    return synth.make_frames(n, seed=2024, sequence=True, start_index=start)


def make_frames(n):
    """synth.make_frames(n, sequence=True), generated in parallel (frame i depends on (seed, i) only)"""
    parts = [(min(500, n - s), s) for s in range(0, n, 500)]
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        return np.ascontiguousarray(np.concatenate(list(ex.map(_frames_part, parts))))


def plan_passes(lengths, F):
    """passes of dh_predict_tracks' plan (longest first, a freed slot takes the next waiting track)"""
    order = sorted((i for i in range(len(lengths)) if lengths[i]), key=lambda i: -lengths[i])
    left = [lengths[i] for i in order[:F]]
    nxt, passes = len(left), 0
    while left:
        passes += 1
        nl = []
        for v in left:
            if v > 1:
                nl.append(v - 1)
            elif nxt < len(order):
                nl.append(lengths[order[nxt]])
                nxt += 1
        left = nl
    return passes


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def same(a, b):
    return np.array_equal(np.ascontiguousarray(a["mid_point"]).view(np.uint32), np.ascontiguousarray(b["mid_point"]).view(np.uint32)) and \
        np.array_equal(np.ascontiguousarray(a["rotation"]).view(np.uint64), np.ascontiguousarray(b["rotation"]).view(np.uint64))


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
    info["workload"] = "configs[1]: 10 trees depth 15, stride 5, synthetic Biwi-shaped 640x480 sequences"
    emit(info)
    ctx = Context(0)
    hp = HoughPrediction.from_arrays(synth.make_forest(seed=1, n_trees=10, max_depth=15), stepwidth=5)
    K = IntrinsicMatrix.default_kinect_intrinsic()
    L = capi.load()
    w, h, px = 640, 480, 640 * 480

    rng = np.random.default_rng(15)
    lengths = rng.integers(400, 901, 24)
    lengths = [int(x) for x in lengths]
    total = sum(lengths)
    starts = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    frames = make_frames(max(total, 24 * 625))
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    torch.cuda.synchronize()
    Ks = matrices(24)
    src = dict(ctx=ctx, device_ptr=dev.data_ptr(), w=w, h=h)

    # ---- biwi_shaped: dh_predict_tracks without starting seeds (dh_predict_sequences has none)
    tracks = lambda: hp.predict_tracks(None, lengths, Ks, **src)

    def per_track():
        r = np.zeros(total, capi.RESULT_DTYPE)
        for s in range(24):
            r[starts[s]:starts[s + 1]] = hp.predict_sequences(None, IntrinsicMatrix(Ks[s]), 500.0, ctx=ctx,
                                                              device_ptr=dev.data_ptr() + 2 * px * int(starts[s]), n_seq=1,
                                                              frames_per_seq=lengths[s], w=w, h=h).reshape(-1)
        return r

    def live_loop():
        r = np.zeros(total, capi.RESULT_DTYPE)
        prev = None
        for t in range(max(lengths)):
            act = np.array([s for s in range(24) if t < lengths[s]])
            idx = starts[act] + t
            batch = dev.index_select(0, torch.from_numpy(idx).cuda())
            torch.cuda.synchronize()  # (the context runs on a stream of its own)
            if t == 0:
                got = hp.predict_frames(None, Ks[act], ctx=ctx, device_ptr=batch.data_ptr(), n=len(act), w=w, h=h)
            else:
                p = prev[act]
                got = hp.predict_frames(None, Ks[act], np.ascontiguousarray(p["mid_point"]), np.ascontiguousarray(p["rotation"]),
                                        p["mid_point"][:, 2] > np.float32(500.0), np.ones(len(act), bool), ctx=ctx,
                                        device_ptr=batch.data_ptr(), n=len(act), w=w, h=h)
            r[idx] = got
            prev = np.zeros(24, capi.RESULT_DTYPE) if prev is None else prev
            prev[act] = got
        return r

    want = tracks()
    assert same(want, per_track()), "biwi_shaped: dh_predict_tracks differs from dh_predict_sequences per track"
    assert same(want, live_loop()), "biwi_shaped: dh_predict_tracks differs from the host live-rule loop"

    # ---- biwi_files
    blob, offsets = biwi.encode_frames(frames[:total])
    tracks_biwi = lambda: biwi.predict_track_files(hp, blob, offsets, lengths, w, h, Ks, ctx=ctx)
    scratch = torch.empty((total, h, w), dtype=torch.int16, device="cuda")

    def decode_then_sequences():
        capi.check(L.dh_biwi_decode_depth(ctx._h, capi.ptr(blob), capi.ptr(offsets), total, w, h, capi.ptr(scratch.data_ptr()),
                                          capi.DH_DEPTH_DEVICE))
        r = np.zeros(total, capi.RESULT_DTYPE)
        for s in range(24):
            r[starts[s]:starts[s + 1]] = hp.predict_sequences(None, IntrinsicMatrix(Ks[s]), 500.0, ctx=ctx,
                                                              device_ptr=scratch.data_ptr() + 2 * px * int(starts[s]), n_seq=1,
                                                              frames_per_seq=lengths[s], w=w, h=h).reshape(-1)
        return r

    assert same(want, tracks_biwi()), "biwi_files: dh_predict_tracks_biwi differs from dh_predict_tracks"
    assert same(want, decode_then_sequences()), "biwi_files: decode + dh_predict_sequences differs"

    # ---- many_short: 2 000 tracks of 1-60 frames over the frames in HBM (repeated where they run out)
    short = [int(x) for x in rng.integers(1, 61, 2000)]
    n_short = sum(short)
    dev_short = torch.empty((n_short, h, w), dtype=torch.int16, device="cuda")
    for f0 in range(0, n_short, len(frames)):
        dev_short[f0:f0 + len(frames)] = dev[:n_short - f0]
    torch.cuda.synchronize()
    Ks_short = Ks[np.arange(2000) % 24]
    many = lambda: hp.predict_tracks(None, short, Ks_short, ctx=ctx, device_ptr=dev_short.data_ptr(), w=w, h=h)

    # ---- equal: 24 x 625, one K
    eq_tracks = lambda: hp.predict_tracks(None, [625] * 24, K, **src)
    eq_seq = lambda: hp.predict_sequences(None, K, 500.0, ctx=ctx, device_ptr=dev.data_ptr(), n_seq=24, frames_per_seq=625, w=w, h=h)
    assert same(eq_tracks(), eq_seq().reshape(-1)), "equal: dh_predict_tracks differs from dh_predict_sequences"

    comparisons = {
        "biwi_shaped": ({"predict_tracks": tracks, "predict_sequences_per_track": per_track, "host_live_rule_predict_frames": live_loop},
                        total, "device-resident"),
        "biwi_files": ({"predict_tracks_biwi": tracks_biwi, "biwi_decode_then_predict_sequences_per_track": decode_then_sequences},
                       total, "biwi files (host)"),
        "many_short": ({"predict_tracks": many}, n_short, "device-resident"),
        "equal": ({"predict_tracks": eq_tracks, "predict_sequences": eq_seq}, 24 * 625, "device-resident"),
    }
    shape = {"biwi_shaped": lengths, "biwi_files": lengths, "many_short": short, "equal": [625] * 24}
    for comp, (variants, n, where) in comparisons.items():
        for fn in variants.values():
            fn()  # warm-up
        for rep in range(a.repeats):
            for name, fn in variants.items():
                dt = timed(fn)
                d = {"comparison": comp, "call": name, "repeat": rep, "frames": n, "tracks": len(shape[comp]), "input": where,
                     "frames_per_s": n / dt, "ms_per_call": 1000.0 * dt, "build_id": bid}
                if name in ("predict_tracks", "predict_tracks_biwi", "predict_sequences"):  # one call: its kernel launches
                    d["launches"] = int(ctx.counters()["launches"])
                if name.startswith("predict_tracks"):
                    d["passes"] = plan_passes(shape[comp], 512)
                    d["frames_per_pass"] = n / d["passes"]
                emit(d)
    ctx.close()


if __name__ == "__main__":
    main()
