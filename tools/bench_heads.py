"""Several heads per frame (dh_predict_frames_heads) against dh_predict_frames on the same frames: 512
synthetic 640x480 frames of two persons each, resident in HBM, on the configs[1] forest (10 trees of depth
15, stride 5).

    python tools/bench_heads.py [--repeats 3] [--calls 5] [--out FILE.jsonl] [--min-votes-scan]

Prints (and appends to --out) the GPU name and power limit, then one JSON line per arm.  The arms run
alternately, --repeats times each, after head 0 of every heads arm has been asserted equal, byte for byte,
to dh_predict_frames' result:
  predict_frames   dh_predict_frames
  heads_1          dh_predict_frames_heads, max_heads 1 (head 0 and its support / patch count only)
  heads_2, heads_4 max_heads 2 and 4 with min_cell_votes 1 and R = 150 mm: every frame tries all
                   2 (max_heads - 1) rounds unless its grid runs out, the most a round can cost
--min-votes-scan: the coarse-cell counts behind DEFAULT_MIN_CELL_VOTES.  It grows the forest the tests
train (dh_train_learn on 40 one-person frames) and reports, from the CPU oracle, the count of the cell
that seeds try 1 (after head 0 is suppressed) on one-person frames and on two-person frames.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_tracks import gpu_info, matrices  # noqa: E402
from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth, train  # noqa: E402


def timed(fn, reps=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def min_votes_scan(ctx, emit):
    from oracle import heads
    K = IntrinsicMatrix.default_kinect_intrinsic()
    tf, tc, tr_, tm = synth.make_frames(40, seed=101, with_truth=True)
    data = [dict(depth=tf[i], mask=tm[i], intrinsic=K, pos3d=tc[i], rot=tr_[i]) for i in range(len(tf))]
    js = train.HoughLearning(10, 80, 80, 8, 4, 1200, 0.3, 150, 20, 5.0).learn_native(8.0, data, seed=7, ctx=ctx).to_json()
    of = heads.HeadsForest.from_json(js)
    one = synth.make_frames(100, seed=999)
    two, centres, _ = synth.make_person_frames(100, seed=5, persons=2)
    spurious, second = [], []
    for i in range(100):
        _, _, tries = of.predict_heads(one[i], synth.KINECT_K, 2, 1, 150.0)
        spurious.append(int(tries[1]["cell_votes"]) if len(tries) > 1 else 0)
        _, _, tries = of.predict_heads(two[i], synth.KINECT_K, 2, 1, 150.0)
        second.append(int(tries[1]["cell_votes"]) if len(tries) > 1 else 0)
    q = [0, 5, 25, 50, 75, 95, 100]
    emit(dict(name="min_votes_scan", frames=100, radius_mm=150.0,
              one_person_try1_cell_votes_percentiles=dict(zip(map(str, q), np.percentile(spurious, q).tolist())),
              two_person_try1_cell_votes_percentiles=dict(zip(map(str, q), np.percentile(second, q).tolist()))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5, help="calls per timed sample")
    ap.add_argument("--out", default=None)
    ap.add_argument("--min-votes-scan", action="store_true")
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
    info["workload"] = "configs[1]: 10 trees depth 15, stride 5, synthetic 640x480 frames of two persons"
    emit(info)
    ctx = Context(0)
    if a.min_votes_scan:
        min_votes_scan(ctx, emit)
    hp = HoughPrediction.from_arrays(synth.make_forest(seed=1, n_trees=10, max_depth=15), stepwidth=5)
    n, w, h = 512, 640, 480
    frames, _, _ = synth.make_person_frames(n, seed=77, persons=2)
    dev = torch.from_numpy(frames.view(np.int16)).cuda()
    Ks = matrices(24)[np.arange(n) % 24]
    src = dict(device_ptr=dev.data_ptr(), n=n, w=w, h=h)
    ref = hp.predict_frames(None, Ks, ctx=ctx, **src)
    arms = {"predict_frames": lambda: hp.predict_frames(None, Ks, ctx=ctx, **src)}
    found = {}
    for m in (1, 2, 4):
        heads, n_heads = hp.predict_frames_heads(None, Ks, max_heads=m, min_cell_votes=1, radius_mm=150.0, ctx=ctx, **src)
        assert heads[:, 0]["pose"].tobytes() == ref.tobytes(), m
        found[m] = np.bincount(n_heads, minlength=m + 1).tolist()
        arms["heads_%d" % m] = (lambda m=m: hp.predict_frames_heads(None, Ks, max_heads=m, min_cell_votes=1, radius_mm=150.0, ctx=ctx,
                                                                    **src))
    for fn in arms.values():  # warm-up
        fn()
    times = {k: [] for k in arms}
    for _ in range(a.repeats):
        for k, fn in arms.items():
            times[k].append(timed(fn, a.calls))
    for k, ts in times.items():
        m = int(k.split("_")[1]) if k.startswith("heads") else None
        emit(dict(name="heads_hbm_two_persons", arm=k, frames=n, calls_per_sample=a.calls, ms_per_call=[1000.0 * t for t in ts],
                  frames_per_s=[n / t for t in ts], head0_equal=True, heads_histogram=found.get(m), build_id=bid))


if __name__ == "__main__":
    main()
