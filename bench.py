#!/usr/bin/env python
"""bench.py — frames/s of the Hough-forest prediction path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path (HoughPrediction::predict_parameter_parallel semantics, seeds
None) over one batch of synthetic frames.  Workload = BASELINE.json configs[1]: 1024 synthetic
640x480 Kinect-shaped depth frames per GPU, random-init forest of 10 trees x depth 15 (reference
JSON format), patch stride 5.

  value    device-timed frames/s with the batch already resident in HBM (CUDA events on the stream
           the kernels run on, max over ranks; `rank_ms` shows the spread over the ranks)
  e2e      the same metric through the C ABI with pinned HOST buffers: every step moves its frames
           host->device and its results device->host inside the timed region (worker threads of
           the library rewrite the frames as run-length files, the GPU expands them; chunks go
           over raw whenever the copy engine would otherwise idle)
  e2e_biwi the same frames handed over as Biwi run-length coded depth files (the database's own
           format, src/db_reader/biwi.rs:81-103) and expanded on the GPU
  roofline the traversal kernel against the MEASURED peak of the resource that carries it: the
           SM's L1 data stage (shared-memory tap wavefronts through the LSU pipe + node-record
           wavefronts through the TEX pipe; peaks from tools/peak_l1_gather.cu on this pool's
           B200s, profiles/measured_l1_peaks.json).  The wavefronts per node visit and the DRAM
           traffic come from an ncu capture of THIS build (profiles/traverse_profile.json carries
           the build id; on a mismatch `traffic` is dropped and the line says so).
           roofline_hbm keeps SURVEY 8(d)'s algorithmic bytes against the HBM copy peak.
  strong_scaling   BASELINE.json configs[2]: ONE Biwi-shaped synthetic sequence of 15 000 frames
           sharded by frame over the N ranks (shard.shard_range), device-resident, max over ranks
  trained_forest / general_rect_forest   the configs[1] frames through a forest TRAINED on the GPU
           (dh_train_learn on synthetic annotated frames) and through a forest with mixed rectangle
           sizes (summed-area table, 8 taps per node) - N = 1 only
  cpu_baseline   the C++ oracle (a restatement of the reference, NOT the Rust binary) timed on
           this box's host cores on a bounded sample of the same workload
--impl reference times that CPU restatement only (the reference is pure Rust + an un-vendored
crate and cannot be built in this image; see DESIGN.md).
--dump-outputs DIR writes the results of the last timed step of `value` (every frame of every rank,
in rank order) as DIR/mid_point.npy (float32), DIR/rotation.npy and DIR/bounding_box.npy (float64).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
Above 64 MB a fixed seeded sample of frames is written, with their indices in DIR/frame_index.npy.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FRAMES_PER_GPU = 1024
W, H = 640, 480
N_TREES, MAX_DEPTH, STRIDE = 10, 15, 5
BYTES_PER_NODE_VISIT = 56   # SURVEY.md §8d: 24 B node record + 8 SAT taps x 4 B
BYTES_PER_LEAF_HEADER = 16  # per patch x tree evaluation
SEQ_FRAMES = 15000          # configs[2]: Biwi-shaped sequence (24 sessions of 625 frames)
WAVEFRONT_BYTES = 128       # one L1 data-stage wavefront
METRIC = "frames/s, 640x480 depth, 10 trees depth 15, stride 5"
WORKLOAD = "configs[1]: batch of 1024 synthetic 640x480 frames per GPU, 10 trees depth 15, patch stride 5"


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_json(name):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.mark = 0
        self.bad = None

    def begin_region(self):
        """Only samples taken after this call count (the sampler itself starts earlier because
        nvidia-smi takes a few hundred ms to produce its first line)."""
        self.mark = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.mark:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                self.bad = ln
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
               "samples": len(sm), "reasons": sorted(reasons)}
        if not sm and self.bad:
            out["nvidia_smi_says"] = self.bad[:200]
        return out


def bind_to_gpu_numa_node(gpu_index: int):
    """Multi-GPU runs: keep this rank's host threads (and therefore its pinned frame buffers, first
    touched below) on the CPU cores next to its GPU, so that eight ranks do not pull their
    host->device copies across the socket interconnect.  Plumbing only; silently skipped when NVML
    or the affinity call is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:  # noqa: BLE001
        return None
    return None


def visible_cores() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def make_workload(rank: int, n_frames: int):
    from depthhead_b200 import synth
    arr = synth.make_forest(seed=1, n_trees=N_TREES, max_depth=MAX_DEPTH)
    frames = synth.make_frames(n_frames, seed=2024, start_index=rank * FRAMES_PER_GPU)
    return arr, frames


def _seq_block(job):
    from depthhead_b200 import synth
    lo, n = job
    return lo, synth.make_frames(n, seed=777, sequence=True, start_index=lo)


def make_sequence_shard(lo: int, hi: int, procs: int) -> np.ndarray:
    """frames [lo, hi) of the Biwi-shaped sequence (frame i depends only on the seed and i, so every
    sharding sees the same 15 000 frames); generated by forked workers BEFORE CUDA is initialised"""
    out = np.zeros((hi - lo, H, W), np.uint16)
    jobs = [(a, min(48, hi - a)) for a in range(lo, hi, 48)]
    if procs <= 1 or len(jobs) <= 1:
        for j in jobs:
            a, fr = _seq_block(j)
            out[a - lo:a - lo + len(fr)] = fr
        return out
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(procs, len(jobs))) as pool:
        for a, fr in pool.imap_unordered(_seq_block, jobs):
            out[a - lo:a - lo + len(fr)] = fr
    return out


def cpu_baseline(arr, frames, sample: int, threads: int, with_single: bool = True):
    """Faithful mode: naive rectangle sums (types.rs:317-339), patches and frames sequential.  Both
    of the reference's entry points are timed: predict_parameter_parallel (trees of one patch
    evaluated by a fork-join pool, the shape of stamm + rayon) and predict_parameter (single core);
    the faster one is reported so the GPU ratio is not flattered by fork-join overhead."""
    import oracle
    of = oracle.OracleForest(arr, STRIDE, 80, 80, 8.0, 20)
    tt = max(1, min(threads, N_TREES))
    sub = frames[:sample]
    t0 = time.perf_counter()
    _, _, evals = of.predict_batch(sub, _K(), mode=oracle.MODE_NAIVE, tree_threads=tt, frame_threads=1)
    dt = time.perf_counter() - t0
    par = {"value": sample / dt, "cores": tt, "seconds": dt, "evals_per_s": evals / dt}
    best = par
    single = None
    if with_single and tt > 1:
        ns = max(2, sample // 4)
        t0 = time.perf_counter()
        _, _, ev1 = of.predict_batch(frames[:ns], _K(), mode=oracle.MODE_NAIVE, tree_threads=1, frame_threads=1)
        d1 = time.perf_counter() - t0
        single = {"value": ns / d1, "cores": 1, "seconds": d1, "evals_per_s": ev1 / d1, "frames": ns}
        if single["value"] > par["value"]:
            best = single
    return {"value": best["value"], "unit": "frames/s", "cores": best["cores"], "kind": "port",
            "sample": "%d frames of the same workload, naive O(area) rectangle sums, %d thread(s): "
                      "oracle restatement of predict_parameter%s, not the Rust binary"
                      % (sample if best is par else single["frames"], best["cores"], "_parallel" if best is par else ""),
            "seconds": par["seconds"] + (single["seconds"] if single else 0.0), "evals_per_s": best["evals_per_s"],
            "tree_parallel": par, "single_core": single}


def cpu_best_effort(arr, frames, sample: int, threads: int):
    import oracle
    of = oracle.OracleForest(arr, STRIDE, 80, 80, 8.0, 20)
    sub = frames[:sample]
    t0 = time.perf_counter()
    of.predict_batch(sub, _K(), mode=oracle.MODE_SAT, tree_threads=1, frame_threads=threads)
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": "frames/s", "cores": threads,
            "sample": "%d frames, summed-area table + frame-level threads (not the reference's algorithm)" % sample}


def _K():
    from depthhead_b200 import synth
    return synth.KINECT_K


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(res: np.ndarray, out_dir: str) -> None:
    """--dump-outputs: the fields of capi.RESULT_DTYPE a caller receives, one .npy per field; the
    padding word is not an output.  Over DUMP_LIMIT_BYTES, a sample of frames fixed by a seed."""
    fields = {"mid_point": np.float32, "rotation": np.float64, "bounding_box": np.float64}
    out = {k: np.ascontiguousarray(res[k], dt) for k, dt in fields.items()}
    row_bytes = sum(a[:1].nbytes for a in out.values()) + 8
    keep = (DUMP_LIMIT_BYTES - 4096) // row_bytes          # 4 kB for the .npy headers
    if len(res) > keep:
        idx = np.sort(np.random.default_rng(0).choice(len(res), keep, replace=False))
        out = {k: a[idx] for k, a in out.items()}
        out["frame_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_reference(args):
    """--impl reference: the CPU restatement on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    arr, frames = make_workload(0, max(8, args.ref_sample))
    ncores = visible_cores()
    sample = args.ref_sample
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_baseline(arr, frames, min(2, sample), ncores)
    times, cb = [], None
    for i in range(args.steps):
        cb = cpu_baseline(arr, frames, sample, ncores, with_single=False)
        times.append(cb["seconds"])
    ms = 1000.0 * float(np.mean(times))
    val = sample / (ms / 1000.0)
    cb["value"] = val
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "step": "%d-frame sample of the workload on the host CPU" % sample,
                       "host_cores_visible": ncores},
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def traverse_roofline(counters, trav_ms, launches, clocks, n_sms, build_id):
    """roofline of traverse_kernel against the measured peaks of the SM's L1 data stage: the walk uses
    two pipes of it (LSU: shared-memory taps and the node records of the first levels; TEX: the node
    records of the deeper levels), so its roof is the pipe that runs closest to ITS measured peak"""
    peaks = load_json("measured_l1_peaks.json")
    prof = load_json("traverse_profile.json")
    visits = counters["node_visits"]
    sm_hz = 1e6 * float((clocks or {}).get("sm_mhz") or 1965.0)
    out = {"kernel": "traverse_kernel", "bound": "l1", "unit": "GB/s", "achieved": None, "peak": None, "frac": None, "traffic": None,
           "launches": launches, "avg_launch_ms": trav_ms / launches if launches else None,
           "node_visits_per_launch": visits / launches if launches else None, "build_id": build_id}
    if trav_ms > 0:
        out["node_visits_per_cycle_per_sm"] = visits / (trav_ms / 1000.0) / sm_hz / n_sms
    if peaks:
        out["measured_peaks"] = {k: peaks[k] for k in peaks if k.endswith("_per_sm")}
    if peaks and prof and trav_ms > 0:
        match = prof.get("build_id") == build_id
        to_gbs = visits * WAVEFRONT_BYTES / (trav_ms / 1000.0) / 1e9          # wavefronts per visit -> GB/s of wavefronts
        peak_gbs = lambda per_cycle: per_cycle * WAVEFRONT_BYTES * n_sms * sm_hz / 1e9  # noqa: E731
        pipes = {}
        for pipe in ("lsu", "tex"):
            wf = float(prof["%s_wavefronts_per_visit" % pipe])
            pk = float(peaks["%s_wavefronts_per_cycle_per_sm" % pipe])
            pipes[pipe] = {"achieved": wf * to_gbs, "peak": peak_gbs(pk), "frac": wf * to_gbs / peak_gbs(pk),
                           "wavefronts_per_node_visit": wf, "peak_wavefronts_per_cycle_per_sm": pk}
        top = max(pipes, key=lambda k: pipes[k]["frac"])
        out.update(achieved=pipes[top]["achieved"], peak=pipes[top]["peak"], frac=pipes[top]["frac"], pipe=top)
        both = float(peaks["concurrent_wavefronts_per_cycle_per_sm"])
        wf_both = pipes["lsu"]["wavefronts_per_node_visit"] + pipes["tex"]["wavefronts_per_node_visit"]
        out["pipes"] = pipes
        out["both_pipes"] = {"achieved": wf_both * to_gbs, "peak": peak_gbs(both), "frac": wf_both * to_gbs / peak_gbs(both),
                             "peak_wavefronts_per_cycle_per_sm": both}
        out["peak_source"] = ("measured with tools/peak_l1_gather.cu on this pool's B200s (profiles/measured_l1_peaks.json): divergent loads "
                              "through one pipe of the L1 data stage alone reach %.3f (LSU) and %.3f (TEX) wavefronts per cycle per SM, both "
                              "pipes loaded together %.3f; x 128 B x %d SMs x the SM clock of this run.  `frac` is the %s pipe, the one "
                              "closer to its own peak; `both_pipes` is the sum against the concurrent peak"
                              % (float(peaks["lsu_wavefronts_per_cycle_per_sm"]), float(peaks["tex_wavefronts_per_cycle_per_sm"]), both, n_sms,
                                 top.upper()))
        out["wavefront_source"] = {"source": prof.get("source"), "profile_build_id": prof.get("build_id"), "profile_matches_this_build": match}
        if match:
            out["traffic"] = float(prof["dram_bytes_per_launch"]) * (visits / launches) / float(prof["node_visits_per_launch"])
            out["traffic_note"] = "dram__bytes_read.sum + dram__bytes_write.sum of one launch from the ncu capture of this build, scaled by node visits"
        else:
            out["traffic_note"] = "dropped: profiles/traverse_profile.json was captured on build %s, this library is build %s" % (prof.get("build_id"), build_id)
        out["other_ceilings"] = {"l2_to_l1_sectors_per_cycle_per_sm": {"kernel": prof.get("l2_sectors_per_cycle_per_sm"),
                                                                       "measured_random_gather_ceiling": peaks.get("l2_random_sectors_per_cycle_per_sm")}}
    out["note"] = ("achieved = data-stage wavefronts per node visit of the named pipe (ncu capture of the named build) x node visits of this run "
                   "x 128 B / CUDA-event time of the kernel; the taps are served from the TMA-staged shared-memory tile and the node records "
                   "from L1/L2, so HBM carries almost none of it (roofline_hbm).  The walk is a dependent chain (fetch node -> two taps -> "
                   "compare -> next node): it is bound by the latency of that chain under L1 misses, with both pipes below their peaks")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step")
    ap.add_argument("--ref-sample", type=int, default=32, help="frames per reference step / CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 15 000-frame strong-scaling pass (configs[2])")
    ap.add_argument("--no-extra-forests", action="store_true", help="skip the trained / general-rectangle forest lines")
    ap.add_argument("--seq-frames", type=int, default=SEQ_FRAMES)
    ap.add_argument("--forest-from", default="json", choices=["json", "arrays"],
                    help="load the model through the reference JSON document (default) or the flat arrays")
    ap.add_argument("--chunk", type=int, default=0, help="frames per pipeline pass (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    cores = visible_cores()
    cores_per_rank = max(1, cores // max(1, local_world))

    # ---- host-side workloads first: plain numpy, generated by forked workers before CUDA exists in this process
    from depthhead_b200 import shard
    n = args.frames
    arr, frames = make_workload(rank, n)
    seq = None
    t_seq = 0.0
    if not args.no_strong:
        lo, hi = shard.shard_range(args.seq_frames, rank, world)
        t0 = time.perf_counter()
        seq = make_sequence_shard(lo, hi, cores_per_rank)
        t_seq = time.perf_counter() - t0

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libdepthhead_cuda has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))

    from depthhead_b200 import Context, HoughPrediction, IntrinsicMatrix, capi, synth
    build_id = capi.load().dh_build_id().decode()
    t_load = time.perf_counter()
    if args.forest_from == "json":
        js = synth.forest_to_json(arr, stepwidth=STRIDE)
        hp = HoughPrediction.from_json(js)
        model_src = "reference JSON document (%.0f MB)" % (len(js) / 1e6)
        del js
    else:
        hp = HoughPrediction.from_arrays(arr, stepwidth=STRIDE)
        model_src = "flat arrays"
    t_load = time.perf_counter() - t_load
    K = IntrinsicMatrix.default_kinect_intrinsic()
    ctx = Context(local)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    if args.chunk:
        ctx.set_chunk_frames(args.chunk)
    if world > 1:
        # the ranks of one host share its cores: each rank's run-length workers get their share
        ctx.set_encode_threads(max(1, cores_per_rank - (1 if cores_per_rank > 2 else 0)))
    n_sms = torch.cuda.get_device_properties(local).multi_processor_count

    pinned = torch.from_numpy(frames.view(np.int16)).pin_memory()
    host_np = pinned.numpy().view(np.uint16)
    dev = pinned.cuda(non_blocking=False)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        return hp.predict_batch(None, K, ctx=ctx, device_ptr=dev.data_ptr(), n=n, w=W, h=H)

    def step_host():
        return hp.predict_batch(host_np, K, ctx=ctx)

    # the same frames as Biwi depth files in one pinned blob (encoded once, outside every timed region)
    from depthhead_b200 import biwi
    blob_np, offsets = biwi.pack_files([biwi.encode_depth(f) for f in frames])
    blob_pinned = torch.from_numpy(blob_np).pin_memory()
    blob_host = blob_pinned.numpy()

    def step_biwi():
        return biwi.predict_files(hp, blob_host, offsets, W, H, K, ctx=ctx)

    def rank_spread(ms):
        """max over ranks (the number that counts) plus where the ranks stand"""
        if dist is None:
            return ms, {"min": ms, "median": ms, "max": ms, "slowest_rank": 0}
        t = torch.tensor([ms], device="cuda")
        allv = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        v = [float(x.item()) for x in allv]
        return max(v), {"min": min(v), "median": float(np.median(v)), "max": max(v), "slowest_rank": int(np.argmax(v))}

    def timed(fn, steps, with_stages=False):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage = {}
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            out = fn()
            if with_stages:
                for k, v in ctx.stage_ms().items():
                    stage[k] = stage.get(k, 0.0) + v
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        ms, spread = rank_spread(e0.elapsed_time(e1))
        # work counters: read once, after the timed region (every step does the same work)
        counters = {k: v * steps for k, v in ctx.counters().items()}
        return ms, wall * 1000.0, stage, counters, out, spread

    # ---- warm-up (also sizes scratch and the accumulator pool)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step_device()
    for _ in range(min(args.warmup, 2)):
        step_host()
        step_biwi()
    # keep the GPU under the same load until nvidia-smi is producing samples (untimed)
    t_wait = time.perf_counter()
    while len(sampler.lines) < 2 and time.perf_counter() - t_wait < 3.0:
        step_device()
    sampler.begin_region()
    ms_dev, wall_dev, _, counters, out_dev, spread_dev = timed(step_device, args.steps)
    ms_e2e, wall_e2e, _, _, out_host, spread_e2e = timed(step_host, args.steps)
    xfer = ctx.transfer_info()
    ms_biwi, wall_biwi, _, _, out_biwi, _ = timed(step_biwi, args.steps)
    # per-stage times (and the roofline of the traversal kernel): the same steps again with the
    # pipeline serialised on one stream, CUDA events between the stages
    ctx.enable_stage_timing(True)
    ms_ser, _, stage, counters_ser, _, _ = timed(step_device, args.steps, with_stages=True)
    ctx.enable_stage_timing(False)
    # the timed regions last ~0.2 s: extend the sampled window with identical untimed steps so the
    # clock record has enough samples under the same load
    t_wait = time.perf_counter()
    while len(sampler.lines) - sampler.mark < 8 and time.perf_counter() - t_wait < 2.0:
        step_device()
    clocks = sampler.stop()
    assert np.array_equal(out_dev["mid_point"], out_host["mid_point"]) and np.array_equal(out_dev["rotation"], out_host["rotation"])
    assert np.array_equal(out_dev["mid_point"], out_biwi["mid_point"]) and np.array_equal(out_dev["rotation"], out_biwi["rotation"])
    if args.dump_outputs:
        res_all = shard.gather_results(out_dev, n * world, dist)
        if rank == 0:
            dump_outputs(res_all, args.dump_outputs)

    # ---- strong scaling, configs[2]: one 15 000-frame sequence sharded by frame over the ranks
    strong = None
    if seq is not None:
        seq_dev = torch.empty(seq.shape, dtype=torch.int16, device="cuda")
        for a0 in range(0, len(seq), 512):  # pageable -> device in pieces
            seq_dev[a0:a0 + 512].copy_(torch.from_numpy(seq[a0:a0 + 512].view(np.int16)))
        torch.cuda.synchronize()
        ns = len(seq)

        def step_seq():
            if ns == 0:
                return np.zeros(0, capi.RESULT_DTYPE)
            return hp.predict_batch(None, K, ctx=ctx, device_ptr=seq_dev.data_ptr(), n=ns, w=W, h=H)
        step_seq()
        passes = 3
        ms_seq, _, _, _, out_seq, spread_seq = timed(step_seq, passes)
        res_all = shard.gather_results(out_seq, args.seq_frames, dist)
        sha = None
        if res_all is not None:
            sha = hashlib.sha1(np.ascontiguousarray(res_all["mid_point"]).tobytes() + np.ascontiguousarray(res_all["rotation"]).tobytes()).hexdigest()
        strong = {"workload": "configs[2]: one Biwi-shaped synthetic sequence of %d frames (24 sessions of 625 frames with smooth pose "
                              "trajectories), sharded by frame over the ranks (shard.shard_range), configs[1] forest, stride %d"
                              % (args.seq_frames, STRIDE),
                  "scaling": "strong", "value": args.seq_frames * passes / (ms_seq / 1000.0), "unit": "frames/s", "n_gpus": world,
                  "passes": passes, "ms_per_pass": ms_seq / passes, "frames_this_rank": ns, "rank_ms": spread_seq,
                  "host_generation_seconds": t_seq, "results_sha1": sha,
                  "note": "device-resident frames, CUDA events on the launching stream, barrier on both sides, max over ranks; "
                          "results_sha1 covers all %d poses in frame order and is the same for every N" % args.seq_frames}

    # the reference's live use (examples/live_prediction.rs:76,86): ONE frame per call, host buffer in,
    # result out, previous result as the next seed — wall-clock latency of dh_predict
    lat = []
    res = hp.predict_parameter_parallel(host_np[0], K, ctx=ctx)
    for i in range(60):
        f = host_np[i % n]
        t0 = time.perf_counter()
        res = hp.predict_parameter_parallel(f, K, res.mid_point, res.rotation, ctx=ctx)
        lat.append((time.perf_counter() - t0) * 1000.0)
    lat = sorted(lat[10:])
    single = {"median_ms": lat[len(lat) // 2], "p90_ms": lat[int(len(lat) * 0.9)], "calls": len(lat),
              "note": "dh_predict wall clock: one 640x480 host frame in, pose out, seeded with the previous pose"}

    # ---- the configs[1] frames through other models (N = 1 only)
    extra = {}
    if world == 1 and not args.no_extra_forests:
        def model_line(hp2, label, nf=512):
            nf = min(nf, n)
            d2 = dev[:nf]
            for _ in range(2):
                hp2.predict_batch(None, K, ctx=ctx, device_ptr=d2.data_ptr(), n=nf, w=W, h=H)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(3):
                o2 = hp2.predict_batch(None, K, ctx=ctx, device_ptr=d2.data_ptr(), n=nf, w=W, h=H)
            e1.record(stream)
            torch.cuda.synchronize()
            ms2 = e0.elapsed_time(e1) / 3
            ctx.enable_stage_timing(True)
            hp2.predict_batch(None, K, ctx=ctx, device_ptr=d2.data_ptr(), n=nf, w=W, h=H)
            st2, c2 = ctx.stage_ms(), ctx.counters()
            ctx.enable_stage_timing(False)
            return {"model": label, "frames": nf, "value": nf / (ms2 / 1000.0), "unit": "frames/s",
                    "nodes": hp2.n_nodes, "leaves": hp2.n_leaves, "votes": hp2.n_votes,
                    "stage_ms_per_frame": {k: v / nf for k, v in st2.items()},
                    "mean_visited_depth": c2["node_visits"] / max(1, c2["evals"]),
                    "votes_per_frame": (c2["centre_votes"] + c2["rot_votes"]) / nf, "cube_rebuilds": c2["cube_rebuilds"]}, o2
        try:
            from depthhead_b200 import train
            tf, tc, tr, tm = synth.make_frames(300, seed=101, with_truth=True)
            data = [dict(depth=tf[i], mask=tm[i], intrinsic=K, pos3d=tc[i], rot=tr[i]) for i in range(len(tf))]
            hl = train.HoughLearning(10, 80, 80, 15, 10, 5200, 0.3, 500, 20, 5.0)
            t0 = time.perf_counter()
            hpt = hl.learn_native(8.0, data, seed=1, ctx=ctx)
            t_train = time.perf_counter() - t0
            hpt.stepwidth = STRIDE
            line_t, o2 = model_line(hpt, "forest TRAINED on the GPU (dh_train_learn: 300 synthetic annotated frames, 10 trees, depth <= 15, "
                                         "5200 samples per tree, 500 candidates per node), stride 5")
            _, centres, _, _ = synth.make_frames(min(64, n), seed=2024, with_truth=True)   # the ground truth of the bench frames
            d = o2["mid_point"][:len(centres)].astype(np.float64) - centres
            line_t.update({"train_seconds": t_train, "median_lateral_error_mm": float(np.median(np.hypot(d[:, 0], d[:, 1]))),
                           "median_depth_error_mm": float(np.median(d[:, 2]))})
            extra["trained_forest"] = line_t
            hpt.close()
            del tf, tm, data
        except Exception as e:  # noqa: BLE001
            extra["trained_forest"] = {"error": repr(e)[:300]}
        try:
            arr_g = synth.make_forest(seed=1, n_trees=N_TREES, max_depth=MAX_DEPTH, ragged_rects=True)
            hpg = HoughPrediction.from_arrays(arr_g, stepwidth=STRIDE)
            line_g, _ = model_line(hpg, "random-init forest with MIXED rectangle sizes (10 trees, depth 15): summed-area table front end, "
                                        "8 taps per node, general node test; stride 5")
            extra["general_rect_forest"] = line_g
            hpg.close()
            del arr_g
        except Exception as e:  # noqa: BLE001
            extra["general_rect_forest"] = {"error": repr(e)[:300]}

    # ---- seeded sequences (the reference's live use, batched): 24 sequences x 625 frames, every frame
    #      seeded with the pose of the frame before it (examples/live_prediction.rs:75-88)
    if world == 1 and seq is not None and len(seq) >= 24 * 625:
        try:
            sq = seq_dev[:24 * 625]
            hp.predict_sequences(None, K, 500.0, ctx=ctx, device_ptr=sq.data_ptr(), n_seq=24, frames_per_seq=625, w=W, h=H)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            o_seq = hp.predict_sequences(None, K, 500.0, ctx=ctx, device_ptr=sq.data_ptr(), n_seq=24, frames_per_seq=625, w=W, h=H)
            e1.record(stream)
            torch.cuda.synchronize()
            ms_sq = e0.elapsed_time(e1)
            extra["seeded_sequences"] = {
                "workload": "the 15 000-frame Biwi-shaped sequence as 24 sessions x 625 frames: frame t of every session in one pass, "
                            "seeded on the device with the pose of frame t - 1 (centre seed if z > 500 mm), device-resident",
                "value": 24 * 625 / (ms_sq / 1000.0), "unit": "frames/s", "ms": ms_sq, "passes": 625, "frames_per_pass": 24,
                "launches": int(ctx.counters()["launches"]),
                "seeded_equals_unseeded_share": float(np.mean(np.all(o_seq.reshape(-1)["mid_point"] == out_seq[:24 * 625]["mid_point"], axis=1)))
                if strong is not None and world == 1 else None}
        except Exception as e:  # noqa: BLE001
            extra["seeded_sequences"] = {"error": repr(e)[:300]}

    total_frames = n * world * args.steps
    value = total_frames / (ms_dev / 1000.0)
    e2e_value = total_frames / (ms_e2e / 1000.0)

    # ---- rooflines from this rank's live stage timers
    peak, peak_src = measured_peak_gbs()
    dev_chunk = args.chunk or 512  # library default for device-resident input
    launches = max(1, (n + dev_chunk - 1) // dev_chunk) * args.steps
    trav_ms = stage.get("traverse", 0.0)
    roofline = traverse_roofline(counters_ser, trav_ms, launches, clocks, n_sms, build_id)
    alg_bytes = counters_ser["node_visits"] * BYTES_PER_NODE_VISIT + counters_ser["evals"] * BYTES_PER_LEAF_HEADER
    hbm_achieved = alg_bytes / (trav_ms / 1000.0) / 1e9 if trav_ms > 0 else None
    roofline_hbm = {"kernel": "traverse_kernel", "bound": "hbm", "achieved": hbm_achieved, "peak": peak, "unit": "GB/s",
                    "frac": (hbm_achieved / peak) if hbm_achieved else None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes / launches,
                    "note": "SURVEY 8(d)'s algorithmic bytes (56 B per node visit + 16 B per evaluation) against the HBM copy peak: above 1 "
                            "because these bytes never come from HBM (shared-memory tile + L1/L2); secondary figure, the bound is `roofline`"}
    # the HBM-bound kernel of the step: the front end (box-sum image, or summed-area table for
    # forests with mixed rectangle sizes) reads the depth once and writes its table once
    fe_ms = stage.get("sat", 0.0)
    fe_bytes_frame = W * H * 2 + (W - 24 + 1) * (H - 24 + 1) * 4
    fe_achieved = fe_bytes_frame * counters_ser["frames"] / (fe_ms / 1000.0) / 1e9 if fe_ms > 0 else None
    roofline_front = {"kernel": "box_image_kernel", "bound": "hbm", "achieved": fe_achieved, "peak": peak, "unit": "GB/s",
                      "frac": (fe_achieved / peak) if fe_achieved else None,
                      "algorithmic_bytes_per_frame": fe_bytes_frame, "avg_launch_ms": fe_ms / launches,
                      "note": "614400 B of depth read + 617x457 box sums x 4 B written per frame (24x24 rectangles)"}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_gpu_per_step": n, "global_frames_per_step": n * world,
                   "forest": "%d trees, depth %d, %d nodes, %d leaves, %d votes; loaded from %s in %.1f s"
                             % (N_TREES, MAX_DEPTH, hp.n_nodes, hp.n_leaves, hp.n_votes, model_src, t_load),
                   "sharding": "frames by rank, forest replicated, NO collective on the data path; torch.distributed (NCCL process group) is "
                               "used by this script only for the barrier around the timed regions and the max / all_gather of the per-rank times",
                   "host_affinity": ("rank bound to the %d cores next to its GPU (NVML)" % numa) if numa else "not bound",
                   "host_cores_visible": cores, "build_id": build_id,
                   "l2": "inputs (%.0f MB per step) and the box-sum scratch exceed the 126 MB L2; no flush" % (frames.nbytes / 1e6)},
        "rank_ms": {"value": spread_dev, "e2e": spread_e2e, "note": "CUDA-event milliseconds of the timed region per rank; the line uses the max"},
        "evals_per_s": counters["evals"] * world / (ms_dev / 1000.0),
        "patch_tree_evals_per_frame": counters["evals"] / max(1, counters["frames"]),
        "mean_visited_depth": counters["node_visits"] / max(1, counters["evals"]),
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(xfer["h2d_bytes"]),
                "d2h_bytes_per_step": int(out_host.nbytes), "ms_per_step": ms_e2e / args.steps,
                "wall_ms_per_step": wall_e2e / args.steps, "host_frame_bytes_per_step": int(frames.nbytes),
                "host_threads": int(xfer["encode_threads"]), "chunks_rewritten_per_step": int(xfer["encoded_chunks"]),
                "note": "dh_predict_batch on pinned host u16 frames: worker threads of the library rewrite chunks as run-length files "
                        "(Biwi format, biwi.rs:81-103) in pinned memory and the GPU expands them bit for bit; whenever the copy engine "
                        "would idle meanwhile, a chunk from the back of the batch goes over raw (DH_HOST_ENCODE=0: raw copies only)"},
        "e2e_biwi": {"value": total_frames / (ms_biwi / 1000.0), "unit": "frames/s", "h2d_bytes_per_step": int(offsets[-1]),
                     "d2h_bytes_per_step": int(out_biwi.nbytes), "ms_per_step": ms_biwi / args.steps,
                     "wall_ms_per_step": wall_biwi / args.steps, "compression": float(frames.nbytes) / float(offsets[-1]),
                     "note": "same frames as Biwi run-length coded depth files (biwi.rs:81-103), expanded on the GPU"},
        "single_frame_latency": single,
        "gpu_launches": int(counters["launches"]),
        "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
        "stage_timing": "separate pass of the same steps with the pipeline lanes serialised on one stream "
                        "(%.3f ms per step); the timed `value` pass overlaps chunks on %s lanes" % (ms_ser / args.steps, os.environ.get("DH_LANES", "2")),
        "wall_ms_per_step": wall_dev / args.steps,
        "work_per_step": {k: counters[k] // args.steps for k in ("frames", "valid_patches", "evals", "node_visits", "gate_patches", "hits", "centre_votes", "rot_votes", "meanshift_iters", "cube_rebuilds")},
        "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_front_end": roofline_front, "clocks": clocks,
    }
    if strong is not None:
        line["strong_scaling"] = strong
    line.update(extra)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(arr, frames, min(args.ref_sample, n), cores)
        try:
            cb["best_effort"] = cpu_best_effort(arr, frames, min(4 * args.ref_sample, n), cores)
        except Exception as e:  # noqa: BLE001
            cb["best_effort"] = {"error": str(e)}
        line["cpu_baseline"] = cb
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
