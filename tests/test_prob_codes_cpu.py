"""The patch gate from 8-bit probability codes (patch_gate_kernel, DESIGN.md section 5), restated in numpy
with the thresholds the context computes (dh_ctx.cu: Geometry::gate_pass_codes / gate_fail_codes): a
decision taken from the code sum alone must never contradict the reference's gate, the ordered f64 fold
`sum(prob) / T > 0.7` (prediction.rs:582-584).  CPU only: this pins the arithmetic.  The kernel is pinned
on the GPU by tests/test_gpu_parity.py::test_patch_gate_at_the_threshold, which runs patch_gate_kernel<false>
with codes (passes of at least DH_GATE_SPLIT_MIN frames) on leaf sums at these thresholds, and by
tests/test_gpu_gate_list.py (the kFrameK instantiations, gated-list slices, probabilities outside [0, 1])."""
import math

import numpy as np
import pytest


def gate_min_sum(T: int) -> float:
    """smallest f64 s with fl(s / T) > 0.7 (dh_ctx.cu, the nextafter walk)"""
    t = float(T)
    s = 0.7 * t
    while s / t > 0.7:
        s = math.nextafter(s, -math.inf)
    while not (s / t > 0.7):
        s = math.nextafter(s, math.inf)
    return s


def thresholds(T: int):
    smin = gate_min_sum(T)
    slack = float(T) * float(T) * math.ldexp(1.0, -50)
    pass_codes = int(min(4.0e9, math.ceil((smin + slack) * 256.0)))
    fail_codes = int(max(0.0, min(4.0e9, math.ceil((smin - slack) * 256.0) - 1.0)))
    return smin, pass_codes, fail_codes


def codes_of(prob: np.ndarray) -> np.ndarray:
    return np.minimum(np.floor(prob * 256.0), 255.0).astype(np.int64)  # plan_nodes_kernel


def reference_gate(prob_rows: np.ndarray, T: int) -> np.ndarray:
    s = np.zeros(len(prob_rows), np.float64)
    for t in range(T):  # fold from 0.0 in tree order
        s = s + prob_rows[:, t]
    return (s / float(T)) > 0.7


def check(prob_rows: np.ndarray):
    n, T = prob_rows.shape
    smin, pass_codes, fail_codes = thresholds(T)
    ref = reference_gate(prob_rows, T)
    # the kernel's exact path compares the fold with smin instead of dividing: the same gate
    s = np.zeros(n, np.float64)
    for t in range(T):
        s = s + prob_rows[:, t]
    assert np.array_equal(s >= smin, ref)
    S = codes_of(prob_rows).sum(axis=1)
    sure_pass = S >= pass_codes
    sure_fail = (~sure_pass) & (S + T <= fail_codes)
    assert not np.any(sure_pass & ~ref), "a code sum passed a patch the reference rejects"
    assert not np.any(sure_fail & ref), "a code sum rejected a patch the reference passes"
    return float(np.mean(~(sure_pass | sure_fail)))


@pytest.mark.parametrize("T", [1, 2, 3, 7, 10, 50, 333])
def test_code_decisions_never_contradict_the_fold(T):
    rng = np.random.default_rng(T)
    n = 200_000 // max(1, T // 10)
    undecided = check(rng.random((n, T)))
    assert undecided < 0.6
    # the bench forest's distribution: {0} U [0.5, 1], multiples of 1/1024
    u = rng.random((n, T))
    p = np.where(u < 0.15, 0.0, np.where(u < 0.40, rng.uniform(0.5, 0.8, (n, T)), rng.uniform(0.8, 1.0, (n, T))))
    check(np.round(p * 1024) / 1024)
    # probabilities on and one ulp around the code boundaries k / 256, sums on and around 0.7 * T
    k = rng.integers(0, 257, (n, T)).astype(np.float64) / 256.0
    for shift in (0.0, 1.0, -1.0):
        q = k.copy()
        if shift > 0:
            q = np.nextafter(q, 2.0)
        elif shift < 0:
            q = np.nextafter(q, -1.0)
        check(np.clip(q, 0.0, 1.0))
    base = np.full((n, T), 0.7)
    base += rng.choice([0.0, 2.0 ** -52, -(2.0 ** -52), 1.0 / 300, -1.0 / 300, 2.0 ** -9, -(2.0 ** -9)], (n, T))
    check(np.clip(base, 0.0, 1.0))
    # pure leaves: every probability 0 or 1
    check((rng.random((n, T)) < 0.7).astype(np.float64))


def test_thresholds_for_ten_trees():
    smin, pass_codes, fail_codes = thresholds(10)
    assert smin / 10.0 > 0.7 and not (math.nextafter(smin, -math.inf) / 10.0 > 0.7)
    # 0.7 * 10 * 256 = 1792: a code sum S >= 1793 passes for certain, S + 10 <= 1791 fails for certain
    assert pass_codes == 1793 and fail_codes == 1791
