"""CPU tests of several heads per frame (dh_predict_frames_heads, DESIGN.md §7): the oracle's rules on
hand-built grids and accumulators, max_heads = 1 against the oracle's single-head result, the header /
ctypes / library agreement on the two structs and the signature, and the argument errors returned before
any device work."""
import math
import os
import re

import numpy as np
import pytest

import oracle
from oracle import heads
from depthhead_b200 import HoughPrediction, IntrinsicMatrix, capi, synth
from depthhead_b200.api import DEFAULT_MIN_CELL_VOTES, frame_args

K = IntrinsicMatrix.default_kinect_intrinsic()
H = capi.DH_DEPTH_HOST
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "depthhead_cuda.h")
EMPTY_KEYS, EMPTY_VALS = np.zeros((0, 3), np.int32), np.zeros(0, np.uint32)


def _search(grid, head0, K9, max_heads=4, min_cell_votes=1, radius=150.0, depth_mm=1000, cell0=0xFFFFFFFF):
    """the head search on an empty centre accumulator: every try's centre is its seed (mean-shift breaks on a
    zero sum), over a frame of constant depth"""
    depth = np.full((480, 640), depth_mm, np.uint16)
    g = np.zeros(400, np.uint32)
    for cell, v in grid.items():
        g[cell] = v
    return heads.heads_search(g, EMPTY_KEYS, EMPTY_VALS, depth, K9, head0, cell0, max_heads, min_cell_votes, radius)


def _cell(gx, gy):
    return gy * 20 + gx


def _seed(K9, gx, gy, z):
    """the reference's seed of a cell of a 640x480 frame at constant depth z (img_to_space, truncation)"""
    Ki = np.linalg.inv(np.asarray(K9, np.float64).reshape(3, 3))
    x, y = (gx + 0.5) * 32, (gy + 0.5) * 24
    r = Ki @ np.array([x, y, 1.0])
    return np.trunc(r * z / r[2]).astype(np.int64)


def test_suppression_is_a_closed_disc_around_the_projected_centre():
    # head 0 at z = 560 on the optical axis: (u, v) = (320, 240) and r_px = R * 560 / 560 = R exactly
    kk = synth.KINECT_K
    # cell (13, 10) starts at x = 416: 96 px from u, on the circle of R = 96 (closed: suppressed); (14, 10) at 128 px
    t = _search({_cell(13, 10): 9, _cell(14, 10): 5}, (0, 0, 560), kk, radius=96.0)
    assert [int(x) for x in t["seed_cell"][1:]] == [_cell(14, 10)]
    # a radius just below 96 keeps cell (13, 10), which wins; its own cell and then its disc go next
    t = _search({_cell(13, 10): 9, _cell(14, 10): 5}, (0, 0, 560), kk, radius=95.5)
    assert int(t["seed_cell"][1]) == _cell(13, 10) and int(t["cell_votes"][1]) == 9
    # vertically: cell (10, 14) starts at y = 336, 96 px below v
    t = _search({_cell(10, 14): 3, _cell(10, 15): 2}, (0, 0, 560), kk, radius=96.0)
    assert int(t["seed_cell"][1]) == _cell(10, 15)
    # a centre at z <= 0 suppresses only the cells whose rectangle holds its (clamped) projection
    t = _search({_cell(0, 0): 7, _cell(1, 0): 6}, (-1000, -1000, 0), kk, max_heads=2, radius=1000.0)
    assert int(t["seed_cell"][1]) == _cell(1, 0)


def test_first_maximum_wins_ties_and_seeds_follow_the_reference():
    kk = synth.KINECT_K
    far = {_cell(2, 3): 40, _cell(17, 3): 40, _cell(17, 16): 40}
    t = _search(far, (0, 0, 1000), kk, max_heads=4)
    # ties: the lower index first; each try zeroes its own cell
    assert [int(x) for x in t["seed_cell"][1:]] == [_cell(2, 3), _cell(17, 3), _cell(17, 16)]
    assert all(t["accepted"])
    for tr, (gx, gy) in zip(t[1:], [(2, 3), (17, 3), (17, 16)]):
        assert np.array_equal(tr["centre"], _seed(kk, gx, gy, 1000)), (tr, gx, gy)


def test_duplicates_are_dropped_but_suppress_and_the_try_cap_holds():
    # fx = 280, fy = 1120: R = 150 mm is 42 px at z = 1000 while a cell two rows down is 48 px away, so it
    # survives suppression, yet its seed lies within R of head 0 in space
    kk = np.array([[280, 0, 320], [0, 1120, 240], [0, 0, 1]], np.float32)
    grid = {_cell(10, 12): 30, _cell(10, 13): 20, _cell(2, 2): 10}
    t = _search(grid, (0, 0, 1000), kk, max_heads=3)
    s = _seed(kk, 10, 12, 1000)
    assert s[0] ** 2 + s[1] ** 2 + (s[2] - 1000) ** 2 <= 150 ** 2
    assert int(t["seed_cell"][1]) == _cell(10, 12) and not t["accepted"][1]
    # the dropped try's disc still applies: (10, 13) is within 42 px of its centre, so the next seed is (2, 2)
    assert int(t["seed_cell"][2]) == _cell(2, 2) and t["accepted"][2]
    # max_heads = 2: at most 2 tries after head 0, whatever they find
    grid2 = {_cell(10, 12): 30, _cell(4, 18): 25, _cell(2, 2): 10}
    t2 = _search(grid2, (0, 0, 1000), kk, max_heads=2)
    assert len(t2) == 3 and [bool(a) for a in t2["accepted"]] == [True, False, True]
    # the integer distance test: floor(R)^2, so a centre 150 mm away is a duplicate for R = 150.9 and not for 149.9
    t3 = _search({_cell(10, 12): 30}, (0, 0, 1000), kk, max_heads=2, radius=149.9)
    d2 = int(s[0] ** 2 + s[1] ** 2 + (s[2] - 1000) ** 2)
    assert bool(t3["accepted"][1]) == (d2 > 149 ** 2)


def test_min_cell_votes_stops_the_search():
    kk = synth.KINECT_K
    grid = {_cell(2, 3): 5, _cell(17, 16): 4}
    assert len(_search(grid, (0, 0, 1000), kk, min_cell_votes=6)) == 1
    t = _search(grid, (0, 0, 1000), kk, min_cell_votes=5)
    assert len(t) == 2 and int(t["seed_cell"][1]) == _cell(2, 3)
    assert len(_search(grid, (0, 0, 1000), kk, min_cell_votes=4)) == 3
    # head 0's seed cell is zeroed before the next arg-max
    assert len(_search({_cell(9, 9): 50}, (5000, 0, 1000), kk, cell0=_cell(9, 9))) == 1


def test_support_sums_the_final_window():
    kk = synth.KINECT_K
    keys = np.array([[0, 0, 1000], [9, -10, 1009], [10, 0, 1000], [0, 0, 990]], np.int32)
    vals = np.array([5, 7, 100, 11], np.uint32)
    t = heads.heads_search(np.zeros(400, np.uint32), keys, vals, np.full((480, 640), 1000, np.uint16), kk, (0, 0, 1000),
                            0xFFFFFFFF, 2, 1, 150.0)
    assert int(t["support"][0]) == 5 + 7 + 11  # x = 10 and z = 990 + ... : the window is -10..+9


@pytest.fixture(scope="module")
def synthetic_forest():
    js = synth.forest_to_json(synth.make_forest(seed=0), stepwidth=10)
    return heads.HeadsForest.from_json(js)


def test_one_head_is_the_single_head_result(synthetic_forest):
    frames, _, _ = synth.make_person_frames(3, seed=5)
    for i, (mg, rg) in enumerate([(None, None), ((10.0, -20.0, 900.0), None), (None, (0.1, -0.2, 0.3))]):
        tr = synthetic_forest.f.predict(frames[i], synth.KINECT_K, midp_guess=mg, rot_guess=rg)
        heads, n, tries = synthetic_forest.predict_heads(frames[i], synth.KINECT_K, 1, 1, 150.0, midp_guess=mg, rot_guess=rg)
        assert n == 1 and len(tries) == 1
        assert np.array_equal(heads[0]["mid_point"], tr.mid_point) and np.array_equal(heads[0]["rotation"], tr.rotation)
        assert int(heads[0]["seed_cell"]) == (0xFFFFFFFF if mg is not None else int(np.argmax(tr.guess_pos)))
        more, n4, _ = synthetic_forest.predict_heads(frames[i], synth.KINECT_K, 4, 1, 150.0, midp_guess=mg, rot_guess=rg)
        assert more[0].tobytes() == heads[0].tobytes() and n4 >= 1
        assert not more[n4:].tobytes().strip(b"\0")


def test_make_person_frames():
    frames, centres, counts = synth.make_person_frames(6, seed=2)
    assert frames.shape == (6, 480, 640) and frames.dtype == np.uint16
    assert set(counts.tolist()) <= {1, 2, 3}
    for i in range(6):
        c = centres[i, :counts[i]]
        assert not np.isnan(c).any() and np.isnan(centres[i, counts[i]:]).all()
        for a in range(len(c)):
            for b in range(a):
                assert np.hypot(*(c[a, :2] - c[b, :2])) > 400.0
    f2, _, k2 = synth.make_person_frames(4, seed=2, persons=2)
    assert (k2 == 2).all() and np.array_equal(synth.make_person_frames(6, seed=2)[0], frames)


def _header_struct(name):
    text = open(HEADER).read()
    m = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S)
    assert m, name
    return [" ".join(line.split("/*")[0].split()) for line in m.group(1).splitlines() if line.split("/*")[0].strip()]


def test_structs_and_signature_agree():
    assert _header_struct("dh_heads_params") == ["uint32_t max_heads;", "uint32_t min_cell_votes;", "float radius_mm;",
                                                 "uint32_t _pad;"]
    assert _header_struct("dh_head") == ["dh_result pose;", "uint64_t support;", "uint32_t n_patches;", "uint32_t seed_cell;"]
    P, Hd = capi.HEADS_PARAMS_DTYPE, capi.HEAD_DTYPE
    assert P.itemsize == 16 and [P.fields[k][1] for k in ("max_heads", "min_cell_votes", "radius_mm", "_pad")] == [0, 4, 8, 12]
    assert Hd.itemsize == 72 and [Hd.fields[k][1] for k in ("pose", "support", "n_patches", "seed_cell")] == [0, 56, 64, 68]
    assert Hd.fields["pose"][0] == capi.RESULT_DTYPE and Hd.itemsize == heads.HEAD_DTYPE.itemsize
    assert all(Hd.fields[k] == heads.HEAD_DTYPE.fields[k] for k in ("support", "n_patches", "seed_cell"))
    L = capi.load()
    assert hasattr(L, "dh_predict_frames_heads")
    sig = capi.SIGNATURES["dh_predict_frames_heads"][1]
    assert len(sig) == 11 and sig[:8] == capi.SIGNATURES["dh_predict_frames"][1][:8]
    assert re.search(r"int dh_predict_frames_heads\(dh_ctx\* c, const dh_forest\* f, const uint16_t\* depth, uint32_t n, uint32_t w, "
                     r"uint32_t h,\s+int depth_loc, const dh_frame_args\* args, const dh_heads_params\* params, dh_head\* out,\s+"
                     r"uint32_t\* n_heads\);", open(HEADER).read())
    assert DEFAULT_MIN_CELL_VOTES >= 1


def _err(rc):
    assert rc == capi.DH_E_ARG, rc
    return capi.load().dh_last_error().decode()


def test_argument_errors(small_case):
    """every error below is returned with a NULL context: nothing reached a device"""
    L = capi.load()
    _, js, _ = small_case
    hp = HoughPrediction.from_json(js)
    P = capi.ptr
    depth = np.zeros((3, 80, 80), np.uint16)
    out = np.zeros((3, 8), capi.HEAD_DTYPE)
    nh = np.zeros(3, np.uint32)
    args = frame_args(3, K)

    def call(max_heads=4, votes=1, radius=150.0, a=args, o=out, n_h=nh, loc=H, ctx=None, f=hp._h, d=depth, n=3, params=True):
        p = np.zeros(1, capi.HEADS_PARAMS_DTYPE)
        p["max_heads"], p["min_cell_votes"], p["radius_mm"] = max_heads, votes, radius
        return _err(L.dh_predict_frames_heads(ctx, f, P(d), n, 80, 80, loc, P(a), P(p) if params else None, P(o), P(n_h)))

    assert "NULL params" in call(params=False)
    for bad in (0, 9, 1 << 31):
        assert "max_heads must be 1..8" in call(max_heads=bad)
    for bad in (0.0, -1.0, math.nan, -math.inf):
        assert "radius_mm must be > 0" in call(radius=bad)
    assert "min_cell_votes must be >= 1" in call(votes=0)
    assert "bad depth_loc" in call(loc=7)
    bad_args = args.copy()
    bad_args["has_guess"][1] = 4
    assert "frame 1" in call(a=bad_args)
    assert "NULL out or n_heads" in call(o=None) and "NULL out or n_heads" in call(n_h=None)
    for kw in (dict(), dict(f=None), dict(a=None), dict(d=None)):
        assert "NULL argument" in call(**kw), kw
    # no frames: nothing to write, still a NULL context
    assert "NULL argument" in call(n=0, o=None, n_h=None, d=None)
    api_hp = HoughPrediction.from_json(js)
    with pytest.raises(Exception, match="max_heads"):
        api_hp.predict_frames_heads(depth, K, max_heads=0, ctx=type("C", (), {"_h": None})())
