"""Seeded synthetic inputs: Kinect-shaped depth frames and random-init Hough forests.

The pretrained forest and the BIWI database are not available offline, so tests and bench.py
run on these.  Shapes follow the reference:
  * frames: 640x480 u16 millimetres, 0 = invalid/background (examples/live_prediction.rs:217-264);
  * forest: the hyper-parameters of examples/hough_tree_trainer.rs:70-75,149-168 — 80x80
    sub-image, feature rectangles of scale 0.3 placed like Rect::scale_and_replace
    (src/types.rs:82-91: 24x24, origin floor(u*56)), thresholds uniform in [-256,256)
    (src/hough/houghforest.rs:227-246), leaves {prob, offsets[mm], rotations[deg]}
    (houghforest.rs:204-225), gaussian_sigma 8.0, meanshift_iterations 20 (prediction.rs:232).

All decimals are short exact binary fractions (multiples of 2^-4 / 2^-6) so that every JSON
float parser agrees bit-for-bit.
"""
from __future__ import annotations

import json

import numpy as np

KINECT_K = np.array([[560.0, 0.0, 320.0], [0.0, 560.0, 240.0], [0.0, 0.0, 1.0]], np.float32)  # types.rs:418-420


# ----------------------------------------------------------------------------- frames
def _draw_person(img, hx, hy, hz, rng, mask=None):
    """A torso slab and a head ellipsoid centred at (hx, hy, hz) mm into img [h, w] (nearer surfaces are the
    caller's order: a later person overwrites), the head's pixels set to 255 in mask if given."""
    h, w = img.shape
    fx, fy, cx, cy = 560.0 * w / 640.0, 560.0 * h / 480.0, w / 2.0, h / 2.0
    # torso slab: below the head, slightly behind the head centre
    tz = hz + 40.0
    u0, u1 = int(cx + (hx - 230) * fx / tz), int(cx + (hx + 230) * fx / tz)
    v0, v1 = int(cy + (hy + 115) * fy / tz), h
    u0, u1, v0, v1 = max(u0, 0), min(u1, w), max(v0, 0), min(v1, h)
    if u1 > u0 and v1 > v0:
        uu = np.arange(u0, u1)[None, :]
        vv = np.arange(v0, v1)[:, None]
        shape = tz + 0.00008 * ((uu - (u0 + u1) / 2.0) ** 2) * tz / fx + 0.02 * (vv - v0)
        img[v0:v1, u0:u1] = np.clip(shape + rng.uniform(-3, 3, shape.shape), 1, 65535).astype(np.uint16)
    # head ellipsoid (orthographic approximation around the head centre)
    a, b, c = 75.0, 100.0, 90.0
    ru, rv = int(a * fx / hz) + 2, int(b * fy / hz) + 2
    uc, vc = cx + hx * fx / hz, cy + hy * fy / hz
    u0, u1 = max(int(uc - ru), 0), min(int(uc + ru) + 1, w)
    v0, v1 = max(int(vc - rv), 0), min(int(vc + rv) + 1, h)
    if u1 > u0 and v1 > v0:
        uu = np.arange(u0, u1)[None, :]
        vv = np.arange(v0, v1)[:, None]
        X = (uu - cx) * hz / fx - hx
        Y = (vv - cy) * hz / fy - hy
        q = 1.0 - (X / a) ** 2 - (Y / b) ** 2
        inside = q > 0
        d = hz - c * np.sqrt(np.where(inside, q, 0.0)) + rng.uniform(-3, 3, q.shape)
        reg = img[v0:v1, u0:u1]
        reg[inside] = np.clip(d, 1, 65535).astype(np.uint16)[inside]
        if mask is not None:
            mask[v0:v1, u0:u1][inside] = 255


def make_frames(n: int, seed: int = 0, w: int = 640, h: int = 480, sequence: bool = False,
                start_index: int = 0, with_truth: bool = False):
    """n synthetic depth frames [n,h,w] u16.  One "person": a head ellipsoid (semi-axes
    ~75x100x90 mm) at depth z0~U[700,1200] mm, a torso slab below it, +-3 mm noise, 1-2 %
    dropout to 0.  Frame i depends only on (seed, start_index+i), so shards generated on
    different ranks are identical to the corresponding slice of a single-process run.
    sequence=True: smooth pose trajectories in "sessions" of 625 frames (BIWI-shaped).
    with_truth=True: also the ground truth a Biwi annotation carries (db_reader/reader.rs
    DepthTrue): head centre [n,3] f32 mm, rotation [n,3] f32 (the ellipsoid has no orientation:
    a smooth function of the position stands in), head mask [n,h,w] u8."""
    out = np.zeros((n, h, w), np.uint16)
    centres = np.zeros((n, 3), np.float32)
    masks = np.zeros((n, h, w), np.uint8) if with_truth else None
    for i in range(n):
        gi = start_index + i
        if sequence:
            sess, k = divmod(gi, 625)
            rs = np.random.default_rng([seed, 7919, sess])
            base = rs.uniform([-150, -80, 750], [150, 40, 1150])
            amp = rs.uniform([20, 10, 20], [80, 40, 80])
            ph = rs.uniform(0, 2 * np.pi, 3)
            frq = rs.uniform(0.004, 0.02, 3)
            hc = base + amp * np.sin(ph + frq * k * 2 * np.pi)
        else:
            hc = None
        rng = np.random.default_rng([seed, gi])
        if hc is None:
            hc = rng.uniform([-150, -80, 700], [150, 40, 1200])
        hx, hy, hz = float(hc[0]), float(hc[1]), float(hc[2])
        _draw_person(out[i], hx, hy, hz, rng, masks[i] if with_truth else None)
        centres[i] = (hx, hy, hz)
        # dropout: 1-2 % of pixels to 0
        frac = rng.uniform(0.01, 0.02)
        drop = rng.random((h, w)) < frac
        out[i][drop] = 0
    if with_truth:
        rots = np.stack([centres[:, 0] / 8.0, centres[:, 1] / 4.0, (centres[:, 2] - 950.0) / 16.0], 1).astype(np.float32)
        return out, centres, rots, masks
    return out


def make_person_frames(n: int, seed: int = 0, w: int = 640, h: int = 480, persons=None):
    """n frames [n,h,w] u16 with 1-3 "persons" each (make_frames' person), side by side at different depths,
    and their true head centres: (frames, centres [n,3,3] f32 mm with NaN rows for absent persons, counts [n]).
    persons: None = 1-3 drawn per frame, an int = that many in every frame.  Person k stands in its own
    lateral slot (heads at least 400 mm apart); the nearer persons are drawn last, 1-2 % dropout as make_frames."""
    out = np.zeros((n, h, w), np.uint16)
    centres = np.full((n, 3, 3), np.nan, np.float32)
    counts = np.zeros(n, np.int32)
    slots = {1: [0.0], 2: [-260.0, 260.0], 3: [-440.0, 0.0, 440.0]}
    for i in range(n):
        rng = np.random.default_rng([seed, 104729, i])
        k = int(rng.integers(1, 4)) if persons is None else int(persons)
        hc = np.stack([np.asarray(slots[k]) + rng.uniform(-40, 40, k), rng.uniform(-80, 40, k), rng.uniform(800, 1300, k)], 1)
        for j in np.argsort(-hc[:, 2]):
            _draw_person(out[i], float(hc[j, 0]), float(hc[j, 1]), float(hc[j, 2]), rng)
        centres[i, :k] = hc
        counts[i] = k
        drop = rng.random((h, w)) < rng.uniform(0.01, 0.02)
        out[i][drop] = 0
    return out, centres, counts


# ----------------------------------------------------------------------------- forest
def _q(x, step):
    return np.round(np.asarray(x) / step) * step


def make_forest(seed: int = 0, n_trees: int = 10, max_depth: int = 15, sub_w: int = 80, sub_h: int = 80,
                rect_scale: float = 0.3, stop_prob: float = 0.0, votes_lo: int = 2, votes_hi: int = 8,
                shuffle_nodes: bool = False, ragged_rects: bool = False, tie_thresholds: bool = False) -> dict:
    """Random-init forest as flat arrays (the same layout oracle.forest_arrays_from_doc returns).

    stop_prob == 0: full binary trees (2^D - 1 nodes, 2^D leaves per tree).
    stop_prob  > 0: sparse trees — each would-be internal node below the root becomes a leaf with
    that probability (the 50-tree depth-20 config).
    shuffle_nodes: permute the file order of the nodes of every tree (root stays index 0) to
    exercise the loader's re-layout.  ragged_rects: vary rectangle sizes (incl. a few empty ones,
    count == 0 -> average 0.0, types.rs:335-337) instead of the fixed 24x24."""
    rng = np.random.default_rng([seed, 104729])
    rw, rh = int(sub_w * rect_scale), int(sub_h * rect_scale)
    node_off, leaf_off = [0], [0]
    rects_l, thr_l, child_l = [], [], []
    n_leaves_total = 0
    for _t in range(n_trees):
        # build level by level; frontier = indices of internal nodes at this depth
        children = []  # list of [c0, c1]
        n_nodes, n_leaves = 1, 0
        frontier = [0]
        children.append([0, 0])
        for depth in range(max_depth):
            nxt = []
            nf = len(frontier)
            last = depth == max_depth - 1
            if last:
                leafmask = np.ones((nf, 2), bool)
            elif stop_prob > 0:
                leafmask = rng.random((nf, 2)) < stop_prob
            else:
                leafmask = np.zeros((nf, 2), bool)
            for j, nd in enumerate(frontier):
                for b in range(2):
                    if leafmask[j, b]:
                        children[nd][b] = ~n_leaves
                        n_leaves += 1
                    else:
                        children[nd][b] = n_nodes
                        children.append([0, 0])
                        nxt.append(n_nodes)
                        n_nodes += 1
            frontier = nxt
            if not frontier:
                break
        ch = np.asarray(children, np.int64).reshape(-1, 2)
        # rectangles: origin floor(u*(W-rw)), fixed rw x rh  (types.rs:82-91)
        if ragged_rects:
            ww = rng.integers(0, min(rw * 2, sub_w) + 1, (n_nodes, 2))
            hh = rng.integers(0, min(rh * 2, sub_h) + 1, (n_nodes, 2))
        else:
            ww = np.full((n_nodes, 2), rw)
            hh = np.full((n_nodes, 2), rh)
        ox = np.floor(rng.random((n_nodes, 2)) * (sub_w - ww)).astype(np.int64)
        oy = np.floor(rng.random((n_nodes, 2)) * (sub_h - hh)).astype(np.int64)
        rects = np.stack([ox[:, 0], oy[:, 0], ox[:, 0] + ww[:, 0], oy[:, 0] + hh[:, 0],
                          ox[:, 1], oy[:, 1], ox[:, 1] + ww[:, 1], oy[:, 1] + hh[:, 1]], axis=1).astype(np.int64)
        thr = _q(rng.uniform(-256, 256, n_nodes), 1 / 16).clip(-256, 255.9375)
        if tie_thresholds:
            # thresholds sitting exactly on / next to values avg1 - avg2 can take (multiples of
            # 1/576 for 24x24 rectangles, 0 for identical rectangles): exercises exact ties
            pool = np.array([0.0, -0.0, 1e-12, -1e-12, 1 / 576, -1 / 576, 25 / 576, 1 / 64, -1 / 64, 0.5, -0.5,
                             np.nextafter(1 / 576, 1), np.nextafter(1 / 576, 0), 3.0, -3.0, 1 / 3])
            thr = pool[rng.integers(0, len(pool), n_nodes)]
            same = rng.random(n_nodes) < 0.3
            rects[same, 4:8] = rects[same, 0:4]  # r2 == r1 -> avg1 - avg2 == 0 exactly
        if shuffle_nodes and n_nodes > 2:
            perm = np.concatenate([[0], 1 + rng.permutation(n_nodes - 1)])  # new file position -> old index
            inv = np.empty(n_nodes, np.int64)
            inv[perm] = np.arange(n_nodes)
            rects, thr, ch = rects[perm], thr[perm], ch[perm]
            ch = np.where(ch >= 0, inv[np.clip(ch, 0, None)], ch)
        rects_l.append(rects)
        thr_l.append(thr)
        child_l.append(ch.astype(np.int32))
        node_off.append(node_off[-1] + n_nodes)
        leaf_off.append(leaf_off[-1] + n_leaves)
        n_leaves_total += n_leaves
    NL = n_leaves_total
    # leaves: prob in {0} U [0.5,1], ~60 % >= 0.8
    u = rng.random(NL)
    prob = np.where(u < 0.15, 0.0, np.where(u < 0.40, rng.uniform(0.5, 0.8, NL), rng.uniform(0.8, 1.0, NL)))
    prob = _q(prob, 1 / 1024)
    nv = rng.integers(votes_lo, votes_hi + 1, NL)
    nv = np.where(rng.random(NL) < 0.03, 1, nv)  # a few single-vote leaves (NaN trace -> never vote)
    nv = np.where(prob == 0.0, np.where(rng.random(NL) < 0.5, 0, nv), nv)  # negatives-only leaves may be empty
    vote_off = np.concatenate([[0], np.cumsum(nv)]).astype(np.int64)
    NV = int(vote_off[-1])
    leaf_of_vote = np.repeat(np.arange(NL), nv)
    mu_o = rng.uniform(-80, 80, (NL, 3))
    sd_o = np.where(rng.random(NL) < 0.1, 60.0, 25.0)  # a minority over the 5200 trace gate
    mu_r = rng.uniform(-60, 60, (NL, 3))
    sd_r = np.where(rng.random(NL) < 0.1, 15.0, 6.0)   # a minority over the 400 trace gate
    offsets = _q(mu_o[leaf_of_vote] + rng.normal(0, 1, (NV, 3)) * sd_o[leaf_of_vote, None], 1 / 8).astype(np.float32)
    rotations = _q(mu_r[leaf_of_vote] + rng.normal(0, 1, (NV, 3)) * sd_r[leaf_of_vote, None], 1 / 64)
    return dict(
        n_trees=n_trees,
        tree_node_off=np.asarray(node_off, np.int64),
        tree_leaf_off=np.asarray(leaf_off, np.int64),
        rects=np.concatenate(rects_l).astype(np.int64),
        threshold=np.concatenate(thr_l).astype(np.float64),
        child=np.concatenate(child_l).astype(np.int32),
        prob=prob.astype(np.float64),
        vote_off=vote_off,
        offsets=np.ascontiguousarray(offsets),
        rotations=np.ascontiguousarray(rotations.astype(np.float64)),
        sub_w=sub_w, sub_h=sub_h, max_depth=max_depth,
    )


def forest_to_json(arr: dict, stepwidth: int = 5, gaussian_sigma: float = 8.0, meanshift_iterations: int = 20,
                   sub_w: int | None = None, sub_h: int | None = None) -> str:
    """Serialise to the HoughPrediction JSON document (prediction.rs:239-256).  The depthhead-owned
    structs (NodeParam, LeafParam, Rect, HoughTreeFunctions) follow the reference serde derives;
    the `forest` container layout is the builder-defined stand-in for stamm 0.2.0's (DESIGN.md §3)."""
    sub_w = int(sub_w if sub_w is not None else arr.get("sub_w", 80))
    sub_h = int(sub_h if sub_h is not None else arr.get("sub_h", 80))
    functions = {  # houghforest.rs:89-122 — parsed and ignored by prediction
        "input_size": {"topleft": [0, 0], "bottomright": [sub_w, sub_h]},
        "min_subrect_factor": 0.3, "max_subrect_factor": 0.3, "number_of_gen_features": 2000,
        "steepness": 5.0, "max_depth": int(arr.get("max_depth", 15)), "min_subset_size": 20,
    }
    trees = []
    rects = arr["rects"].tolist()
    thr = arr["threshold"].tolist()
    child = arr["child"].tolist()
    prob = arr["prob"].tolist()
    voff = arr["vote_off"].tolist()
    offs = arr["offsets"].astype(np.float64).tolist()
    rots = arr["rotations"].tolist()
    for t in range(arr["n_trees"]):
        n0, n1 = int(arr["tree_node_off"][t]), int(arr["tree_node_off"][t + 1])
        l0, l1 = int(arr["tree_leaf_off"][t]), int(arr["tree_leaf_off"][t + 1])
        nodes = [{"param": {"r1": {"topleft": r[0:2], "bottomright": r[2:4]},
                            "r2": {"topleft": r[4:6], "bottomright": r[6:8]},
                            "threshold": th},
                  "children": ch}
                 for r, th, ch in zip(rects[n0:n1], thr[n0:n1], child[n0:n1])]
        leaves = [{"prob": prob[i], "offsets": offs[voff[i]:voff[i + 1]], "rotations": rots[voff[i]:voff[i + 1]]}
                  for i in range(l0, l1)]
        trees.append({"functions": functions, "nodes": nodes, "leaves": leaves})
    doc = {
        "stepwidth": int(stepwidth), "subimage_width": sub_w, "subimage_height": sub_h,
        "gaussian_sigma": float(gaussian_sigma), "forest": {"trees": trees},
        "meanshift_iterations": int(meanshift_iterations),
    }
    return json.dumps(doc, separators=(",", ":"))
