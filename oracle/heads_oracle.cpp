// Several heads per frame (dh_predict_frames_heads) — TEST INFRASTRUCTURE, like everything under oracle/.
//
// Builder-defined rules (DESIGN.md §7 "Several heads per frame"), restated on top of the single-head
// restatement: this file includes depthhead_oracle.cpp, so the seeds, the unbounded sparse accumulators,
// the rotation voting and mean-shift below are that file's, not copies.  It builds its own library
// (oracle/heads.py), which carries the whole oracle C API besides the two calls at the end.
#include "depthhead_oracle.cpp"

namespace {

// ---------------------------------------------------------------- several heads per frame
// Builder-defined (DESIGN.md §7 "Several heads per frame"), restated from its rules 1-7, not from the
// product's kernels.  One try: its seed cell (0xffffffff = the caller's seed), final centre, support.
struct HeadTry {
    int32_t seed[3];
    int32_t centre[3];
    uint64_t support;
    uint32_t seed_cell;
    uint32_t cell_votes;  // the seed cell's count in the working grid when it was chosen (0 for head 0)
    int accepted;
};
// sum of the accumulator over the 20^3 window -10..+9 around c (the cells mean-shift reads)
inline uint64_t window_support(const Sparse3D& acc, const int32_t c[3]) {
    uint64_t s = 0;
    for (int32_t x = -10; x < 10; ++x)
        for (int32_t y = -10; y < 10; ++y)
            for (int32_t z = -10; z < 10; ++z)
                s += acc.get((int32_t)((uint32_t)c[0] + (uint32_t)x), (int32_t)((uint32_t)c[1] + (uint32_t)y),
                             (int32_t)((uint32_t)c[2] + (uint32_t)z));
    return s;
}
// Rule 2: zero every cell of grid whose closed pixel rectangle lies within r_px of the projected centre.
inline void suppress_cells(uint32_t grid[400], const Intrinsic& intr, uint32_t w, uint32_t h, float R, const float mid[3]) {
    float p2[2];
    space_to_img_coord(intr, mid, p2);
    float mx = (p2[0] > 0.0f) ? p2[0] : 0.0f;  // clamped as the coarse grid's votes (prediction.rs:19-25, 661-665)
    float u = (mx < (float)(w - 1)) ? mx : (float)(w - 1);
    float my = (p2[1] > 0.0f) ? p2[1] : 0.0f;
    float v = (my < (float)(h - 1)) ? my : (float)(h - 1);
    const float z = mid[2];
    const float r = z > 0.0f ? (R * intr.k[0]) / z : 0.0f;
    const uint32_t gpw = w / (uint32_t)GUESS_GRID_PARTS, gph = h / (uint32_t)GUESS_GRID_PARTS;
    for (uint32_t i = 0; i < 400; ++i) {
        const uint32_t gx = i % 20, gy = i / 20;
        const float x0 = (float)(gx * gpw), x1 = (float)((gx + 1) * gpw), y0 = (float)(gy * gph), y1 = (float)((gy + 1) * gph);
        const float nx = u < x0 ? x0 : (u > x1 ? x1 : u), ny = v < y0 ? y0 : (v > y1 ? y1 : v);
        const float dx = u - nx, dy = v - ny;
        if (dx * dx + dy * dy <= r * r) grid[i] = 0;
    }
}
// Rules 1-5 after head 0: the tries of a frame in order (head 0 first, accepted).
std::vector<HeadTry> search_heads(const uint32_t guess_pos[400], const Sparse3D& mid, const Image& img, Intrinsic& intr,
                                  const int32_t head0[3], uint32_t head0_cell, uint32_t max_heads, uint32_t min_cell_votes,
                                  float R, const std::vector<float>& kernel, uint32_t iterations) {
    std::vector<HeadTry> tries;
    HeadTry t0;
    std::memcpy(t0.centre, head0, sizeof(t0.centre));
    std::memset(t0.seed, 0, sizeof(t0.seed));
    t0.support = window_support(mid, head0);
    t0.seed_cell = head0_cell;
    t0.cell_votes = 0;
    t0.accepted = 1;
    tries.push_back(t0);
    uint32_t grid[400];
    std::memcpy(grid, guess_pos, sizeof(grid));
    const int64_t fr = (int64_t)std::floor(R), lim = fr * fr;
    uint32_t n_acc = 1;
    for (uint32_t k = 1; k <= 2 * (max_heads - 1) && n_acc < max_heads; ++k) {
        const HeadTry& prev = tries.back();
        const float pm[3] = {(float)prev.centre[0], (float)prev.centre[1], (float)prev.centre[2]};
        suppress_cells(grid, intr, img.w, img.h, R, pm);
        if (prev.seed_cell < 400) grid[prev.seed_cell] = 0;
        uint32_t best = 0, idx = 0;  // first maximum: strict > from (0, 0) (prediction.rs:694-702)
        for (uint32_t i = 0; i < 400; ++i)
            if (grid[i] > best) {
                best = grid[i];
                idx = i;
            }
        if (best < min_cell_votes) break;
        // the reference's seed of that cell (prediction.rs:706-729, 750)
        const size_t gpw = (size_t)img.w / GUESS_GRID_PARTS, gph = (size_t)img.h / GUESS_GRID_PARTS;
        const size_t cx = idx % GUESS_GRID_PARTS, cy = idx / GUESS_GRID_PARTS;
        uint64_t zsum = 0;
        size_t zcnt = 0;
        for (size_t yy = 0; yy < gph; ++yy)
            for (size_t xx = 0; xx < gpw; ++xx) {
                const uint16_t v = img.at((uint32_t)(gpw * cx + xx), (uint32_t)(gph * cy + yy));
                if (v > 0) {
                    zsum += v;
                    zcnt += 1;
                }
            }
        const float meanz = zcnt > 0 ? (float)((double)zsum / (double)zcnt) : 0.0f;
        const float mxy[2] = {((float)cx + 0.5f) * (float)gpw, ((float)cy + 0.5f) * (float)gph};
        float s3[3];
        img_to_space_coord(intr, mxy, meanz, s3);
        HeadTry t;
        t.seed[0] = rs_f32_as_i32(s3[0]);
        t.seed[1] = rs_f32_as_i32(s3[1]);
        t.seed[2] = rs_f32_as_i32(s3[2]);
        const Key3 c = meanshift(mid, Key3{t.seed[0], t.seed[1], t.seed[2]}, kernel, 20, iterations, nullptr, nullptr);
        t.centre[0] = c.x;
        t.centre[1] = c.y;
        t.centre[2] = c.z;
        t.support = window_support(mid, t.centre);
        t.seed_cell = idx;
        t.cell_votes = best;
        t.accepted = 1;
        for (const HeadTry& a : tries) {
            if (!a.accepted) continue;
            const int64_t dx = (int64_t)c.x - a.centre[0], dy = (int64_t)c.y - a.centre[1], dz = (int64_t)c.z - a.centre[2];
            if (dx * dx + dy * dy + dz * dz <= lim) t.accepted = 0;
        }
        n_acc += (uint32_t)t.accepted;
        tries.push_back(t);
    }
    return tries;
}
// Rule 6: the rotation of a head from the gated patches within R of its centre: their coarse rotation grid
// (first maximum: prediction.rs:733-747), their rotation accumulator, mean-shift (prediction.rs:458-482).
// Returns the number of those patches.
uint32_t head_rotation(const Forest& forest, const Trace& tr, const float mid[3], float R, const std::vector<float>& kernel,
                       uint32_t iterations, bool want_rotation, double rotation[3]) {
    const int T = forest.n_trees;
    const size_t P = tr.gate.size();
    Sparse3D rot;
    std::vector<uint32_t> grid(8000, 0u);
    uint32_t n = 0;
    for (size_t p = 0; p < P; ++p) {
        if (!tr.gate[p]) continue;
        const float dx = tr.p3[p * 3 + 0] - mid[0], dy = tr.p3[p * 3 + 1] - mid[1], dz = tr.p3[p * 3 + 2] - mid[2];
        if (!((dx * dx + dy * dy) + dz * dz <= R * R)) continue;
        ++n;
        if (!want_rotation) continue;
        for (int t = 0; t < T; ++t) {  // prediction.rs:588-632 for this patch's leaves
            const int64_t L = tr.leaf[p * T + t];
            const double lp = forest.prob[L];
            if (!(lp > 0.0)) continue;
            const int64_t v0 = forest.vote_off[L], v1 = forest.vote_off[L + 1];
            const size_t nv = (size_t)(v1 - v0);
            const uint32_t valtoadd = (uint32_t)(rs_f64_as_usize(1000.0 * lp) / nv);
            double meanr[3], covr[9];
            estimate_mean_cov<double, 3>(&forest.rotations[(size_t)v0 * 3], nv, meanr, covr);
            if (!(mat_trace<double, 3>(covr) <= MAX_VARIANCE_ROT)) continue;
            for (int64_t v = v0; v < v1; ++v) {
                uint32_t u[3];
                for (int k = 0; k < 3; ++k) {
                    int32_t q = rs_f64_as_i32(forest.rotations[(size_t)v * 3 + k] * (double)ROT_GRID_PARTS / 360.0);
                    int32_t rr = (int32_t)((uint32_t)q + (uint32_t)(ROT_GRID_PARTS / 2));
                    if (rr >= (int32_t)ROT_GRID_PARTS) rr = rr - (int32_t)ROT_GRID_PARTS;
                    else if (rr < 0) rr = (int32_t)ROT_GRID_PARTS + rr;
                    u[k] = (uint32_t)rr;
                }
                rot.add((int32_t)u[0], (int32_t)u[1], (int32_t)u[2], valtoadd);
                const size_t flat = (size_t)(u[2] * 20 / 120) * 400 + (size_t)(u[1] * 20 / 120) * 20 + (size_t)(u[0] * 20 / 120);
                grid[flat] += valtoadd;
            }
        }
    }
    if (!want_rotation) return n;
    uint32_t rx = 0, ry = 0, rz = 0, oldc = 0;
    for (size_t i = 0; i < grid.size(); ++i)
        if (grid[i] > 0 && grid[i] > oldc) {
            oldc = grid[i];
            rz = (uint32_t)(i / 400);
            ry = (uint32_t)((i % 400) / 20);
            rx = (uint32_t)(i % 20);
        }
    const uint32_t rc[3] = {rx, ry, rz};
    int32_t seed[3];
    for (int k = 0; k < 3; ++k) seed[k] = rs_f64_as_i32((((double)rc[k] * 360.0 + 180.0) / (double)GUESS_GRID_PARTS) * (double)ROT_GRID_PARTS / 360.0);
    const Key3 r = meanshift(rot, Key3{seed[0], seed[1], seed[2]}, kernel, 20, iterations, nullptr, nullptr);
    const double half = (double)ROT_GRID_PARTS / 2.0, halfi = (double)(ROT_GRID_PARTS / 2);
    rotation[0] = ((double)r.x - half) / halfi * 3.14159;
    rotation[1] = ((double)r.y - half) / halfi * 3.14159;
    rotation[2] = ((double)r.z - half) / halfi * 3.14159;
    return n;
}

}  // namespace

extern "C" {

// dh_head as the product's header lays it out (72 bytes); a try as orc_predict_heads reports it
struct OrcHead {
    float mid_point[3];
    uint32_t pad;
    double rotation[3];
    uint32_t bbox[4];
    uint64_t support;
    uint32_t n_patches;
    uint32_t seed_cell;
};
static_assert(sizeof(OrcHead) == 72, "OrcHead mirrors dh_head");
struct OrcTry {
    int32_t seed[3];  // 0 for head 0
    int32_t centre[3];
    uint32_t seed_cell;
    uint64_t support;
    int32_t accepted;
    uint32_t cell_votes;
};
static void copy_tries(const std::vector<HeadTry>& tries, OrcTry* out, uint32_t* n_tries) {
    for (size_t i = 0; i < tries.size(); ++i) {
        std::memcpy(out[i].seed, tries[i].seed, sizeof(out[i].seed));
        std::memcpy(out[i].centre, tries[i].centre, sizeof(out[i].centre));
        out[i].seed_cell = tries[i].seed_cell;
        out[i].support = tries[i].support;
        out[i].accepted = tries[i].accepted;
        out[i].cell_votes = tries[i].cell_votes;
    }
    *n_tries = (uint32_t)tries.size();
}

// Rules 2-5 on given inputs: the 20x20 grid, the centre accumulator (keys [n][3], vals [n]), the frame (for
// the seeds' depth) and head 0's centre and seed cell.  tries: room for 2 * max_heads - 1.
int orc_heads_search(const uint32_t* guess_pos, const int32_t* keys, const uint32_t* vals, uint64_t n_cells, const uint16_t* depth,
                     uint32_t w, uint32_t h, const float* K, const int32_t* head0, uint32_t head0_cell, uint32_t max_heads,
                     uint32_t min_cell_votes, float R, float sigma, uint32_t iterations, OrcTry* tries, uint32_t* n_tries) {
    Sparse3D mid;
    for (uint64_t i = 0; i < n_cells; ++i) mid.add(keys[i * 3], keys[i * 3 + 1], keys[i * 3 + 2], vals[i]);
    Image img{depth, w, h};
    Intrinsic intr;
    std::memcpy(intr.k, K, sizeof(float) * 9);
    std::vector<float> kernel;
    build_kernel(20, sigma, kernel);
    copy_tries(search_heads(guess_pos, mid, img, intr, head0, head0_cell, max_heads, min_cell_votes, R, kernel, iterations), tries, n_tries);
    return 0;
}

// Rules 1-7 on a frame: heads [max_heads] (unused slots zero), their count, and every try (room for 2 * max_heads - 1).
int orc_predict_heads(const orc_forest* forest, uint32_t stepwidth, uint32_t sub_w, uint32_t sub_h, float sigma, uint32_t iterations,
                      const uint16_t* depth, uint32_t w, uint32_t h, const float* K, const float* midp_guess, const double* rot_guess,
                      uint32_t max_heads, uint32_t min_cell_votes, float R, int mode, OrcHead* heads, uint32_t* n_heads, OrcTry* tries,
                      uint32_t* n_tries) {
    Params prm{stepwidth, sub_w, sub_h, sigma, iterations};
    Image img{depth, w, h};
    Intrinsic intr;
    std::memcpy(intr.k, K, sizeof(float) * 9);
    Trace tr;
    predict(forest->f, prm, img, intr, midp_guess, rot_guess, mode, 1, true, tr);
    if (tr.error) return tr.error;
    std::vector<float> kernel;
    build_kernel(20, sigma, kernel);
    uint32_t cell0 = 0xffffffffu;
    if (!midp_guess) {
        uint32_t best = 0;
        cell0 = 0;
        for (uint32_t i = 0; i < 400; ++i)
            if (tr.guess_pos[i] > best) {
                best = tr.guess_pos[i];
                cell0 = i;
            }
    }
    const int32_t c0[3] = {(int32_t)tr.mid_point[0], (int32_t)tr.mid_point[1], (int32_t)tr.mid_point[2]};
    const std::vector<HeadTry> all = search_heads(tr.guess_pos, tr.mid, img, intr, c0, cell0, max_heads, min_cell_votes, R, kernel, iterations);
    std::memset(heads, 0, sizeof(OrcHead) * max_heads);
    uint32_t n = 0;
    for (size_t i = 0; i < all.size(); ++i) {
        if (!all[i].accepted) continue;
        OrcHead& o = heads[n++];
        for (int k = 0; k < 3; ++k) o.mid_point[k] = (float)all[i].centre[k];
        o.support = all[i].support;
        o.seed_cell = all[i].seed_cell;
        // head 0 keeps the frame-wide rotation (rule 1); the others take the patches within R (rule 6)
        o.n_patches = head_rotation(forest->f, tr, o.mid_point, R, kernel, iterations, i > 0, o.rotation);
        if (i == 0) std::memcpy(o.rotation, tr.rotation, sizeof(o.rotation));
    }
    *n_heads = n;
    copy_tries(all, tries, n_tries);
    return 0;
}

}  // extern "C"
