// dh_types.hpp — plain structs shared by the host model (dh_forest.cpp) and the CUDA kernels.
#pragma once

#include <cstdint>

namespace dh {

// prediction.rs:270-286 compile-time constants of the reference's prediction path
constexpr int kGuessGridParts = 20;        // GUESS_GRID_PARTS
constexpr int kRotGridParts = 120;         // ROT_GRID_PARTS
constexpr double kMaxVarianceRot = 400.0;  // MAX_VARIANCE_ROT (f64)
constexpr float kMaxVarianceOffset = 5200.0f;  // MAX_VARIANCE_OFFSET (f32)
constexpr int kKernelSize = 20;            // build_kernel(20, sigma), prediction.rs:314
constexpr int kKernelCells = kKernelSize * kKernelSize * kKernelSize;  // 8000
constexpr int kPosGridCells = kGuessGridParts * kGuessGridParts;       // 400
constexpr int kRotGridCells = kGuessGridParts * kGuessGridParts * kGuessGridParts;  // 8000

// One internal node, 32 bytes = exactly one L2 sector.  houghforest.rs:63-68 NodeParam
// (two patch-relative half-open rectangles + f64 threshold) plus the two child links.
// child[bit], bit = (avg1 - avg2 > threshold)  (houghforest.rs:185-193).
// child >= 0: global node index;  child < 0: ~(global leaf id).
struct alignas(32) NodeRec {
    uint8_t r[8];      // r1.x0, r1.y0, r1.x1, r1.y1, r2.x0, r2.y0, r2.x1, r2.y1  (bottomright exclusive)
    double threshold;
    int32_t child[2];
    // threshold * c1 * c2 (pixel counts of the two rectangles, empty -> 1), rounded once: lets the
    // kernel decide the node test by exact integer cross-multiplication away from ties.
    double thr_scaled;
};
static_assert(sizeof(NodeRec) == 32, "NodeRec must be one 32-byte sector");

// The same node prepared for one tile plan (the traversal kernel's hot table, built on the device
// by plan_nodes_kernel whenever the forest or the shared-memory tile width changes).  Everything
// the walk needs is precomputed: per rectangle the word offset of its top-left SAT tap inside the
// shared-memory tile (y0 * tile_width + x0, relative to the patch origin) with width and height,
// the two pixel counts (empty -> 1), the child links and threshold * c1 * c2.  NodeRec stays the
// canonical record and is only read again at near-ties (IEEE-division path).
struct alignas(32) HotNode {
    uint32_t r1;       // off00 | width << 16 | height << 24
    uint32_t r2;
    uint32_t counts;   // c1 | c2 << 16, each max(pixel count, 1) <= 65025
    uint32_t spare;
    int32_t child[2];
    double thr_scaled;
};
static_assert(sizeof(HotNode) == 32, "HotNode must be one 32-byte sector");

// Per-leaf static quantities (prediction.rs:594-600,643 — constant per leaf, recomputed per hit by
// the reference).  Filled on the device by leaf_gate_kernel.
struct alignas(16) LeafInfo {
    uint32_t vote_start;  // first vote in the vote tables
    uint32_t n_votes;     // offsets.len() == rotations.len()
    uint32_t valtoadd;    // ((1000.0*prob) as usize / n) as u32
    uint32_t flags;       // bit0 rot_ok (trace(cov rot) <= 400), bit1 off_ok (trace(cov off) <= 5200),
                          // bit2 votes (prob > 0, valtoadd != 0 and bit0 | bit1)
};
static_assert(sizeof(LeafInfo) == 16, "LeafInfo must be 16 bytes");
// Node of a forest whose feature rectangles all have one size (HostForest::uniform_rw/rh): the
// traversal reads box sums, so a rectangle is ONE tap.  16 bytes = one texture fetch.  e2 encodes
// the threshold for the integer node test 2*(s1 - s2) > e2 (plan_nodes_kernel); an exact
// 2*(s1 - s2) == e2 falls back to NodeRec and IEEE division.
struct alignas(16) UniNode {
    uint32_t taps;     // off00 of rectangle 1 | off00 of rectangle 2 << 16  (y0 * tile_width + x0)
    int32_t child[2];
    int32_t e2;
};
static_assert(sizeof(UniNode) == 16, "UniNode must be 16 bytes");

// Everything the accumulator-cube kernel needs to know about a leaf before it touches its votes, in ONE
// 32-byte sector (the kernel gathers one record per gated patch x tree pair, 13.7 M per 1024 frames of
// configs[1], and the L1 miss path delivers about half a sector per cycle per SM: with LeafInfo and a
// separate 32-byte box it fetched three sectors per pair): the vote range, the weight, the spread
// gates, and the bounding boxes of the votes — rotation bins per axis exactly, offsets (mm) per axis
// as bfloat16 rounded outwards (min towards -inf, max towards +inf), which keeps the skip test
// conservative.  A non-finite offset opens its axis to (-inf, +inf), so such a leaf is never skipped.
struct alignas(32) LeafBox {
    uint32_t vote_start;
    uint32_t n_votes_flags;   // n_votes (< 2^20) | LeafInfo flag bits 0..2 << 24
    uint32_t valtoadd;
    uint8_t rmin[3], rmax0;   // rotation bins in [0, 120)
    uint8_t rmax1, rmax2;
    uint16_t omin0;           // bfloat16 bit patterns
    uint16_t omin1, omin2;
    uint16_t omax[3];
    uint16_t spare;
};
static_assert(sizeof(LeafBox) == 32, "LeafBox must be one 32-byte sector");
constexpr uint32_t kLeafRotOk = 1u, kLeafOffOk = 2u, kLeafVotes = 4u;
// LeafInfo::flags bits 8..31: number of entries of the leaf's compact rotation seed-grid list
// (ForestDev::rot_cells): distinct cells of the 20^3 grid its rotation votes fall into, with their
// multiplicities (the contribution of a leaf to that grid is static, prediction.rs:630-636)
constexpr uint32_t kLeafRotCellsShift = 8u;
constexpr uint32_t kRotCellBits = 13u;                    // 8000 cells
constexpr uint32_t kRotCellMaxCount = (1u << (32u - kRotCellBits)) - 1u;

}  // namespace dh
