// dh_kernels.cuh — launch interfaces of the sm_100a kernels (definitions in dh_kernels.cu).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "dh_types.hpp"
#include "../../include/depthhead_cuda.h"

namespace dh {

// Per-frame device bookkeeping, zeroed at the start of every pipeline pass.
struct alignas(16) FrameState {
    uint32_t n_chits;         // patch x tree pairs that cast centre votes
    uint32_t n_rhits;         // patch x tree pairs that cast rotation votes
    uint32_t n_valid;         // non-background patches
    uint32_t n_gate;          // patches with mean prob > 0.7 = entries of the frame's gated-patch list
    unsigned long long n_mid_votes;  // centre votes the hits cast
    unsigned long long n_rot_votes;
    unsigned long long node_visits;
    int32_t seed_mid[3];
    int32_t seed_rot[3];
    uint32_t ms_iters[2];     // mean-shift rounds actually executed (centre, rotation)
    uint32_t ms_flags[2];     // bit0 zero-sum break
    uint32_t rebuilds[2];     // times the accumulator cube had to be rebuilt around a new position
    int32_t box_org[2][3];    // origin of the accumulator cube (seed - 16, or the last rebuild)
    uint32_t box_valid[2];
    uint32_t has_guess;       // bit0 midp_guess, bit1 rot_guess supplied by the caller
    float midp_guess[3];
    double rot_guess[3];
    uint32_t work_next;       // frame 0's: accumulators handed out to the persistent mean-shift CTAs beyond the first round
    uint32_t active;          // extra heads (launch_heads_round): bit w = accumulator w of this frame's try runs its mean-shift
    unsigned long long support;  // FrameBuffers::support: u32 cells of the centre accumulator in the final 20^3 window
};

struct Geometry {
    uint32_t w, h;            // image
    uint32_t sw, sh;          // sub-image (patch)
    uint32_t left_w, left_h;  // sw/2, sh/2 (prediction.rs:535-538)
    uint32_t stride;          // stepwidth
    uint32_t npx, npy, P;     // patches per row / column / frame
    uint32_t sat_pitch;       // elements per SAT row (multiple of 4)
    uint32_t n_trees;
    uint32_t magic_w, magic_h;  // n / w == umulhi(n, magic_w) for n <= 20 * (w - 1), 0 = divide
    // box-sum image mode (forests whose feature rectangles all have one size rw x rh): the front
    // end writes B[y][x] = sum of the rw x rh rectangle at (x, y) instead of a summed-area table.
    uint32_t rw, rh;          // 0 = summed-area-table mode
    uint32_t box_w, box_h;    // w - rw + 1, h - rh + 1
    uint32_t box_pitch;       // elements per row of B (multiple of 4)
    float K[9], Kinv[9];
    uint32_t gate_pass_codes; // patch gate from 8-bit probability codes (patch_gate_kernel): a code sum >= this passes for certain,
    uint32_t gate_fail_codes; // a code sum + n_trees <= this fails for certain, anything between takes the exact fold
    double gate_min_sum;      // smallest f64 s with fl(s / n_trees) > 0.7: the patch gate of prediction.rs:582-584
                              // without the division (IEEE division by a positive constant is monotone in s)
};

struct TilePlan {
    uint32_t tpx, tpy;        // patches per tile
    uint32_t tiles_x, tiles_y;
    uint32_t tw, th;          // extent of the shared-memory tile in elements (tw multiple of 4): summed-area
                              // table window, or box-sum image window in box-image mode
    uint32_t smem_bytes;
    uint32_t threads;
};

struct ForestDev {
    const NodeRec* nodes;
    const HotNode* hot;        // nodes prepared for the current tile plan (plan_nodes_kernel)
    cudaTextureObject_t hot_tex;  // the same table as a uint4 texture (0 = fetch through the LSU path)
    const UniNode* uni;        // uniform-rectangle forests: 16-byte nodes for the box-sum traversal (or nullptr)
    uint32_t uni_rw, uni_rh;   // the common rectangle size
    const int32_t* roots;
    // Unused: holds the offsets of the fields below, which the kernels that take ForestDev by value
    // read (ptxas schedules patch_gate_kernel and gate_coarse_kernel differently when they move)
    const void* unused_[4];
    const double* leaf_prob;
    const LeafInfo* leaf_info;
    const float4* offsets;     // per vote: x, y, z (mm), w unused — one 16-byte load
    const uint32_t* rot_bins;  // per vote
    const uint32_t* rot_cells;  // per leaf, at its vote_start: compact list of (cell of the 20^3 rotation seed grid | votes in it << 13)
    const LeafBox* leaf_box;   // per leaf: bounding boxes of its votes
    const float* ms_kernel;    // 8000
    int32_t n_trees;
};

struct FrameBuffers {
    const uint16_t* depth;  // [F][h][w]
    uint32_t* sat;          // [F][h+1][pitch]
    uint32_t* band_u;       // [F][bands][w+1] per-band column-sum scans of the banded SAT pass (or nullptr)
    uint32_t* box;          // [F][box_h][box_pitch] box-sum image (box-image mode, else nullptr)
    int32_t* leaf;          // [F][T][P]
    float* p3;              // [F][P][3]
    uint8_t* gate;          // [F][P]
    float4* gated;          // [F][P] gate-passing patches: p3 (prediction.rs:554) + patch index
    uint32_t* grids;        // [F][400 + 8000]
    FrameState* fs;         // [F]
    uint32_t* cubes;        // [F][2][kBox^3] accumulator cubes (centre, rotation), z fastest
    dh_result* results;     // [F]
    int32_t* ms_trace;      // [F][2][iters][3] or nullptr
    uint32_t ms_trace_cap;  // iterations per trace
    uint32_t leaf_mask;     // leaf id = leaf word & leaf_mask: kLeafIdMask when the words carry probability codes, else 0x7fffffff
    uint32_t debug;         // 1: compute the seed grids even when the caller supplied seeds
    uint32_t clear_cubes;   // 1: meanshift_kernel zeroes its accumulator cube when it is done with it (the next
                            // pass finds the cubes empty without a memset of all of them)
    uint32_t support;       // 1: meanshift_kernel sums the final window of every centre accumulator into FrameState::support
};

// Leaf words: the walk stores ~child of the node it left; with probability codes in the uniform node
// table (plan_nodes_kernel) that is leaf id | code << 23, and FrameBuffers::leaf_mask recovers the id.
constexpr uint32_t kProbCodeShift = 23u;
constexpr uint32_t kLeafIdMask = (1u << kProbCodeShift) - 1u;

int launch_sat(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, cudaStream_t s);
// allow_whole: rectangles whose width is a multiple of 8 may take the whole-group box sums (false: every
// width goes through the warp-wide prefix sums); bands: bands per frame, 0 = the launch heuristic
int launch_box_image(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, int n_sms, bool allow_whole, uint32_t bands,
                     cudaStream_t s);
bool box_image_supported(uint32_t w, uint32_t h, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh);
void launch_traverse(const CUtensorMap& sat_map, const FrameBuffers& b, const Geometry& g, const TilePlan& tp,
                     const ForestDev& f, uint32_t n_frames, cudaStream_t s);
void launch_plan_nodes(const NodeRec* nodes, HotNode* hot, UniNode* uni, size_t n_nodes, uint32_t tile_width,
                       const double* prob_codes, cudaStream_t s);
// from_list: the patch gate runs as its own kernel and writes the frames' gated-patch lists; the seed-grid CTAs take
// slices of the lists instead of gating the patches of their own index range.
// want_ctas: seed-grid CTAs per frame of a from_list launch, 0 = the launch heuristic.
// frame_k: nullptr = every frame has Geometry's K / Kinv; else a device table [n_frames][18] of each
// frame's K then K^-1 (row-major), read by the kernels that project (dh_predict_frames).
int launch_gate_coarse(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, bool from_list, int n_sms,
                       uint32_t want_ctas, cudaStream_t s, const float* frame_k = nullptr);
int launch_seed_and_cubes(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames,
                          uint32_t iterations, cudaStream_t s, const float* frame_k = nullptr);
int launch_meanshift(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint32_t iterations,
                     int n_sms, cudaStream_t s);
uint32_t sat_band_rows();
uint32_t vote_box_cells();
uint32_t vote_box_dim();
void launch_leaf_gates(const double* leaf_prob, const uint32_t* vote_start, const uint32_t* n_votes,
                       const float* offsets, const double* rotations, const uint32_t* rot_bins, LeafInfo* out,
                       LeafBox* box_out, uint32_t* rot_cells, uint32_t n_leaves, cudaStream_t s);
// 2-D back ends over n_frames frames (grids carry the frame; per-frame images are [F][h][w]).
// frame_k of the two that project: as in launch_gate_coarse (nullptr = Geometry's K / Kinv).
void launch_mask(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint8_t* mask, cudaStream_t s);
void launch_hough_votes(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint32_t* acc32, cudaStream_t s,
                        const float* frame_k = nullptr);
void launch_narrow_u16(const uint32_t* acc32, uint16_t* out16, size_t n, cudaStream_t s);
// gaussian blur of u32 vote sums narrowed to u16: in -> tmp (horizontal) -> out (vertical; nullptr = not written);
// k: 2 * radius + 1 taps on the device; keys != nullptr: per-frame arg-max keys (zeroed by the caller)
int launch_gaussian_blur(const uint32_t* in, uint16_t* tmp, uint16_t* out, unsigned long long* keys, uint32_t w, uint32_t h,
                         uint32_t n_frames, const float* k, int radius, cudaStream_t s);
void launch_hough2d_pose(const unsigned long long* keys, const uint16_t* depth, const Geometry& g, uint32_t n_frames, dh_result* out,
                         cudaStream_t s, const float* frame_k = nullptr);
// dh_predict_frames_heads: the extra heads of a pose pass (DESIGN.md §7), in rounds after run_back.  Round 0
// writes head 0 (the pass's own result) and starts the search; round k >= 1 serves try k of every frame that is
// still searching: its seed from the working grid, centre cube and mean-shift, the patches within R of the
// centre, their rotation grid, cube and mean-shift, and the head if it is accepted.
constexpr uint32_t kMaxHeads = 8;
struct HeadsState {
    int32_t centre[kMaxHeads][3];  // accepted heads' centres (the mid_points as integers)
    uint32_t n_acc;                // heads accepted so far
    uint32_t searching;            // 0: no further try
    uint32_t seed_cell;            // coarse cell of the current try, 0xffffffff for a caller seed
    uint32_t n_patches;            // gated patches within R of the current try's centre
};
struct HeadsBuffers {
    HeadsState* st;       // [F]
    uint32_t* grid;       // [F][400] working copy of the frame's position grid
    FrameState* fs;       // [F] seeds, cube origins, mean-shift state and support of the current try
    dh_result* res;       // [F] pose of the current try
    float4* gated;        // [F][P] gated patches within R of the current try's centre
    uint32_t* cubes;      // [F][2][kBox^3] the try's accumulator cubes (left empty by the mean-shift CTAs)
    dh_head* out;         // [F][max_heads]
    uint32_t* n_heads;    // [F]
    uint32_t max_heads, min_cell_votes;
    float radius;         // R (mm)
};
// b: the pass's buffers (b.support set, so FrameState::support holds head 0's); frame_k as in launch_gate_coarse
// (the heads call always has per-frame intrinsics).  Returns the launches made.
int launch_heads_round(const FrameBuffers& b, const HeadsBuffers& hb, const Geometry& g, const ForestDev& f, uint32_t n_frames,
                       uint32_t round, uint32_t iterations, int n_sms, const float* frame_k, cudaStream_t s);
void launch_seq_guess(FrameState* fs, const dh_result* prev, uint32_t n, float min_seed_z, cudaStream_t s);

// dh_predict_tracks: one slot of a pass (frame = global frame index, track = its track, prev = the
// track's position in the previous pass or -1 for its first frame) and the arguments of one track
struct TrackSlot {
    int32_t frame, track, prev;
};
struct TrackArgs {
    float K[18];          // K then K^-1 (row-major, K^-1 by mat3_inverse_f32 on the host)
    float midp_guess[3];  // seeds of the track's first frame
    uint32_t has_guess;
    double rot_guess[3];
};
// slot i: frame state and K / K^-1 row (frame_k [n][18]); status (pass-local Biwi decode status) may be nullptr
void launch_track_guess(FrameState* fs, float* frame_k, const TrackSlot* slots, const TrackArgs* tracks, const dh_result* prev,
                        uint32_t n, float min_seed_z, const uint32_t* status, unsigned long long* bad, cudaStream_t s);
// predict_mask of a pass whose frames are scattered over the output: slot i goes to frame slots[i].frame of
// mask ([..][h][w] u8), or to frame frame0 + i * frame_step when slots is nullptr.  Every pixel of those
// frames is written (no memset before it).
void launch_track_mask(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, const TrackSlot* slots,
                       uint32_t frame0, uint32_t frame_step, uint8_t* mask, cudaStream_t s);
// dst[i] = frame slots[i].frame of src (device memory, [..][frame_px] u16)
void launch_track_gather(const uint16_t* src, uint16_t* dst, const TrackSlot* slots, uint32_t n, size_t frame_px, cudaStream_t s);
void launch_counters(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, unsigned long long* out,
                     cudaStream_t s);
// Biwi run-length decode: frame i = blob[offsets[i] - blob_base, offsets[i+1] - blob_base), or up to ends[i] - blob_base
// when `ends` is given (files with gaps between them); out [n][h][w] must be zero
void launch_biwi_decode(const uint8_t* blob, const unsigned long long* offsets, const unsigned long long* ends,
                        unsigned long long blob_base, uint32_t n, uint32_t w, uint32_t h, uint16_t* out, uint32_t* status, cudaStream_t s);
void launch_box_dump(const FrameBuffers& b, uint32_t frame, int which, int32_t* keys, uint32_t* vals,
                     unsigned long long* count, cudaStream_t s);

// smem bytes the traversal kernel needs for a tile (tile + barrier + alignment slack)
uint32_t traverse_smem_bytes(uint32_t tw, uint32_t th, uint32_t patches_per_tile);
int traverse_kernel_attrs(int* regs, int* max_smem);

}  // namespace dh
