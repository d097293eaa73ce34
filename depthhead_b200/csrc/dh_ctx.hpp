// dh_ctx.hpp — per-GPU prediction context (see dh_ctx.cu).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <memory>
#include <utility>
#include <vector>

#include "dh_forest.hpp"
#include "dh_hostenc.hpp"
#include "dh_kernels.cuh"

namespace dh {

// One pipeline lane: a stream plus the per-chunk scratch its kernels work in.  Chunks of a batch
// go round-robin over the lanes, so kernels of different chunks (HBM-bound summed-area tables,
// shared-memory-bound traversal, issue-bound voting, latency-bound mean-shift) overlap on the GPU.
struct Lane {
    cudaStream_t stream = nullptr;  // lane 0: the context's stream; others: their own
    cudaStream_t own = nullptr;
    cudaEvent_t done = nullptr;
    uint32_t* sat = nullptr;        // [F][h+1][pitch]
    uint32_t* band_u = nullptr;     // [F][bands][w+1]
    uint32_t* box = nullptr;        // [F][h-rh+1][pitch] box-sum image (replaces sat/band_u in box-image mode)
    int32_t* leaf = nullptr;        // [F][T][P]
    float* p3 = nullptr;            // [F][P][3]   (debug export)
    uint8_t* gate = nullptr;        // [F][P]      (debug export)
    float4* gated = nullptr;        // [F][P]
    uint32_t* grids = nullptr;      // [F][400 + 8000]
    FrameState* fs = nullptr;       // [F]
    float* frame_k = nullptr;       // [F][18] K, K^-1 of every frame of a pass with per-frame arguments (BackEnd::args)
    dh_result* results = nullptr;   // [F]
    int32_t* ms_trace = nullptr;    // [F][2][iters][3] (debug export)
    uint32_t* cubes = nullptr;      // [F][2][kBox^3]
    // 2-D back ends (predict_mask, build_hough_image, from2d): allocated by the first such call
    uint32_t* img32 = nullptr;      // [F][h][w] u32 vote sums
    uint16_t* img16 = nullptr;      // [2][F][h][w] horizontal blur, then the image handed out (mask: u8 in the second plane)
    unsigned long long* img_keys = nullptr;  // [F] arg-max keys of the from2d pass
    dh_result* img_results = nullptr;        // [F] from2d poses of a pose pass (dh_predict_frames_hough; L.results holds its poses)
    size_t img_px = 0;              // F * h * w the image scratch holds
    // pose back end with host-bound masks (dh_predict_frames_mask): the u8 masks of a chunk, allocated by the first such call
    uint8_t* mask_plane = nullptr;  // [F][h][w]
    size_t mask_px = 0;             // F * h * w it holds
    // dh_predict_frames_heads: the tries of extra heads (HeadsBuffers), allocated by the first such call
    HeadsState* heads_st = nullptr;   // [F]
    uint32_t* heads_grid = nullptr;   // [F][400]
    FrameState* heads_fs = nullptr;   // [F]
    dh_result* heads_res = nullptr;   // [F]
    float4* heads_gated = nullptr;    // [F][P]
    uint32_t* heads_cubes = nullptr;  // [F][2][kBox^3], zero between tries
    dh_head* heads_out = nullptr;     // [F][kMaxHeads]
    uint32_t* heads_n = nullptr;      // [F]
    uint32_t heads_frames = 0;        // F the above hold
    // a host-bound image copy of this lane's last chunk, issued before the lane's next chunk (a copy
    // to pageable memory blocks the host: deferred, it overlaps the other lane's kernels)
    void* pending_dst = nullptr;
    const void* pending_src = nullptr;
    size_t pending_bytes = 0;
    CUtensorMap sat_map{};
    bool allocated = false;
    bool cubes_clean = false;       // every cube is zero (meanshift_kernel cleared behind itself)
};
constexpr int kMaxLanes = 4;

// The checks dh_predict_batch_biwi makes of n + 1 Biwi file offsets (monotone, 4-byte aligned starts,
// files below 4 GB); DH_E_ARG naming the frame
void check_biwi_offsets(const uint64_t* offsets, uint32_t n);

// What a batch computes after the front end (SAT + traversal) of every chunk.
struct BackEnd {
    enum Kind { kPose, kMask, kVotes, kBlurred } kind = kPose;
    dh_result* results = nullptr;  // kPose: poses [n]; kBlurred: from2d poses [n] or nullptr (host memory)
    const dh_frame_args* args = nullptr;  // intrinsics and seeds of every frame [n] (host memory), or nullptr: the call's
                                          // one K and no seeds (kVotes / kBlurred: intrinsics only; kMask: unused)
    void* image = nullptr;         // kMask: u8 [n][h][w]; kVotes / kBlurred: u16 [n][h][w] (kBlurred: may be nullptr);
                                   // kPose: u8 head masks [n][h][w] from the pose pass's own leaf words, or nullptr
    bool image_on_device = false;  // image points to device memory on the context's GPU
    // kPose (dh_predict_frames_hough): the Hough image of the same frames from the pose pass's own leaf
    // words, with the frames' own K; asked for iff image or from2d is set.  Never together with a mask.
    struct Hough {
        bool blur = false;              // build_hough_image, or the vote image before its blur
        uint16_t* image = nullptr;      // u16 [n][h][w], or nullptr (blurred: from2d only)
        bool image_on_device = false;
        dh_result* from2d = nullptr;    // predict_parameter_from2dhough [n] (host memory; needs blur), or nullptr
        bool wanted() const { return image || from2d; }
    } hough;
    // image back ends, and the pose back end with a Hough image, keep image scratch and cap their chunks by it
    bool image_scratch() const { return kind != kPose || hough.wanted(); }
    // kPose (dh_predict_frames_heads): the extra heads of every frame after its pose (run_heads), or nullptr
    const dh_heads_params* heads = nullptr;
    dh_head* heads_out = nullptr;   // [n][max_heads] (host memory)
    uint32_t* n_heads = nullptr;    // [n] (host memory)
};
// Image back ends keep a u32 accumulator and two u16 planes per frame of a chunk (8 bytes per
// pixel, 2.4 MB per VGA frame): their chunks hold at most this much image scratch per lane.
constexpr size_t kImageScratchBytes = 256ull << 20;

struct TrainSet;  // dh_train.cu
void trainset_free(TrainSet* t);

struct ScratchKey {
    uint32_t w = 0, h = 0, sw = 0, sh = 0, stride = 0, n_trees = 0, frames = 0, trace_iters = 0;
    uint32_t rw = 0, rh = 0;  // box-image mode: the forest's common rectangle size (0 = summed-area-table mode)
    bool same_shape(const ScratchKey& o) const {
        return w == o.w && h == o.h && sw == o.sw && sh == o.sh && stride == o.stride && n_trees == o.n_trees &&
               trace_iters == o.trace_iters && rw == o.rw && rh == o.rh;
    }
};

class Context {
public:
    explicit Context(int device);
    ~Context();
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;

    void set_stream(void* s);
    void set_chunk_frames(uint32_t f);
    void set_encode_threads(uint32_t n);   // 0 = default (default_encode_threads()); see run_batch_encoded
    uint32_t encode_threads() const { return pool_ ? pool_->size() : 0u; }
    uint32_t last_encoded_chunks() const { return last_encoded_chunks_; }
    uint64_t last_h2d_bytes() const { return last_h2d_bytes_; }
    void synchronize();
    void enable_timing(bool on) { timing_ = on; }
    void enable_debug(bool on) { debug_ = on; if (!on) have_debug_ = false; }
    const float* stage_ms() const { return stage_ms_; }
    const uint64_t* counters() const { return counters_; }

    void predict(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                 const float* midp_guess, const double* rot_guess, dh_result* out);
    void predict_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                       const float K[9], int depth_loc, dh_result* out);
    // n_seq independent sequences of frames_per_seq frames (sequence-major): frame t of every sequence in one pass,
    // seeded with the pose of frame t - 1 (examples/live_prediction.rs:75-88)
    void predict_sequences(const HostForest& hf, const uint16_t* depth, uint32_t n_seq, uint32_t frames_per_seq, uint32_t w, uint32_t h,
                           const float K[9], int depth_loc, float min_seed_z, dh_result* out);
    // n_seq tracks: track s owns frames [seq_off[s], seq_off[s+1]) of depth at depth_loc, or of the Biwi
    // files of blob / offsets (blob != nullptr); seq_args[s]: its K and the seeds of its first frame
    // mask != nullptr (dh_predict_tracks_mask): also every frame's predict_mask to [total][h][w] u8 at mask_loc, in input order
    void predict_tracks(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n_seq,
                        const uint64_t* seq_off, uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* seq_args, float min_seed_z,
                        dh_result* out, uint8_t* mask = nullptr, int mask_loc = DH_DEPTH_HOST);
    // Biwi run-length coded frames (biwi.rs:81-103): blob/offsets in host memory, see depthhead_cuda.h
    void biwi_decode(const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h, uint16_t* out, int out_loc);
    void predict_batch_biwi(const HostForest& hf, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h,
                            const float K[9], dh_result* out);
    // dh_predict for every frame with its own arguments: depth at depth_loc, or Biwi files (blob != nullptr)
    // mask != nullptr (dh_predict_frames_mask): also every frame's predict_mask to [n][h][w] u8 at mask_loc
    void predict_frames(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                        uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* args, dh_result* out, uint8_t* mask = nullptr,
                        int mask_loc = DH_DEPTH_HOST);
    // the same poses, and every frame's Hough image (blur: build_hough_image, else the raw votes) to
    // [n][h][w] u16 at hough_loc and / or its predict_parameter_from2dhough to from2d [n] (dh_predict_frames_hough)
    void predict_frames_hough(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                              uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* args, dh_result* out, bool blur,
                              uint16_t* hough, int hough_loc, dh_result* from2d);
    // up to params.max_heads heads of every frame (dh_predict_frames_heads): out [n][max_heads], n_heads [n] (host)
    void predict_frames_heads(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                              const dh_frame_args* args, const dh_heads_params& params, dh_head* out, uint32_t* n_heads);
    // training: split scoring (dh_train.cu; houghforest.rs:250-295)
    TrainSet* trainset_create(const uint16_t* patches, uint64_t n, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh,
                              const uint8_t* is_object, const float* offsets, const double* rotations);
    void train_score_level(const TrainSet& ts, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                           const int32_t* cand_rects, const double* cand_thr, uint32_t m, uint64_t depth, double steepness,
                           dh_split_stats* out);
    HostForest* train_forest(const dh_train_params& tp, const uint16_t* patches, uint64_t n, const uint8_t* is_object,
                             const float* offsets, const double* rotations);
    HostForest* train_learn(const dh_train_params& tp, uint32_t n_frames, uint32_t w, uint32_t h, const uint16_t* depth,
                            const uint8_t* mask, const float* K, const float* pos3d, const float* rot);
    void train_split_level(const TrainSet& ts, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                           const int32_t* rects, const double* thr, uint8_t* bits);
    void predict_mask(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, uint8_t* mask);
    // batched 2-D back ends: depth [n][h][w] at depth_loc, images [n][h][w] at image_loc (DH_DEPTH_HOST / DH_DEPTH_DEVICE)
    void predict_mask_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                            uint8_t* mask, int mask_loc);
    void hough_image_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, const float K[9],
                           int depth_loc, bool blur, uint16_t* votes, int votes_loc, dh_result* from2d);
    // the same with frame i's intrinsics at K[9 * i .. 9 * i + 9): depth at depth_loc, or Biwi files (blob != nullptr)
    void hough_image_frames(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                            uint32_t w, uint32_t h, int depth_loc, const float* K, bool blur, uint16_t* votes, int votes_loc,
                            dh_result* from2d);
    void predict_mask_batch_biwi(const HostForest& hf, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h,
                                 uint8_t* mask, int mask_loc);
    void hough_image_raw(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                         uint16_t* votes);
    void hough_image(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9], uint16_t* votes,
                     bool blur, dh_result* from2d);

    void debug_dims(uint32_t* npx, uint32_t* npy, uint32_t* n_trees) const;
    void debug_leaf(int32_t* leaf);
    void debug_patches(float* p3, uint8_t* gate);
    void debug_seeds(uint32_t* guess_pos, uint32_t* guess_rot, int32_t* seed_mid, int32_t* seed_rot);
    void debug_votes(int which, int32_t* keys, uint32_t* vals, uint64_t* n, int32_t* box_origin, int32_t* box_dim);
    void debug_meanshift(int which, int32_t* pos, uint32_t* n_iter);
    void debug_leaf_static(const HostForest& hf, uint32_t* valtoadd, uint8_t* rot_ok, uint8_t* off_ok);
    uint32_t last_ms_flags(int which) const { return last_ms_flags_[which & 1]; }
    const TilePlan& tile_plan() const { return tiles_; }

private:
    void ensure_forest(const HostForest& hf);
    void free_forest();
    // heads: the frames also keep the scratch of extra heads (ensure_heads_scratch), counted in the per-frame budget
    void ensure_scratch(const HostForest& hf, uint32_t w, uint32_t h, uint32_t n_frames_hint, const float K[9], int n_lanes = 1,
                        bool heads = false);
    void alloc_lane(Lane& L);
    void free_lane(Lane& L);
    void ensure_staging(int slots);
    void ensure_biwi(const uint64_t* offsets, uint32_t n, uint32_t chunk, int slots);
    void check_biwi_status(uint32_t n);
    void run_batch(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                   uint32_t h, const float K[9], int depth_loc, const BackEnd& be);
    uint32_t pick_chunk(uint32_t n_frames, int depth_loc) const;
    bool want_encode(uint32_t n, uint32_t w, uint32_t h) const;
    void ensure_encode(uint32_t n, uint32_t F);
    void run_batch_encoded(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, const float K[9],
                           const BackEnd& be);
    void ensure_results(uint32_t n, bool from2d = false);
    void ensure_frame_args(uint32_t n);
    void ensure_image_scratch(int n_lanes);
    void ensure_mask_plane(int n_lanes);
    void ensure_blur_taps(const HostForest& hf);
    void ensure_heads_scratch(int n_lanes);
    void ensure_heads_results(uint32_t n, uint32_t max_heads);
    // kPose with extra heads: the rounds of launch_heads_round after the chunk's back end, and the copies of its heads
    void run_heads(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, uint32_t iterations, const BackEnd& be);
    // after run_front: the chunk's back end and the copies of its results (frames f0 .. f0 + n - 1 of the batch)
    void run_chunk_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, uint32_t iterations, const BackEnd& be);
    void run_image_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd& be);
    // the Hough image of a chunk (kVotes / kBlurred, and the pose back end's Hough destination)
    uint16_t* run_hough(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, bool blur, uint16_t* image, bool image_on_device,
                        dh_result* poses, const float* frame_k);
    // kPose with a mask destination: the chunk's masks from the leaf words its traversal left
    void run_pose_mask(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd& be);
    // kPose with a Hough destination: the chunk's Hough image and from2d poses from the same leaf words
    void run_pose_hough(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd::Hough& hb);
    void flush_pending(Lane& L);
    void free_scratch();
    TilePlan plan_tiles(const Geometry& g) const;
    FrameBuffers buffers(const Lane& L, const uint16_t* depth) const;
    // args: per-frame arguments of the batch (frames f0 .. f0 + n - 1 are this pass's) or nullptr
    // fs_written: a kernel of the caller has already written the pass's frame states (track_guess_kernel)
    void run_front(Lane& L, const FrameBuffers& b, uint32_t n, const FrameState* guess_state, const dh_result* prev_results = nullptr,
                   float min_seed_z = 0.0f, const dh_frame_args* args = nullptr, uint32_t f0 = 0, bool fs_written = false);
    void run_back(Lane& L, const FrameBuffers& b, uint32_t n, uint32_t iterations, const float* frame_k = nullptr);
    void begin_call();
    void end_call();
    cudaEvent_t next_event();
    void mark(int stage);
    void stage_check(const char* name);
    void require_debug() const;

    int device_ = 0;
    int n_sms_ = 148;
    uint32_t smem_optin_ = 0;
    cudaStream_t own_stream_ = nullptr, copy_stream_ = nullptr, stream_ = nullptr;
    static constexpr int kStageSlots = 4;   // device staging slots for host frames: 0, 1 everywhere; 2, 3 the raw stream of the hybrid host path
    cudaEvent_t ev_copied_[kStageSlots] = {nullptr, nullptr, nullptr, nullptr}, ev_consumed_[kStageSlots] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t copy_stream2_ = nullptr;   // raw chunks of the hybrid host path (their own copy stream beside the rewritten chunks')

    // device copy of the model
    uint64_t df_serial_ = 0, df_sigma_version_ = 0;
    size_t df_n_leaves_ = 0;
    NodeRec* df_nodes_ = nullptr;
    HotNode* df_hot_ = nullptr;            // df_nodes_ prepared for tile width hot_tw_ (plan_nodes_kernel)
    uint32_t hot_tw_ = 0;
    cudaTextureObject_t hot_tex_ = 0;
    UniNode* df_uni_ = nullptr;            // uniform-rectangle forests: box-sum nodes for tile width hot_tw_
    uint32_t uni_rw_ = 0, uni_rh_ = 0;
    size_t df_n_nodes_ = 0;
    int32_t* df_roots_ = nullptr;
    double* df_leaf_prob_ = nullptr;
    LeafInfo* df_leaf_info_ = nullptr;
    float4* df_offsets_ = nullptr;
    float* df_offsets3_ = nullptr;
    uint32_t* df_rot_bins_ = nullptr;
    uint32_t* df_rot_cells_ = nullptr;
    LeafBox* df_leaf_box_ = nullptr;
    float* df_kernel_ = nullptr;
    ForestDev fdev_{};
    // taps of build_hough_image's gaussian blur for (blur_serial_, blur_sigma_version_)
    float* d_blur_taps_ = nullptr;
    int blur_radius_ = 0;
    uint64_t blur_serial_ = 0, blur_sigma_version_ = 0;

    // scratch for one chunk of frames
    ScratchKey sk_;
    Geometry geom_{};
    TilePlan tiles_{};
    Lane lanes_[kMaxLanes];
    int max_lanes_ = 2;           // DH_LANES
    cudaEvent_t ev_fork_ = nullptr;
    uint32_t chunk_frames_ = 0;   // 0 = adaptive
    uint32_t call_chunk_ = 1;
    uint16_t* d_depth_[kStageSlots] = {nullptr, nullptr, nullptr, nullptr};
    size_t staging_elems_ = 0;
    unsigned long long* d_counters_ = nullptr;
    // Biwi input: compressed bytes of a chunk (two slots), file offsets, per-frame decode status
    uint8_t* d_blob_[2] = {nullptr, nullptr};
    size_t blob_cap_ = 0;
    unsigned long long* d_offsets_ = nullptr;
    uint32_t* d_status_ = nullptr;
    uint32_t* h_status_ = nullptr;
    size_t biwi_frames_cap_ = 0;

    // Compressed host->device path (run_batch_encoded): worker threads write the frames of a chunk
    // as Biwi run-length files into a pinned slot, in groups of kEncGroup frames; a group owns a
    // fixed region of the slot, so its bytes are known only to the worker that wrote them and the
    // groups are copied one cudaMemcpyAsync each.
    static constexpr int kEncSlots = 3;       // pinned slots: one being copied, two being written
    static constexpr uint32_t kEncGroup = 4;  // most frames per worker task (and per copy of rewritten bytes)
    std::unique_ptr<WorkerPool> pool_;
    uint32_t encode_threads_req_ = 0;
    int host_encode_ = -1;                    // DH_HOST_ENCODE: 0 never, 1 whenever possible, -1 by sampled density
    uint8_t* h_enc_[kEncSlots] = {nullptr, nullptr, nullptr};
    unsigned long long* h_enc_meta_[kEncSlots] = {nullptr, nullptr, nullptr};  // [2][F]: begin, end of every frame inside the slot
    unsigned long long* d_enc_meta_[2] = {nullptr, nullptr};
    cudaEvent_t ev_enc_copied_[kEncSlots] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_copy_tail_ = nullptr;      // after the last copy handed to the copy stream (is the copy engine idle?)
    size_t enc_slot_bytes_ = 0, enc_frame_bound_ = 0;
    uint32_t enc_frames_ = 0;
    uint32_t last_encoded_chunks_ = 0;
    uint64_t last_h2d_bytes_ = 0;

    // pinned host staging
    FrameState* h_fs_ = nullptr;
    unsigned long long* h_counters_ = nullptr;
    dh_result* h_results_ = nullptr;      // batch results (grows with the batch; never referenced by a captured graph)
    size_t h_results_cap_ = 0;
    dh_result* h_from2d_ = nullptr;       // from2d poses of dh_predict_frames_hough, beside the poses in h_results_ (grows likewise)
    size_t h_from2d_cap_ = 0;
    dh_head* h_heads_ = nullptr;          // heads of dh_predict_frames_heads [n][max_heads] (grows likewise)
    uint32_t* h_n_heads_ = nullptr;       // [n]
    size_t h_heads_cap_ = 0, h_n_heads_cap_ = 0;
    dh_result* h_result1_ = nullptr;      // dh_predict's own fixed slot: the D2H copy node of its CUDA graph targets it
    // dh_predict_frames: every frame's FrameState (seeds) and K, K^-1, packed per chunk (grows with the batch)
    FrameState* h_frame_fs_ = nullptr;
    float* h_frame_k_ = nullptr;
    size_t h_frame_cap_ = 0;

    // dh_predict_tracks / dh_predict_sequences (predict_tracks): buffers of the pass loop, grown and kept.
    // Results and slot tables move in windows of passes; none of these depends on the call's frame count.
    struct TrackBuffers {
        TrackSlot* d_plan[2] = {nullptr, nullptr};   // a window's slot tables, by window parity
        TrackSlot* h_plan[2] = {nullptr, nullptr};   // (pinned)
        dh_result* d_win = nullptr;                  // results of the window's passes, [passes][F]
        dh_result* h_win[2] = {nullptr, nullptr};    // (pinned, by window parity)
        size_t win_cap = 0;                          // entries of each of the six above
        TrackArgs* d_tracks = nullptr;               // [n_seq]
        TrackArgs* h_tracks = nullptr;               // (pinned)
        size_t tracks_cap = 0;
        uint8_t* h_blob[2] = {nullptr, nullptr};     // Biwi passes: (start, end) pairs then the files (pinned, by staging slot)
        size_t blob_cap = 0;
        uint32_t* d_status = nullptr;                // [F] decode status of a Biwi pass
        size_t status_cap = 0;
        unsigned long long* d_bad = nullptr;         // lowest bad Biwi frame << 2 | its status
        unsigned long long* h_bad = nullptr;
        cudaEvent_t ev_win[2] = {nullptr, nullptr};  // the window's results are in h_win
        // host-bound masks of dh_predict_tracks_mask: a window's masks in pass order, [passes][F][h][w] u8
        uint8_t* d_mwin[2] = {nullptr, nullptr};     // (device, by window parity; written by track_mask_kernel)
        uint8_t* h_mwin[2] = {nullptr, nullptr};     // (pinned, by window parity)
        size_t mwin_cap = 0;                         // bytes of each of the four above
        cudaEvent_t ev_mwin_ready[2] = {nullptr, nullptr};   // the window's masks are in d_mwin
        cudaEvent_t ev_mwin_copied[2] = {nullptr, nullptr};  // ... and in h_mwin
    } tb_;
    void free_track_buffers();

    // dh_predict as a CUDA graph: the single-frame pipeline is a dozen small launches, i.e. bound
    // by launch overhead; after one eager call with a given (model, shape, intrinsics, stream) the
    // same sequence is captured once and replayed.  Kernel arguments are baked into the graph, so
    // anything they depend on is part of the key.
    struct GraphKey {
        uint64_t serial = 0, sigma_version = 0;
        uint32_t w = 0, h = 0, stride = 0, iterations = 0;
        float K[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        void* stream = nullptr;
        const void* depth = nullptr;
        const void* scratch = nullptr;
        const void* result = nullptr;
        bool operator==(const GraphKey& o) const {
            return serial == o.serial && sigma_version == o.sigma_version && w == o.w && h == o.h && stride == o.stride &&
                   iterations == o.iterations && std::memcmp(K, o.K, sizeof(K)) == 0 && stream == o.stream && depth == o.depth &&
                   scratch == o.scratch && result == o.result;
        }
    };
    void drop_graph();
    cudaGraphExec_t graph_exec_ = nullptr;
    GraphKey graph_key_{}, graph_seen_{};
    bool graph_seen_valid_ = false;
    uint64_t graph_launches_ = 0;
    bool use_graphs_ = true;
    bool prob_codes_ok_ = false;     // the uploaded forest's leaf probabilities can ride in the node table as 8-bit codes
    bool leaf_codes_ = false;        // ... and do: leaf words carry them (FrameBuffers::leaf_mask, patch_gate_kernel)
    uint32_t gate_split_min_ = 64;   // frames per pass from which the patch gate runs as its own kernel (DH_GATE_SPLIT_MIN)
    bool box_whole_ = true;          // DH_BOX_WHOLE=0: every box image through the warp-wide prefix sums
    uint32_t box_bands_ = 0;         // DH_BOX_BANDS: box-image bands per frame (0 = the launch heuristic)
    uint32_t gate_ctas_ = 0;         // DH_GATE_CTAS: seed-grid CTAs per frame on the gated-patch lists (0 = the launch heuristic)

    // measurement
    bool timing_ = false, debug_ = false, have_debug_ = false, debug_sync_ = false;
    uint32_t debug_iterations_ = 0;
    uint32_t last_ms_flags_[2] = {0, 0};
    std::vector<cudaEvent_t> timing_events_;
    size_t ev_used_ = 0;
    std::vector<std::pair<int, cudaEvent_t>> marks_;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> copy_marks_;
    float stage_ms_[DH_N_STAGES];
    uint64_t counters_[DH_N_COUNTERS];
    uint64_t launches_ = 0;
};

}  // namespace dh
