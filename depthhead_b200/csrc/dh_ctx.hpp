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
    float* frame_k = nullptr;       // [F][18] K, K^-1 of every frame of a dh_predict_frames pass
    dh_result* results = nullptr;   // [F]
    int32_t* ms_trace = nullptr;    // [F][2][iters][3] (debug export)
    uint32_t* cubes = nullptr;      // [F][2][kBox^3]
    // 2-D back ends (predict_mask, build_hough_image, from2d): allocated by the first such call
    uint32_t* img32 = nullptr;      // [F][h][w] u32 vote sums
    uint16_t* img16 = nullptr;      // [2][F][h][w] horizontal blur, then the image handed out (mask: u8 in the second plane)
    unsigned long long* img_keys = nullptr;  // [F] arg-max keys of the from2d pass
    size_t img_px = 0;              // F * h * w the image scratch holds
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

// What a batch computes after the front end (SAT + traversal) of every chunk.
struct BackEnd {
    enum Kind { kPose, kMask, kVotes, kBlurred } kind = kPose;
    dh_result* results = nullptr;  // kPose: poses [n]; kBlurred: from2d poses [n] or nullptr (host memory)
    const dh_frame_args* args = nullptr;  // kPose: intrinsics and seeds of every frame [n] (host memory), or nullptr:
                                          // the call's one K and no seeds
    void* image = nullptr;         // kMask: u8 [n][h][w]; kVotes / kBlurred: u16 [n][h][w] (kBlurred: may be nullptr)
    bool image_on_device = false;  // image points to device memory on the context's GPU
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
    // Biwi run-length coded frames (biwi.rs:81-103): blob/offsets in host memory, see depthhead_cuda.h
    void biwi_decode(const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h, uint16_t* out, int out_loc);
    void predict_batch_biwi(const HostForest& hf, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h,
                            const float K[9], dh_result* out);
    // dh_predict for every frame with its own arguments: depth at depth_loc, or Biwi files (blob != nullptr)
    void predict_frames(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                        uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* args, dh_result* out);
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
    void build_pair_tables(const HostForest& hf, const std::vector<int32_t>& dev_index);
    void ensure_scratch(const HostForest& hf, uint32_t w, uint32_t h, uint32_t n_frames_hint, const float K[9], int n_lanes = 1);
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
    void ensure_results(uint32_t n);
    void ensure_frame_args(uint32_t n);
    void ensure_image_scratch(int n_lanes);
    void ensure_blur_taps(const HostForest& hf);
    // after run_front: the chunk's back end and the copies of its results (frames f0 .. f0 + n - 1 of the batch)
    void run_chunk_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, uint32_t iterations, const BackEnd& be);
    void run_image_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd& be);
    void flush_pending(Lane& L);
    void free_scratch();
    TilePlan plan_tiles(const Geometry& g) const;
    FrameBuffers buffers(const Lane& L, const uint16_t* depth) const;
    // args: per-frame arguments of the batch (frames f0 .. f0 + n - 1 are this pass's) or nullptr
    void run_front(Lane& L, const FrameBuffers& b, uint32_t n, const FrameState* guess_state, const dh_result* prev_results = nullptr,
                   float min_seed_z = 0.0f, const dh_frame_args* args = nullptr, uint32_t f0 = 0);
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
    // two-levels-per-record tables for the box-sum traversal (PairRec, dh_types.hpp; DH_TRAV_PAIR)
    PairRec* df_pair_recs_ = nullptr;
    PairTopo* df_pair_topo_ = nullptr;
    int32_t* df_pair_roots_ = nullptr;
    int32_t* df_pair_perm_ = nullptr;
    size_t df_n_pairs_ = 0;
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
    dh_result* h_result1_ = nullptr;      // dh_predict's own fixed slot: the D2H copy node of its CUDA graph targets it
    // dh_predict_frames: every frame's FrameState (seeds) and K, K^-1, packed per chunk (grows with the batch)
    FrameState* h_frame_fs_ = nullptr;
    float* h_frame_k_ = nullptr;
    size_t h_frame_cap_ = 0;

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
    bool gate_split_ = true;         // DH_GATE_SPLIT=0: the patch gate inside the seed-grid kernel instead of its own kernel + list
    bool cube_clear_fused_ = true;   // DH_CUBE_CLEAR_FUSED=0: one memset of all cubes per pass instead

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
