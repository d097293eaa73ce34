// dh_ctx.cu — per-GPU context: device copy of the model, scratch, TMA descriptor, and the chunked
// prediction pipeline that stands in for HoughPrediction::predict_parameter_generic
// (prediction.rs:421-493).  Host orchestration only; the arithmetic is in dh_kernels.cu.
#include "dh_ctx.hpp"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

namespace dh {

#define DH_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            throw ModelError(DH_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));            \
    } while (0)

namespace {

template <typename T>
void dev_alloc(T*& p, size_t n) {
    p = nullptr;
    if (n == 0) n = 1;
    DH_CUDA(cudaMalloc(reinterpret_cast<void**>(&p), n * sizeof(T)));
}
template <typename T>
void dev_free(T*& p) {
    if (p) cudaFree((void*)p);
    p = nullptr;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    DH_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !p) throw ModelError(DH_E_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
    fn = reinterpret_cast<PFN_encodeTiled>(p);
    return fn;
}

// frames per chunk of the image back ends: kImageScratchBytes of u32 sums and two u16 planes per lane
uint32_t image_chunk_cap(uint32_t w, uint32_t h) {
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(1u << 30, kImageScratchBytes / (8ull * w * h + 8)));
}

uint32_t env_u32(const char* name, uint32_t dflt) {
    const char* v = std::getenv(name);
    if (!v || !*v) return dflt;
    long x = std::strtol(v, nullptr, 10);
    return x > 0 ? (uint32_t)x : dflt;
}
// on/off switch: "0" turns it off
bool env_flag(const char* name, bool dflt) {
    const char* v = std::getenv(name);
    if (!v || !*v) return dflt;
    return std::strtol(v, nullptr, 10) != 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
Context::Context(int device) : device_(device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        throw ModelError(DH_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                        " (libdepthhead_cuda has no CPU fallback)");
    if (device < 0 || device >= count) throw ModelError(DH_E_ARG, "device index out of range");
    DH_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    DH_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        throw ModelError(DH_E_CUDA, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                                        "; this library contains sm_100a code only");
    n_sms_ = prop.multiProcessorCount;
    smem_optin_ = (uint32_t)prop.sharedMemPerBlockOptin;
    DH_CUDA(cudaStreamCreateWithFlags(&own_stream_, cudaStreamNonBlocking));
    DH_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
    stream_ = own_stream_;
    max_lanes_ = (int)std::min<uint32_t>(kMaxLanes, env_u32("DH_LANES", 2));
    DH_CUDA(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
    for (int i = 0; i < kMaxLanes; ++i) {
        DH_CUDA(cudaEventCreateWithFlags(&lanes_[i].done, cudaEventDisableTiming));
        if (i > 0) DH_CUDA(cudaStreamCreateWithFlags(&lanes_[i].own, cudaStreamNonBlocking));
    }
    DH_CUDA(cudaStreamCreateWithFlags(&copy_stream2_, cudaStreamNonBlocking));
    for (int i = 0; i < kStageSlots; ++i) {
        DH_CUDA(cudaEventCreateWithFlags(&ev_copied_[i], cudaEventDisableTiming));
        DH_CUDA(cudaEventCreateWithFlags(&ev_consumed_[i], cudaEventDisableTiming));
    }
    dev_alloc(d_counters_, DH_N_COUNTERS);
    DH_CUDA(cudaHostAlloc((void**)&h_fs_, sizeof(FrameState), cudaHostAllocDefault));
    DH_CUDA(cudaHostAlloc((void**)&h_counters_, sizeof(unsigned long long) * DH_N_COUNTERS, cudaHostAllocDefault));
    DH_CUDA(cudaHostAlloc((void**)&h_result1_, sizeof(dh_result), cudaHostAllocDefault));
    for (int i = 0; i < kEncSlots; ++i) DH_CUDA(cudaEventCreateWithFlags(&ev_enc_copied_[i], cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
        DH_CUDA(cudaEventCreateWithFlags(&tb_.ev_win[i], cudaEventDisableTiming));
        DH_CUDA(cudaEventCreateWithFlags(&tb_.ev_mwin_ready[i], cudaEventDisableTiming));
        DH_CUDA(cudaEventCreateWithFlags(&tb_.ev_mwin_copied[i], cudaEventDisableTiming));
    }
    DH_CUDA(cudaEventCreateWithFlags(&ev_copy_tail_, cudaEventDisableTiming));
    if (const char* v = std::getenv("DH_HOST_ENCODE")) host_encode_ = *v ? (int)std::strtol(v, nullptr, 10) : -1;
    use_graphs_ = env_flag("DH_GRAPH", true);
    gate_split_min_ = env_u32("DH_GATE_SPLIT_MIN", 64);
    chunk_frames_ = env_u32("DH_CHUNK_FRAMES", 0);  // 0 = adaptive (128 for host input, 512 for device input)
    debug_sync_ = env_u32("DH_DEBUG_SYNC", 0) != 0;
    box_whole_ = env_flag("DH_BOX_WHOLE", true);
    box_bands_ = env_u32("DH_BOX_BANDS", 0);
    gate_ctas_ = env_u32("DH_GATE_CTAS", 0);
    std::memset(stage_ms_, 0, sizeof(stage_ms_));
    std::memset(counters_, 0, sizeof(counters_));
}

Context::~Context() {
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    drop_graph();
    free_scratch();
    free_forest();
    dev_free(d_counters_);
    for (int i = 0; i < 2; ++i) dev_free(d_blob_[i]);
    dev_free(d_offsets_);
    dev_free(d_status_);
    if (h_status_) cudaFreeHost(h_status_);
    if (h_fs_) cudaFreeHost(h_fs_);
    if (h_counters_) cudaFreeHost(h_counters_);
    if (h_results_) cudaFreeHost(h_results_);
    if (h_from2d_) cudaFreeHost(h_from2d_);
    if (h_heads_) cudaFreeHost(h_heads_);
    if (h_n_heads_) cudaFreeHost(h_n_heads_);
    if (h_result1_) cudaFreeHost(h_result1_);
    if (h_frame_fs_) cudaFreeHost(h_frame_fs_);
    if (h_frame_k_) cudaFreeHost(h_frame_k_);
    free_track_buffers();
    for (int i = 0; i < 2; ++i) {
        if (tb_.ev_win[i]) cudaEventDestroy(tb_.ev_win[i]);
        if (tb_.ev_mwin_ready[i]) cudaEventDestroy(tb_.ev_mwin_ready[i]);
        if (tb_.ev_mwin_copied[i]) cudaEventDestroy(tb_.ev_mwin_copied[i]);
    }
    pool_.reset();
    for (int i = 0; i < kEncSlots; ++i) {
        if (h_enc_[i]) cudaFreeHost(h_enc_[i]);
        if (h_enc_meta_[i]) cudaFreeHost(h_enc_meta_[i]);
        if (ev_enc_copied_[i]) cudaEventDestroy(ev_enc_copied_[i]);
    }
    if (ev_copy_tail_) cudaEventDestroy(ev_copy_tail_);
    for (int i = 0; i < 2; ++i) dev_free(d_enc_meta_[i]);
    for (auto ev : timing_events_) cudaEventDestroy(ev);
    if (copy_stream2_) cudaStreamDestroy(copy_stream2_);
    for (int i = 0; i < kStageSlots; ++i) {
        if (ev_copied_[i]) cudaEventDestroy(ev_copied_[i]);
        if (ev_consumed_[i]) cudaEventDestroy(ev_consumed_[i]);
    }
    for (int i = 0; i < kMaxLanes; ++i) {
        if (lanes_[i].done) cudaEventDestroy(lanes_[i].done);
        if (lanes_[i].own) cudaStreamDestroy(lanes_[i].own);
    }
    if (ev_fork_) cudaEventDestroy(ev_fork_);
    if (own_stream_) cudaStreamDestroy(own_stream_);
    if (copy_stream_) cudaStreamDestroy(copy_stream_);
}

void Context::set_stream(void* s) { stream_ = s ? reinterpret_cast<cudaStream_t>(s) : own_stream_; }
void Context::set_chunk_frames(uint32_t f) { chunk_frames_ = f ? std::min<uint32_t>(f, 32768u) : env_u32("DH_CHUNK_FRAMES", 0); }
void Context::set_encode_threads(uint32_t n) {
    if (n != encode_threads_req_) pool_.reset();
    encode_threads_req_ = n;
}
void Context::synchronize() {
    DH_CUDA(cudaSetDevice(device_));
    DH_CUDA(cudaStreamSynchronize(stream_));
}

// ------------------------------------------------------------------------------------------------ model upload
void Context::free_forest() {
    drop_graph();
    dev_free(df_nodes_);
    dev_free(df_hot_);
    dev_free(df_uni_);
    if (hot_tex_) cudaDestroyTextureObject(hot_tex_);
    hot_tex_ = 0;
    hot_tw_ = 0;
    dev_free(df_roots_);
    dev_free(df_leaf_prob_);
    dev_free(df_leaf_info_);
    dev_free(df_offsets_);
    dev_free(df_offsets3_);
    dev_free(df_rot_bins_);
    dev_free(df_rot_cells_);
    dev_free(df_leaf_box_);
    dev_free(df_kernel_);
    df_serial_ = 0;
    dev_free(d_blur_taps_);
    blur_serial_ = 0;
}

void Context::ensure_forest(const HostForest& hf) {
    if (df_serial_ != hf.serial) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        free_forest();
        const size_t NL = hf.n_leaves(), NV = hf.n_votes();
        size_t NN = hf.n_nodes();
        // Node fetches go through the texture path when the table fits a 1-D texture (2^27
        // texels); forests whose rectangles all have one size get the 16-byte box-sum nodes.
        uni_rw_ = uni_rh_ = 0;
        const bool use_tex = env_flag("DH_TEX", true);
        const bool want_uni = NN && env_flag("DH_UNIFORM", true) && hf.uniform_rw && use_tex && NN < (1ull << 26);
        // Device order of the box-sum node table.  The host keeps every tree in breadth-first order
        // (dh_forest.cpp), so the internal children of a node are neighbours; with 16-byte nodes a
        // 32-byte sector holds two of them, and a pad record in front of a pair that would straddle
        // two sectors makes the lanes of a warp that part ways at a node fetch ONE sector for both
        // sides (pads are never visited).  Other forests keep the host order.
        std::vector<NodeRec> dev_nodes;
        std::vector<int32_t> dev_roots(hf.roots);
        if (want_uni) {
            std::vector<int32_t> dev_index(NN, -1);
            int32_t d = 0;
            bool ok = true;
            for (int32_t t = 0; t < hf.n_trees && ok; ++t) {
                const int64_t n0 = hf.tree_node_off[(size_t)t], n1 = hf.tree_node_off[(size_t)t + 1];
                if (n1 == n0) continue;
                dev_index[(size_t)n0] = d++;
                int64_t next = n0 + 1;  // breadth-first: the next node without a place is the next child met
                for (int64_t h = n0; h < n1 && ok; ++h) {
                    const NodeRec& r = hf.nodes[(size_t)h];
                    const int kids = (r.child[0] >= 0 ? 1 : 0) + (r.child[1] >= 0 ? 1 : 0);
                    if (kids == 2 && (d & 1)) ++d;  // the pad
                    for (int b = 0; b < 2; ++b)
                        if (r.child[b] >= 0) {
                            if (r.child[b] != (int32_t)next || next >= n1) { ok = false; break; }
                            dev_index[(size_t)next++] = d++;
                        }
                }
                if (next != n1) ok = false;
            }
            // NN < 2^26 (want_uni) bounds d, pads included, below 2 * NN
            if (!ok || (size_t)d >= (1ull << 27))
                throw ModelError(DH_E_STATE, "internal error: the host node table is not in breadth-first order");
            NodeRec pad;
            std::memset(&pad, 0, sizeof(pad));
            pad.child[0] = pad.child[1] = -1;
            dev_nodes.assign((size_t)d, pad);
            for (size_t h = 0; h < NN; ++h) {
                NodeRec r = hf.nodes[h];
                for (int b = 0; b < 2; ++b)
                    if (r.child[b] >= 0) r.child[b] = dev_index[(size_t)r.child[b]];
                dev_nodes[(size_t)dev_index[h]] = r;
            }
            for (int32_t& r : dev_roots)
                if (r >= 0) r = dev_index[(size_t)r];
            NN = (size_t)d;
        }
        dev_alloc(df_nodes_, NN);
        dev_alloc(df_hot_, NN);
        df_n_nodes_ = NN;
        if (want_uni) {
            dev_alloc(df_uni_, NN);
            uni_rw_ = hf.uniform_rw;
            uni_rh_ = hf.uniform_rh;
        }
        if (use_tex && NN && (df_uni_ || NN * 2 < (1ull << 27))) {
            cudaResourceDesc rd{};
            rd.resType = cudaResourceTypeLinear;
            rd.res.linear.devPtr = df_uni_ ? (void*)df_uni_ : (void*)df_hot_;
            rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
            rd.res.linear.sizeInBytes = df_uni_ ? NN * sizeof(UniNode) : NN * sizeof(HotNode);
            cudaTextureDesc td{};
            td.readMode = cudaReadModeElementType;
            DH_CUDA(cudaCreateTextureObject(&hot_tex_, &rd, &td, nullptr));
        }
        dev_alloc(df_roots_, (size_t)hf.n_trees);
        dev_alloc(df_leaf_prob_, NL);
        dev_alloc(df_leaf_info_, NL);
        dev_alloc(df_offsets_, NV);       // float4 per vote
        dev_alloc(df_offsets3_, NV * 3);  // packed copy, only for the leaf-gate kernel below
        dev_alloc(df_rot_bins_, NV);
        dev_alloc(df_rot_cells_, NV);
        dev_alloc(df_leaf_box_, NL);
        dev_alloc(df_kernel_, (size_t)kKernelCells);
        if (NN)
            DH_CUDA(cudaMemcpyAsync(df_nodes_, dev_nodes.empty() ? hf.nodes.data() : dev_nodes.data(), NN * sizeof(NodeRec),
                                    cudaMemcpyHostToDevice, stream_));
        DH_CUDA(cudaMemcpyAsync(df_roots_, dev_roots.data(), dev_roots.size() * sizeof(int32_t), cudaMemcpyHostToDevice, stream_));
        DH_CUDA(cudaMemcpyAsync(df_leaf_prob_, hf.leaf_prob.data(), NL * sizeof(double), cudaMemcpyHostToDevice, stream_));
        std::vector<float4> off4(NV);
        for (size_t v = 0; v < NV; ++v) off4[v] = make_float4(hf.offsets[v * 3], hf.offsets[v * 3 + 1], hf.offsets[v * 3 + 2], 0.0f);
        if (NV) {
            DH_CUDA(cudaMemcpyAsync(df_offsets_, off4.data(), NV * sizeof(float4), cudaMemcpyHostToDevice, stream_));
            DH_CUDA(cudaMemcpyAsync(df_offsets3_, hf.offsets.data(), NV * 3 * sizeof(float), cudaMemcpyHostToDevice, stream_));
            DH_CUDA(cudaMemcpyAsync(df_rot_bins_, hf.rot_bins.data(), NV * sizeof(uint32_t), cudaMemcpyHostToDevice, stream_));
        }
        // K5: per-leaf covariance-trace gates + valtoadd, computed on the device once per model
        uint32_t *d_vs = nullptr, *d_nv = nullptr;
        double* d_rot = nullptr;
        dev_alloc(d_vs, NL);
        dev_alloc(d_nv, NL);
        dev_alloc(d_rot, NV * 3);
        DH_CUDA(cudaMemcpyAsync(d_vs, hf.leaf_vote_start.data(), NL * sizeof(uint32_t), cudaMemcpyHostToDevice, stream_));
        DH_CUDA(cudaMemcpyAsync(d_nv, hf.leaf_n_votes.data(), NL * sizeof(uint32_t), cudaMemcpyHostToDevice, stream_));
        if (NV) DH_CUDA(cudaMemcpyAsync(d_rot, hf.rotations.data(), NV * 3 * sizeof(double), cudaMemcpyHostToDevice, stream_));
        launch_leaf_gates(df_leaf_prob_, d_vs, d_nv, df_offsets3_, d_rot, df_rot_bins_, df_leaf_info_, df_leaf_box_, df_rot_cells_,
                          (uint32_t)NL, stream_);
        DH_CUDA(cudaGetLastError());
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(d_vs);
        dev_free(d_nv);
        dev_free(d_rot);
        dev_free(df_offsets3_);
        // probability codes in the node table (plan_nodes_kernel, GateTail): 23 bits of leaf id, prob in [0, 1]
        prob_codes_ok_ = NL < (size_t)kLeafIdMask;
        for (size_t l = 0; l < NL && prob_codes_ok_; ++l)
            if (!(hf.leaf_prob[l] >= 0.0 && hf.leaf_prob[l] <= 1.0)) prob_codes_ok_ = false;
        if (!env_flag("DH_PROB_CODES", true)) prob_codes_ok_ = false;
        // the walks store the packed words only from the uniform (box-sum) node table, one level per fetch
        leaf_codes_ = prob_codes_ok_ && df_uni_;
        df_serial_ = hf.serial;
        df_sigma_version_ = 0;
        df_n_leaves_ = NL;
    }
    const uint64_t sv = hf.sigma_version.load();
    if (df_sigma_version_ != sv) {
        // get_or_build_kernel (prediction.rs:310-317): rebuilt lazily after update_sigma
        std::vector<float> k((size_t)kKernelCells);
        build_meanshift_kernel(hf.gaussian_sigma, k.data());
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaMemcpy(df_kernel_, k.data(), k.size() * sizeof(float), cudaMemcpyHostToDevice));
        df_sigma_version_ = sv;
    }
    fdev_.nodes = df_nodes_;
    fdev_.hot = df_hot_;
    fdev_.hot_tex = hot_tex_;
    fdev_.uni = df_uni_;
    fdev_.uni_rw = uni_rw_;
    fdev_.uni_rh = uni_rh_;
    fdev_.roots = df_roots_;
    fdev_.leaf_prob = df_leaf_prob_;
    fdev_.leaf_info = df_leaf_info_;
    fdev_.offsets = df_offsets_;
    fdev_.rot_bins = df_rot_bins_;
    fdev_.rot_cells = df_rot_cells_;
    fdev_.leaf_box = df_leaf_box_;
    fdev_.ms_kernel = df_kernel_;
    fdev_.n_trees = hf.n_trees;
}

// ------------------------------------------------------------------------------------------------ scratch
void Context::free_lane(Lane& L) {
    dev_free(L.sat);
    dev_free(L.band_u);
    dev_free(L.box);
    dev_free(L.leaf);
    dev_free(L.p3);
    dev_free(L.gate);
    dev_free(L.gated);
    dev_free(L.cubes);
    dev_free(L.grids);
    dev_free(L.fs);
    dev_free(L.frame_k);
    dev_free(L.results);
    dev_free(L.ms_trace);
    dev_free(L.img32);
    dev_free(L.img16);
    dev_free(L.img_keys);
    dev_free(L.img_results);
    L.img_px = 0;
    dev_free(L.mask_plane);
    L.mask_px = 0;
    dev_free(L.heads_st);
    dev_free(L.heads_grid);
    dev_free(L.heads_fs);
    dev_free(L.heads_res);
    dev_free(L.heads_gated);
    dev_free(L.heads_cubes);
    dev_free(L.heads_out);
    dev_free(L.heads_n);
    L.heads_frames = 0;
    L.pending_bytes = 0;
    L.allocated = false;
    L.cubes_clean = false;
}

void Context::drop_graph() {
    if (graph_exec_) cudaGraphExecDestroy(graph_exec_);
    graph_exec_ = nullptr;
    graph_seen_valid_ = false;
}

void Context::free_scratch() {
    drop_graph();
    for (int i = 0; i < kStageSlots; ++i) dev_free(d_depth_[i]);
    staging_elems_ = 0;
    for (int i = 0; i < kMaxLanes; ++i) free_lane(lanes_[i]);
    sk_ = ScratchKey();
}

void Context::alloc_lane(Lane& L) {
    const Geometry& g = geom_;
    const size_t F = sk_.frames, P = std::max<uint32_t>(g.P, 1u), T = g.n_trees;
    const uint32_t w = g.w, h = g.h;
    if (g.rw) {
        dev_alloc(L.box, F * (size_t)g.box_h * g.box_pitch);
    } else {
        dev_alloc(L.sat, F * (size_t)(h + 1) * g.sat_pitch);
        DH_CUDA(cudaMemsetAsync(L.sat, 0, F * (size_t)(h + 1) * g.sat_pitch * sizeof(uint32_t), stream_));  // row 0 stays 0
        if (w + 1 <= 1024 && env_flag("DH_SAT_BANDS", true))
            dev_alloc(L.band_u, F * (size_t)((h + sat_band_rows() - 1) / sat_band_rows()) * (w + 1));
    }
    dev_alloc(L.leaf, F * P * T);
    dev_alloc(L.p3, F * P * 3);
    dev_alloc(L.gate, F * P);
    dev_alloc(L.gated, F * P);
    dev_alloc(L.cubes, F * 2 * (size_t)vote_box_cells());
    DH_CUDA(cudaMemsetAsync(L.cubes, 0, sizeof(uint32_t) * F * 2 * (size_t)vote_box_cells(), stream_));
    L.cubes_clean = true;
    dev_alloc(L.grids, F * (size_t)(kPosGridCells + kRotGridCells));
    dev_alloc(L.fs, F);
    dev_alloc(L.frame_k, F * 18);
    dev_alloc(L.results, F);
    if (sk_.trace_iters) dev_alloc(L.ms_trace, F * 2 * (size_t)sk_.trace_iters * 3);
    if (g.P) {
        // TMA descriptor over the SAT scratch [F][h+1][pitch] u32 (or the box-sum image
        // [F][box_h][box_pitch]), box = one tile; out-of-range elements read as zero
        const cuuint64_t gdim[3] = {(cuuint64_t)(g.rw ? g.box_w : w + 1), (cuuint64_t)(g.rw ? g.box_h : h + 1), (cuuint64_t)F};
        const cuuint64_t row_bytes = (cuuint64_t)(g.rw ? g.box_pitch : g.sat_pitch) * 4u;
        const cuuint64_t gstr[2] = {row_bytes, row_bytes * (g.rw ? g.box_h : h + 1)};
        const cuuint32_t box[3] = {tiles_.tw, tiles_.th, 1u};
        const cuuint32_t estr[3] = {1u, 1u, 1u};
        CUresult r = get_encode_fn()(&L.sat_map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, g.rw ? L.box : L.sat, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) throw ModelError(DH_E_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    }
    DH_CUDA(cudaStreamSynchronize(stream_));
    L.allocated = true;
}

TilePlan Context::plan_tiles(const Geometry& g) const {
    // Choose the patch tile that minimises total shared-memory fill traffic per frame, subject to
    // the tile (plus bookkeeping) fitting `limit` bytes so that several CTAs share an SM.
    // 1024-thread CTAs, two per SM, when the tile fits kTwoPerSm bytes; 512-thread CTAs, three per SM,
    // for larger tiles (DH_TRAV_THREADS below 1024 forces them)
    constexpr uint32_t kTwoPerSm = 113000u;  // bytes per CTA that still let two CTAs share an SM
    const bool big = env_u32("DH_TRAV_THREADS", 1024) >= 1024;
    const uint32_t limits[3] = {big ? kTwoPerSm : 75000u, kTwoPerSm, smem_optin_ > 2048u ? smem_optin_ - 1024u : smem_optin_};
    for (uint32_t limit : limits) {
        TilePlan best{};
        double best_cost = 1e300;
        for (uint32_t tpy = 1; tpy <= std::min<uint32_t>(g.npy, 64u); ++tpy)
            for (uint32_t tpx = 1; tpx <= std::min<uint32_t>(g.npx, 64u); ++tpx) {
                // the TMA origin is rounded down to 4 elements (16 B); unless every tile origin is
                // already aligned, the window needs up to 3 extra columns
                const uint32_t slack = ((tpx * g.stride) & 3u) ? 3u : 0u;
                // summed-area table: sw + 1 taps per patch row; box-sum image: sw - rw + 1
                const uint32_t tw = ((tpx - 1) * g.stride + g.sw + 1 - g.rw + slack + 3) & ~3u;
                const uint32_t th = (tpy - 1) * g.stride + g.sh + 1 - g.rh;
                if (tw > 256 || th > 256) continue;  // TMA box limit per dimension
                const uint32_t bytes = traverse_smem_bytes(tw, th, tpx * tpy);
                if (bytes > limit) continue;
                const uint32_t tiles_x = (g.npx + tpx - 1) / tpx, tiles_y = (g.npy + tpy - 1) / tpy;
                // per-tile fixed cost ~ 8 KB equivalent (launch, barrier, compaction)
                const double cost = (double)tiles_x * tiles_y * ((double)tw * th * 4.0 + 8192.0);
                if (cost < best_cost) {
                    best_cost = cost;
                    best = TilePlan{tpx, tpy, tiles_x, tiles_y, tw, th, bytes, (big && limit <= kTwoPerSm) ? 1024u : 512u};
                }
            }
        if (best.tpx) {
            // a warp walks a block of 8 x 4 neighbouring patches (traverse_kernel).  On one node lane (c, r)
            // reads word stride * (c + r * tw) + const: with stride * tw = 8 (mod 32) and an odd stride the
            // 32 lanes hit 32 different banks.
            for (uint32_t tw2 = best.tw; tw2 < best.tw + 32u && tw2 <= 256u; tw2 += 4u) {
                const uint32_t bytes = traverse_smem_bytes(tw2, best.th, best.tpx * best.tpy);
                if (((g.stride * tw2) & 31u) == 8u && bytes <= limit) {
                    best.tw = tw2;
                    best.smem_bytes = bytes;
                    break;
                }
            }
            return best;
        }
    }
    throw ModelError(DH_E_SHAPE, "sub-image too large: its summed-area window does not fit in shared memory");
}

uint32_t Context::pick_chunk(uint32_t n_frames, int depth_loc) const {
    // Host input: small chunks so the H2D copy of chunk c+1 hides behind the kernels of chunk c
    // and the first kernels start early.  Device input: chunks large enough to fill the GPU
    // several times over, small enough that a batch spreads over all pipeline lanes.
    uint32_t c = chunk_frames_ ? chunk_frames_ : (depth_loc == DH_DEPTH_DEVICE ? 512u : 128u);
    return std::max<uint32_t>(1u, std::min<uint32_t>(c, std::max<uint32_t>(n_frames, 1u)));
}

void Context::ensure_scratch(const HostForest& hf, uint32_t w, uint32_t h, uint32_t n_frames_hint, const float K[9], int n_lanes,
                             bool heads) {
    const uint32_t sw = hf.subimage_width, sh = hf.subimage_height, stride = hf.stepwidth.load();
    if (stride == 0) throw ModelError(DH_E_SHAPE, "stepwidth 0: the reference's sliding window never advances");
    if (w < sw || h < sh)
        throw ModelError(DH_E_SHAPE, "image smaller than the sub-image (the reference underflows u32 at prediction.rs:546-548)");
    if (w > 32768 || h > 32768) throw ModelError(DH_E_SHAPE, "image larger than 32768 pixels per side is not supported");
    if (w < (uint32_t)kGuessGridParts || h < (uint32_t)kGuessGridParts)
        throw ModelError(DH_E_SHAPE, "image smaller than 20 pixels per side: the reference's 20x20 seed grid has empty cells");
    // frames per pass: the requested chunk, but never more than ~12 GB of per-frame scratch
    uint32_t cap = std::max<uint32_t>(1u, n_frames_hint);
    {
        const uint64_t npx = (w - sw + stride - 1) / stride, npy = (h - sh + stride - 1) / stride;
        const uint64_t PT = std::max<uint64_t>(npx * npy, 1) * (uint64_t)hf.n_trees;
        const uint64_t per_frame = (uint64_t)(h + 1) * ((w + 4) & ~3ull) * 4 + PT * 4 + npx * npy * 29 +
                                   (uint64_t)w * h * 4 + 2ull * vote_box_cells() * 4 + 40000 +
                                   (heads ? 2ull * vote_box_cells() * 4 + npx * npy * 16 + 4000 : 0ull);
        const uint64_t budget = 12ull << 30;
        cap = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(cap, budget / per_frame));
    }
    ScratchKey k{w, h, sw, sh, stride, (uint32_t)hf.n_trees, cap, debug_ ? hf.meanshift_iterations.load() : 0u};
    if (df_uni_ && env_flag("DH_BOX_IMAGE", true) && box_image_supported(w, h, sw, sh, uni_rw_, uni_rh_)) {
        k.rw = uni_rw_;
        k.rh = uni_rh_;
    }
    call_chunk_ = cap;  // frames per pass of this call (the scratch may be larger)
    Geometry& g = geom_;
    if (!k.same_shape(sk_) || k.frames > sk_.frames) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        free_scratch();
        g = Geometry();
        g.w = w; g.h = h; g.sw = sw; g.sh = sh;
        g.left_w = sw / 2; g.left_h = sh / 2;  // prediction.rs:535-538
        g.stride = stride;
        // y = left_h; while y < h - right_h { .. y += s }  (prediction.rs:544-548,684-686)
        const uint32_t right_w = sw - g.left_w, right_h = sh - g.left_h;
        const uint32_t span_x = (w - right_w) - g.left_w, span_y = (h - right_h) - g.left_h;  // = w - sw, h - sh
        g.npx = span_x == 0 ? 0 : (span_x + stride - 1) / stride;
        g.npy = span_y == 0 ? 0 : (span_y + stride - 1) / stride;
        g.P = g.npx * g.npy;
        g.sat_pitch = (w + 1 + 3) & ~3u;
        g.rw = k.rw;
        g.rh = k.rh;
        if (g.rw) {
            g.box_w = w - g.rw + 1;
            g.box_h = h - g.rh + 1;
            g.box_pitch = (g.box_w + 3) & ~3u;
        }
        g.n_trees = (uint32_t)hf.n_trees;
        // exact division by multiply-high: floor(n / d) == umulhi(n, floor(2^32 / d) + 1) whenever n * d < 2^32
        auto magic = [](uint32_t d) -> uint32_t {
            const uint64_t nmax = (uint64_t)kGuessGridParts * (d - 1);
            return (d >= 2 && nmax * d < (1ull << 32)) ? (uint32_t)((1ull << 32) / d) + 1u : 0u;
        };
        g.magic_w = magic(w);
        g.magic_h = magic(h);
        {
            // prob = sum / n_trees > 0.7 (prediction.rs:582-584) as a comparison of the sum: walk to the
            // smallest double whose rounded quotient exceeds 0.7
            const double t = (double)g.n_trees;
            double smin = 0.7 * t;
            while (smin / t > 0.7) smin = std::nextafter(smin, -HUGE_VAL);
            while (!(smin / t > 0.7)) smin = std::nextafter(smin, HUGE_VAL);
            g.gate_min_sum = smin;
            // the f64 fold of T probabilities differs from their real sum by less than T^2 * 2^-52
            const double slack = t * t * std::ldexp(1.0, -50);
            g.gate_pass_codes = (uint32_t)std::min(4.0e9, std::ceil((smin + slack) * 256.0));
            g.gate_fail_codes = (uint32_t)std::max(0.0, std::min(4.0e9, std::ceil((smin - slack) * 256.0) - 1.0));
        }
        if ((uint64_t)g.P * g.n_trees > 0x7fffffffull) throw ModelError(DH_E_SHAPE, "too many patch x tree pairs per frame");
        if (g.P) tiles_ = plan_tiles(g);
        sk_ = k;
    }
    for (int i = 0; i < std::max(1, std::min(n_lanes, kMaxLanes)); ++i)
        if (!lanes_[i].allocated) alloc_lane(lanes_[i]);
    std::memcpy(g.K, K, sizeof(float) * 9);
    mat3_inverse_f32(K, g.Kinv);
}

void Context::ensure_staging(int slots) {
    const size_t n = (size_t)call_chunk_ * sk_.w * sk_.h;
    if (n > staging_elems_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream2_));
        for (int i = 0; i < kStageSlots; ++i) dev_free(d_depth_[i]);
        staging_elems_ = n;
    }
    for (int i = 0; i < slots && i < kStageSlots; ++i)
        if (!d_depth_[i]) dev_alloc(d_depth_[i], staging_elems_);
}

FrameBuffers Context::buffers(const Lane& L, const uint16_t* depth) const {
    FrameBuffers b{};
    b.depth = depth;
    b.sat = L.sat;
    b.band_u = L.band_u;
    b.box = L.box;
    b.leaf = L.leaf;
    b.p3 = debug_ ? L.p3 : nullptr;      // per-patch exports of debug passes only
    b.gate = debug_ ? L.gate : nullptr;
    b.gated = L.gated;
    b.grids = L.grids;
    b.fs = L.fs;
    b.cubes = L.cubes;
    b.results = L.results;
    b.ms_trace = L.ms_trace;
    b.ms_trace_cap = sk_.trace_iters;
    b.leaf_mask = leaf_codes_ ? kLeafIdMask : 0x7fffffffu;
    b.debug = debug_ ? 1u : 0u;
    b.clear_cubes = debug_ ? 0u : 1u;  // debug passes export the cubes after the call
    b.support = 0;
    return b;
}

// ------------------------------------------------------------------------------------------------ timing helpers
cudaEvent_t Context::next_event() {
    if (ev_used_ == timing_events_.size()) {
        cudaEvent_t e;
        DH_CUDA(cudaEventCreate(&e));
        timing_events_.push_back(e);
    }
    return timing_events_[ev_used_++];
}
void Context::stage_check(const char* name) {
    if (!debug_sync_) return;
    cudaError_t e = cudaStreamSynchronize(stream_);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) throw ModelError(DH_E_CUDA, std::string("stage `") + name + "` failed: " + cudaGetErrorString(e));
}
void Context::mark(int stage_begin_of) {
    if (!timing_) return;
    cudaEvent_t e = next_event();
    DH_CUDA(cudaEventRecord(e, stream_));
    marks_.push_back({stage_begin_of, e});
}

// ------------------------------------------------------------------------------------------------ one pass
// Front end shared by every entry point: SAT + traversal (+ zeroed per-frame state).
void Context::run_front(Lane& L, const FrameBuffers& b, uint32_t n, const FrameState* guess_state, const dh_result* prev_results,
                        float min_seed_z, const dh_frame_args* args, uint32_t f0, bool fs_written) {
    const Geometry& g = geom_;
    cudaStream_t st = L.stream;
    if (args) {
        // per-frame arguments: the pass's frame states (zero but for the seeds, as dh_predict's) and
        // every frame's K, K^-1 (as ensure_scratch computes them for one matrix) replace the memset.
        // Frames keep their index in the batch, so the staging of a chunk is never reused in the call.
        FrameState* hfs = h_frame_fs_ + f0;
        float* hk = h_frame_k_ + (size_t)f0 * 18;
        std::memset(hfs, 0, sizeof(FrameState) * n);
        for (uint32_t i = 0; i < n; ++i) {
            const dh_frame_args& a = args[f0 + i];
            hfs[i].has_guess = a.has_guess;
            if (a.has_guess & 1u)
                for (int k = 0; k < 3; ++k) hfs[i].midp_guess[k] = a.midp_guess[k];
            if (a.has_guess & 2u)
                for (int k = 0; k < 3; ++k) hfs[i].rot_guess[k] = a.rot_guess[k];
            std::memcpy(hk + (size_t)i * 18, a.K, sizeof(float) * 9);
            mat3_inverse_f32(a.K, hk + (size_t)i * 18 + 9);
        }
        DH_CUDA(cudaMemcpyAsync(L.fs, hfs, sizeof(FrameState) * n, cudaMemcpyHostToDevice, st));
        DH_CUDA(cudaMemcpyAsync(L.frame_k, hk, sizeof(float) * 18 * n, cudaMemcpyHostToDevice, st));
    } else if (!fs_written) {
        DH_CUDA(cudaMemsetAsync(L.fs, 0, sizeof(FrameState) * n, st));
    }
    DH_CUDA(cudaMemsetAsync(L.grids, 0, sizeof(uint32_t) * (size_t)(kPosGridCells + kRotGridCells) * n, st));
    if (guess_state) {
        *h_fs_ = *guess_state;
        DH_CUDA(cudaMemcpyAsync(L.fs, h_fs_, sizeof(FrameState), cudaMemcpyHostToDevice, st));
    }
    if (prev_results) {  // seeded sequences: the seeds of this pass are the poses of the previous one, on the device
        launch_seq_guess(L.fs, prev_results, n, min_seed_z, st);
        launches_ += 1;
    }
    if (g.P && hot_tw_ != tiles_.tw) {  // node table for this tile plan (once per forest x plan)
        launch_plan_nodes(df_nodes_, df_hot_, df_uni_, df_n_nodes_, tiles_.tw, leaf_codes_ ? df_leaf_prob_ : nullptr, stream_);
        DH_CUDA(cudaStreamSynchronize(stream_));
        hot_tw_ = tiles_.tw;
    }
    mark(DH_STAGE_SAT);
    launches_ += (uint64_t)(g.rw ? launch_box_image(b, g, n, n_sms_, box_whole_, box_bands_, st) : launch_sat(b, g, n, st));
    stage_check("sat");
    mark(DH_STAGE_TRAVERSE);
    if (g.P) {
        // leaf ids start at -1 (background); the traversal writes the non-background patches only.
        // Every reader decides "background" on the slice of tree 0, so only that slice is filled
        // (36 KB instead of 358 KB per frame); debug passes export all of it and fill all of it.
        if (debug_)
            DH_CUDA(cudaMemsetAsync(L.leaf, 0xFF, sizeof(int32_t) * (size_t)n * g.n_trees * g.P, st));
        else
            DH_CUDA(cudaMemset2DAsync(L.leaf, sizeof(int32_t) * (size_t)g.n_trees * g.P, 0xFF, sizeof(int32_t) * (size_t)g.P, n, st));
        launch_traverse(L.sat_map, b, g, tiles_, fdev_, n, st);
        launches_ += 1;
        stage_check("traverse");
    }
}

void Context::run_back(Lane& L, const FrameBuffers& b, uint32_t n, uint32_t iterations, const float* frame_k) {
    const Geometry& g = geom_;
    cudaStream_t st = L.stream;
    mark(DH_STAGE_GATE);
    // small passes (single frames, the passes of seeded sequences) are bound by the chain of launches: they keep the
    // patch gate inside the seed-grid kernel (one launch less; 0.168 instead of 0.187 ms per single frame)
    launches_ += (uint64_t)launch_gate_coarse(b, g, fdev_, n, n >= gate_split_min_, n_sms_, gate_ctas_, st, frame_k);
    stage_check("gate + coarse grids");
    mark(DH_STAGE_VOTE);
    // the accumulator cubes of this pass start empty: either the previous pass's mean-shift CTAs
    // cleared them behind themselves, or they are cleared here
    if (iterations && !L.cubes_clean) DH_CUDA(cudaMemsetAsync(L.cubes, 0, sizeof(uint32_t) * 2 * (size_t)vote_box_cells() * n, st));
    if (iterations) L.cubes_clean = false;
    launches_ += (uint64_t)launch_seed_and_cubes(b, g, fdev_, n, iterations, st, frame_k);
    stage_check("seeds + accumulator cubes");
    mark(DH_STAGE_MEANSHIFT);
    launches_ += (uint64_t)launch_meanshift(b, g, fdev_, n, iterations, n_sms_, st);
    if (b.clear_cubes) L.cubes_clean = true;
    stage_check("mean-shift");
    mark(DH_STAGE_D2H);
    launch_counters(b, g, n, d_counters_, st);
    launches_ += 1;
    DH_CUDA(cudaGetLastError());
}

void Context::begin_call() {
    DH_CUDA(cudaSetDevice(device_));
    lanes_[0].stream = stream_;
    for (int i = 1; i < kMaxLanes; ++i) lanes_[i].stream = lanes_[i].own;
    for (int i = 0; i < kMaxLanes; ++i) lanes_[i].pending_bytes = 0;  // (left behind by a call that failed)
    launches_ = 0;
    ev_used_ = 0;
    marks_.clear();
    std::memset(stage_ms_, 0, sizeof(stage_ms_));
    DH_CUDA(cudaMemsetAsync(d_counters_, 0, sizeof(unsigned long long) * DH_N_COUNTERS, stream_));
}

void Context::end_call() {
    DH_CUDA(cudaMemcpyAsync(h_counters_, d_counters_, sizeof(unsigned long long) * DH_N_COUNTERS, cudaMemcpyDeviceToHost, stream_));
    DH_CUDA(cudaStreamSynchronize(stream_));
    for (int k = 0; k < DH_N_COUNTERS; ++k) counters_[k] = h_counters_[k];
    counters_[9] = launches_;
    if (timing_) {
        // marks_ are (stage that begins here, event); a stage lasts until the next mark
        for (size_t i = 0; i + 1 < marks_.size(); ++i) {
            if (marks_[i].first < 0) continue;
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, marks_[i].second, marks_[i + 1].second) == cudaSuccess) stage_ms_[marks_[i].first] += ms;
        }
        for (auto& c : copy_marks_) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, c.first, c.second) == cudaSuccess) stage_ms_[DH_STAGE_H2D] += ms;
        }
    }
    copy_marks_.clear();
}

// ------------------------------------------------------------------------------------------------ public entry points
void Context::predict(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                      const float* midp_guess, const double* rot_guess, dh_result* out) {
    begin_call();
    ensure_forest(hf);
    ensure_scratch(hf, w, h, 1, K);
    ensure_staging(1);
    const uint32_t iterations = hf.meanshift_iterations.load();
    DH_CUDA(cudaMemcpyAsync(d_depth_[0], depth, (size_t)w * h * sizeof(uint16_t), cudaMemcpyHostToDevice, stream_));
    FrameState gs;
    std::memset(&gs, 0, sizeof(gs));
    if (midp_guess) {
        gs.has_guess |= 1u;
        for (int k = 0; k < 3; ++k) gs.midp_guess[k] = midp_guess[k];
    }
    if (rot_guess) {
        gs.has_guess |= 2u;
        for (int k = 0; k < 3; ++k) gs.rot_guess[k] = rot_guess[k];
    }
    // everything after the input copy: per-frame state, front end, back end, result and counters to pinned memory
    auto enqueue = [&] {
        FrameBuffers b = buffers(lanes_[0], d_depth_[0]);
        run_front(lanes_[0], b, 1, &gs);
        run_back(lanes_[0], b, 1, iterations);
        DH_CUDA(cudaMemcpyAsync(h_result1_, lanes_[0].results, sizeof(dh_result), cudaMemcpyDeviceToHost, stream_));
    };
    bool replayed = false;
    // (a pass that left the cubes dirty — a debug pass — must be followed by an eager pass, which clears them)
    if (use_graphs_ && !timing_ && !debug_ && !debug_sync_ && lanes_[0].cubes_clean) {
        GraphKey key;
        key.serial = hf.serial; key.sigma_version = df_sigma_version_;
        key.w = w; key.h = h; key.stride = geom_.stride; key.iterations = iterations;
        std::memcpy(key.K, K, sizeof(key.K));
        key.stream = (void*)stream_; key.depth = d_depth_[0]; key.scratch = lanes_[0].fs; key.result = h_result1_;
        if (graph_exec_ && !(graph_key_ == key)) drop_graph();
        if (!graph_exec_ && graph_seen_valid_ && graph_seen_ == key) {
            // second call with this key: capture the sequence (the first, eager call planned the node
            // table and configured every kernel)
            cudaGraph_t graph = nullptr;
            const uint64_t before = launches_;
            if (cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
                cudaGetLastError();
                use_graphs_ = false;  // e.g. the legacy default stream: eager launches for the rest of this context's life
            } else {
                try {
                    enqueue();
                } catch (...) {
                    cudaStreamEndCapture(stream_, &graph);
                    if (graph) cudaGraphDestroy(graph);
                    throw;
                }
                cudaError_t e = cudaStreamEndCapture(stream_, &graph);
                graph_launches_ = launches_ - before;
                launches_ = before;
                if (e == cudaSuccess) e = cudaGraphInstantiate(&graph_exec_, graph, 0);
                if (graph) cudaGraphDestroy(graph);
                if (e != cudaSuccess) {
                    graph_exec_ = nullptr;
                    use_graphs_ = false;
                    cudaGetLastError();
                } else {
                    graph_key_ = key;
                }
            }
        }
        graph_seen_ = key;
        graph_seen_valid_ = true;
        if (graph_exec_) {
            *h_fs_ = gs;  // the graph's copy node reads the caller's seeds from this pinned struct
            DH_CUDA(cudaGraphLaunch(graph_exec_, stream_));
            launches_ += graph_launches_;
            replayed = true;
        }
    }
    if (!replayed) enqueue();
    mark(-1);
    end_call();
    *out = *h_result1_;
    have_debug_ = debug_;
    debug_iterations_ = iterations;
}

void Context::predict_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                            const float K[9], int depth_loc, dh_result* out) {
    BackEnd be;
    be.results = out;
    run_batch(hf, depth, nullptr, nullptr, n, w, h, K, depth_loc, be);
}

void Context::predict_batch_biwi(const HostForest& hf, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                                 uint32_t h, const float K[9], dh_result* out) {
    BackEnd be;
    be.results = out;
    run_batch(hf, nullptr, blob, offsets, n, w, h, K, DH_DEPTH_HOST, be);
}

// dh_predict_frames / dh_predict_frames_biwi: the pose pipeline of dh_predict_batch, every frame with
// the arguments of its own dh_predict call.  The kernels that project read the frame's K, K^-1 from
// the lane's table (Lane::frame_k); the call's matrix in Geometry (frame 0's) is not used.
// With a mask destination (dh_predict_frames_mask) the back end also writes predict_mask of every
// frame from the leaf words of the same traversal (run_pose_mask): chunks, lanes and staging stay
// those of the pose call.
void Context::predict_frames(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                             uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* args, dh_result* out, uint8_t* mask,
                             int mask_loc) {
    static const float kIdentity[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    BackEnd be;
    be.results = out;
    be.args = args;
    be.image = mask;
    be.image_on_device = mask_loc == DH_DEPTH_DEVICE;
    run_batch(hf, depth, blob, offsets, n, w, h, n ? args[0].K : kIdentity, blob ? DH_DEPTH_HOST : depth_loc, be);
}

// dh_predict_frames_hough / _biwi: the poses of predict_frames, and what hough_image_frames computes with
// K[i] = args[i].K, from the leaf words of the same traversal (run_pose_hough).  Chunks, lanes and image
// scratch are those of the 2-D calls (image_chunk_cap), so that scratch stays bounded per lane.
void Context::predict_frames_hough(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                                   uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* args, dh_result* out, bool blur,
                                   uint16_t* hough, int hough_loc, dh_result* from2d) {
    static const float kIdentity[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    BackEnd be;
    be.results = out;
    be.args = args;
    be.hough.blur = blur;
    be.hough.image = hough;
    be.hough.image_on_device = hough_loc == DH_DEPTH_DEVICE;
    be.hough.from2d = from2d;
    run_batch(hf, depth, blob, offsets, n, w, h, n ? args[0].K : kIdentity, blob ? DH_DEPTH_HOST : depth_loc, be);
}

// dh_predict_frames_heads: the pose pipeline of predict_frames, then the extra heads of every chunk (run_heads)
void Context::predict_frames_heads(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                                   const dh_frame_args* args, const dh_heads_params& params, dh_head* out, uint32_t* n_heads) {
    static const float kIdentity[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    BackEnd be;
    be.args = args;
    be.heads = &params;
    be.heads_out = out;
    be.n_heads = n_heads;
    run_batch(hf, depth, nullptr, nullptr, n, w, h, n ? args[0].K : kIdentity, depth_loc, be);
}

void check_biwi_offsets(const uint64_t* offsets, uint32_t n) {
    for (uint32_t i = 0; i < n; ++i) {
        if (offsets[i + 1] < offsets[i]) throw ModelError(DH_E_ARG, "Biwi offsets are not monotone at frame " + std::to_string(i));
        if (offsets[i] & 3u) throw ModelError(DH_E_ARG, "Biwi frame " + std::to_string(i) + " does not start at a multiple of 4 bytes");
        if (offsets[i + 1] - offsets[i] > 0xfffffff0ull) throw ModelError(DH_E_ARG, "Biwi frame " + std::to_string(i) + " is larger than 4 GB");
    }
}

namespace {
// DH_E_ARG for Biwi frame i, whose decode status is `status` (biwi_decode_kernel)
[[noreturn]] void throw_biwi_status(size_t i, uint32_t status) {
    static const char* what[] = {"", "is truncated (the reference fails with UnexpectedEof, biwi.rs:90-96)",
                                 "has a run past the last pixel (the reference panics, biwi.rs:92,97)",
                                 "has a header that differs from the requested width x height"};
    throw ModelError(DH_E_ARG, "Biwi frame " + std::to_string(i) + " " + what[std::min<uint32_t>(status, 3u)]);
}
}  // namespace

// Device copies of the file offsets and room for the compressed bytes of one chunk per slot.
void Context::ensure_biwi(const uint64_t* offsets, uint32_t n, uint32_t chunk, int slots) {
    check_biwi_offsets(offsets, n);
    size_t need = 0;
    for (uint32_t f0 = 0; f0 < n; f0 += chunk) need = std::max<size_t>(need, (size_t)(offsets[std::min(n, f0 + chunk)] - offsets[f0]));
    need += 64;  // the decode kernel reads whole 4-byte words
    if (need > blob_cap_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream_));
        for (int i = 0; i < 2; ++i) dev_free(d_blob_[i]);
        blob_cap_ = need;
    }
    for (int i = 0; i < slots && i < 2; ++i)
        if (!d_blob_[i]) dev_alloc(d_blob_[i], blob_cap_);
    if ((size_t)n + 1 > biwi_frames_cap_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(d_offsets_);
        dev_free(d_status_);
        if (h_status_) cudaFreeHost(h_status_);
        h_status_ = nullptr;
        biwi_frames_cap_ = (size_t)n + 1;
        dev_alloc(d_offsets_, biwi_frames_cap_);
        dev_alloc(d_status_, biwi_frames_cap_);
        DH_CUDA(cudaHostAlloc((void**)&h_status_, sizeof(uint32_t) * biwi_frames_cap_, cudaHostAllocDefault));
    }
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "offset width");
    DH_CUDA(cudaMemcpyAsync(d_offsets_, offsets, sizeof(uint64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, stream_));
}

void Context::check_biwi_status(uint32_t n) {
    DH_CUDA(cudaMemcpyAsync(h_status_, d_status_, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, stream_));
    DH_CUDA(cudaStreamSynchronize(stream_));
    for (uint32_t i = 0; i < n; ++i)
        if (h_status_[i]) throw_biwi_status(i, h_status_[i]);
}

void Context::biwi_decode(const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h, uint16_t* out,
                          int out_loc) {
    begin_call();
    have_debug_ = false;
    if (n == 0) {
        end_call();
        return;
    }
    if ((uint64_t)w * h == 0 || (uint64_t)w * h > 0x3fffffffull) throw ModelError(DH_E_SHAPE, "Biwi frame of 0 or more than 2^30 pixels");
    const size_t frame_px = (size_t)w * h;
    const uint32_t chunk = std::max<uint32_t>(1u, (uint32_t)std::min<uint64_t>(n, (1ull << 30) / (frame_px * 2)));
    ensure_biwi(offsets, n, chunk, 1);
    uint16_t* d_out = out;
    uint16_t* tmp = nullptr;
    if (out_loc != DH_DEPTH_DEVICE) {
        dev_alloc(tmp, (size_t)chunk * frame_px);
        d_out = tmp;
    }
    try {
        for (uint32_t f0 = 0; f0 < n; f0 += chunk) {
            const uint32_t nc = std::min(chunk, n - f0);
            uint16_t* dst = out_loc == DH_DEPTH_DEVICE ? d_out + (size_t)f0 * frame_px : d_out;
            DH_CUDA(cudaMemcpyAsync(d_blob_[0], blob + offsets[f0], (size_t)(offsets[f0 + nc] - offsets[f0]), cudaMemcpyHostToDevice, stream_));
            DH_CUDA(cudaMemsetAsync(dst, 0, (size_t)nc * frame_px * sizeof(uint16_t), stream_));
            launch_biwi_decode(d_blob_[0], d_offsets_ + f0, nullptr, offsets[f0], nc, w, h, dst, d_status_ + f0, stream_);
            launches_ += 1;
            DH_CUDA(cudaGetLastError());
            if (out_loc != DH_DEPTH_DEVICE)
                DH_CUDA(cudaMemcpyAsync(out + (size_t)f0 * frame_px, dst, (size_t)nc * frame_px * sizeof(uint16_t), cudaMemcpyDeviceToHost, stream_));
            DH_CUDA(cudaStreamSynchronize(stream_));  // d_blob_[0] (and tmp) are reused by the next chunk
        }
        check_biwi_status(n);
    } catch (...) {
        cudaStreamSynchronize(stream_);
        dev_free(tmp);
        end_call();
        throw;
    }
    dev_free(tmp);
    mark(-1);
    end_call();
}

void Context::run_batch(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                        uint32_t w, uint32_t h, const float K[9], int depth_loc, const BackEnd& be) {
    begin_call();
    have_debug_ = false;
    if (n == 0) {
        end_call();
        return;
    }
    ensure_forest(hf);
    last_encoded_chunks_ = 0;
    last_h2d_bytes_ = 0;
    if (!blob && depth_loc != DH_DEPTH_DEVICE && want_encode(n, w, h)) {
        run_batch_encoded(hf, depth, n, w, h, K, be);
        return;
    }
    // Chunks go round-robin over the lanes.  Stage timing needs the kernels of a pass back to
    // back on one stream, so it runs single-lane.
    // Biwi input: the run-length expansion is latency-bound (one thread per frame walks the run
    // headers), so its chunks are larger: more frames in flight per launch
    uint32_t want_chunk = (blob && !chunk_frames_) ? std::min<uint32_t>(512u, n) : pick_chunk(n, depth_loc);
    if (be.image_scratch()) want_chunk = std::min(want_chunk, image_chunk_cap(w, h));
    const int n_lanes = timing_ ? 1 : (int)std::max<uint32_t>(1u, std::min<uint32_t>((uint32_t)max_lanes_, (n + want_chunk - 1) / want_chunk));
    ensure_scratch(hf, w, h, want_chunk, K, n_lanes, be.heads != nullptr);
    if (be.image_scratch()) ensure_image_scratch(n_lanes);
    if (be.heads) ensure_heads_scratch(n_lanes);
    if (be.kind == BackEnd::kPose && be.image && !be.image_on_device) ensure_mask_plane(n_lanes);
    if (be.kind == BackEnd::kBlurred || be.hough.blur) ensure_blur_taps(hf);
    const uint32_t iterations = hf.meanshift_iterations.load();
    const uint32_t F = call_chunk_;
    const uint32_t n_chunks = (n + F - 1) / F;
    const size_t frame_px = (size_t)w * h;
    ensure_results(n, be.hough.from2d != nullptr);
    if (be.heads) ensure_heads_results(n, be.heads->max_heads);  // pinned staging for the results
    if (be.args) ensure_frame_args(n);
    if (depth_loc != DH_DEPTH_DEVICE) ensure_staging(2);
    if (blob) ensure_biwi(offsets, n, F, 2);
    // fork: the other lanes (and the copy stream) start after everything already queued on the caller's stream
    DH_CUDA(cudaEventRecord(ev_fork_, stream_));
    for (int i = 1; i < n_lanes; ++i) DH_CUDA(cudaStreamWaitEvent(lanes_[i].stream, ev_fork_, 0));
    auto enqueue_chunk = [&](uint32_t c, const uint16_t* d_depth) {
        Lane& L = lanes_[c % (uint32_t)n_lanes];
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        FrameBuffers b = buffers(L, d_depth);
        flush_pending(L);
        run_front(L, b, nc, nullptr, nullptr, 0.0f, be.args, f0);
        run_chunk_back(L, b, f0, nc, iterations, be);
    };
    if (depth_loc == DH_DEPTH_DEVICE) {
        for (uint32_t c = 0; c < n_chunks; ++c) enqueue_chunk(c, depth + (size_t)c * F * frame_px);
    } else {
        // double-buffered staging: the copy of chunk c+1 overlaps the kernels of chunk c.  Biwi
        // input: the COMPRESSED bytes are copied, and the lane expands them into the staging slot.
        for (uint32_t c = 0; c < n_chunks; ++c) {
            const int slot = (int)(c & 1u);
            Lane& L = lanes_[c % (uint32_t)n_lanes];
            const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
            if (c >= 2) DH_CUDA(cudaStreamWaitEvent(copy_stream_, ev_consumed_[slot], 0));
            else DH_CUDA(cudaStreamWaitEvent(copy_stream_, ev_fork_, 0));
            cudaEvent_t t0 = nullptr, t1 = nullptr;
            if (timing_) {
                t0 = next_event();
                t1 = next_event();
                DH_CUDA(cudaEventRecord(t0, copy_stream_));
            }
            if (blob) {
                DH_CUDA(cudaMemcpyAsync(d_blob_[slot], blob + offsets[f0], (size_t)(offsets[f0 + nc] - offsets[f0]), cudaMemcpyHostToDevice,
                                        copy_stream_));
                last_h2d_bytes_ += (uint64_t)(offsets[f0 + nc] - offsets[f0]);
            } else {
                DH_CUDA(cudaMemcpyAsync(d_depth_[slot], depth + (size_t)f0 * frame_px, (size_t)nc * frame_px * sizeof(uint16_t),
                                        cudaMemcpyHostToDevice, copy_stream_));
                last_h2d_bytes_ += (uint64_t)nc * frame_px * sizeof(uint16_t);
            }
            if (timing_) {
                DH_CUDA(cudaEventRecord(t1, copy_stream_));
                copy_marks_.push_back({t0, t1});
            }
            DH_CUDA(cudaEventRecord(ev_copied_[slot], copy_stream_));
            DH_CUDA(cudaStreamWaitEvent(L.stream, ev_copied_[slot], 0));
            if (blob) {
                mark(DH_STAGE_H2D);  // the expansion counts as input transfer
                DH_CUDA(cudaMemsetAsync(d_depth_[slot], 0, (size_t)nc * frame_px * sizeof(uint16_t), L.stream));
                launch_biwi_decode(d_blob_[slot], d_offsets_ + f0, nullptr, offsets[f0], nc, w, h, d_depth_[slot], d_status_ + f0, L.stream);
                launches_ += 1;
            }
            enqueue_chunk(c, d_depth_[slot]);
            DH_CUDA(cudaEventRecord(ev_consumed_[slot], L.stream));
        }
    }
    for (int i = 0; i < n_lanes; ++i) flush_pending(lanes_[i]);
    if (n_lanes > 1) {  // join: the caller's stream continues after every lane
        for (int i = 1; i < n_lanes; ++i) {
            DH_CUDA(cudaEventRecord(lanes_[i].done, lanes_[i].stream));
            DH_CUDA(cudaStreamWaitEvent(stream_, lanes_[i].done, 0));
        }
    }
    mark(-1);
    DH_CUDA(cudaStreamSynchronize(stream_));
    end_call();
    if (blob) check_biwi_status(n);
    if (be.results) std::memcpy(be.results, h_results_, sizeof(dh_result) * n);
    if (be.hough.from2d) std::memcpy(be.hough.from2d, h_from2d_, sizeof(dh_result) * n);
    if (be.heads) {
        std::memcpy(be.heads_out, h_heads_, sizeof(dh_head) * n * be.heads->max_heads);
        std::memcpy(be.n_heads, h_n_heads_, sizeof(uint32_t) * n);
    }
}

void Context::ensure_results(uint32_t n, bool from2d) {
    if (h_results_cap_ < n) {
        if (h_results_) cudaFreeHost(h_results_);
        h_results_ = nullptr;
        DH_CUDA(cudaHostAlloc((void**)&h_results_, sizeof(dh_result) * n, cudaHostAllocDefault));
        h_results_cap_ = n;
    }
    if (from2d && h_from2d_cap_ < n) {
        if (h_from2d_) cudaFreeHost(h_from2d_);
        h_from2d_ = nullptr;
        h_from2d_cap_ = 0;
        DH_CUDA(cudaHostAlloc((void**)&h_from2d_, sizeof(dh_result) * n, cudaHostAllocDefault));
        h_from2d_cap_ = n;
    }
}

// pinned staging of the per-frame arguments of a batch (BackEnd::args; run_front packs it chunk by chunk)
void Context::ensure_frame_args(uint32_t n) {
    if (h_frame_cap_ >= n) return;
    if (h_frame_fs_) cudaFreeHost(h_frame_fs_);
    if (h_frame_k_) cudaFreeHost(h_frame_k_);
    h_frame_fs_ = nullptr;
    h_frame_k_ = nullptr;
    h_frame_cap_ = 0;
    DH_CUDA(cudaHostAlloc((void**)&h_frame_fs_, sizeof(FrameState) * n, cudaHostAllocDefault));
    DH_CUDA(cudaHostAlloc((void**)&h_frame_k_, sizeof(float) * 18 * (size_t)n, cudaHostAllocDefault));
    h_frame_cap_ = n;
}

// ------------------------------------------------------------------------------------------------ compressed host input
// dh_predict_batch from HOST frames is bound by the PCIe copy of the raw pixels (614 KB per VGA
// frame, ~53 GB/s).  Depth frames are mostly background (0 = invalid), so worker threads rewrite
// every chunk as Biwi run-length files (biwi.rs:81-103: the format biwi_decode_kernel expands)
// straight into pinned memory; only those bytes cross PCIe and the frames are rebuilt on the GPU,
// bit for bit.  Chunks whose sampled density says the rewrite would not pay are copied raw.
// A context with only a few worker threads copies raw (unless DH_HOST_ENCODE=1 insists): that is a rank of
// a multi-GPU box, where the contexts together are bound by the host's memory system, not by one PCIe link,
// and a rewritten frame costs that system 870 KB of traffic against 614 KB for a raw copy (8 ranks with 3
// workers each on a 32-core box: 264 k frames/s rewriting, 303 k copying raw; one rank with 15 workers:
// 135 k against 86 k).
bool Context::want_encode(uint32_t n, uint32_t w, uint32_t h) const {
    if (host_encode_ == 0) return false;
    if (host_encode_ < 0 && (encode_threads_req_ ? encode_threads_req_ : default_encode_threads()) < 6u) return false;
    const size_t px = (size_t)w * h;
    return px >= 16384 && px <= 0x3fffffffull && (size_t)n * px >= (size_t)8 * 640 * 480;
}

void Context::ensure_encode(uint32_t n, uint32_t F) {
    if (!pool_) pool_.reset(new WorkerPool(encode_threads_req_ ? encode_threads_req_ : default_encode_threads()));
    const size_t bound = rle_frame_bound(sk_.w, sk_.h);
    const uint32_t groups = (F + kEncGroup - 1) / kEncGroup;
    const size_t slot = (size_t)(groups + 1) * kEncGroup * bound;  // tasks of up to kEncGroup frames at a fixed stride: room for a ragged last task
    if (slot > enc_slot_bytes_ || F > enc_frames_ || bound != enc_frame_bound_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream_));
        for (int i = 0; i < kEncSlots; ++i) {
            if (h_enc_[i]) cudaFreeHost(h_enc_[i]);
            if (h_enc_meta_[i]) cudaFreeHost(h_enc_meta_[i]);
            h_enc_[i] = nullptr;
            h_enc_meta_[i] = nullptr;
        }
        for (int i = 0; i < 2; ++i) dev_free(d_enc_meta_[i]);
        enc_slot_bytes_ = std::max(slot, enc_slot_bytes_);
        enc_frames_ = std::max(F, enc_frames_);
        enc_frame_bound_ = bound;
        for (int i = 0; i < kEncSlots; ++i) {
            DH_CUDA(cudaHostAlloc((void**)&h_enc_[i], enc_slot_bytes_, cudaHostAllocDefault));
            DH_CUDA(cudaHostAlloc((void**)&h_enc_meta_[i], sizeof(unsigned long long) * 2 * enc_frames_, cudaHostAllocDefault));
        }
        for (int i = 0; i < 2; ++i) dev_alloc(d_enc_meta_[i], (size_t)2 * enc_frames_);
    }
    if (enc_slot_bytes_ + 64 > blob_cap_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream_));
        for (int i = 0; i < 2; ++i) dev_free(d_blob_[i]);
        blob_cap_ = enc_slot_bytes_ + 64;
    }
    for (int i = 0; i < 2; ++i)
        if (!d_blob_[i]) dev_alloc(d_blob_[i], blob_cap_);
    if ((size_t)n + 1 > biwi_frames_cap_) {
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(d_offsets_);
        dev_free(d_status_);
        if (h_status_) cudaFreeHost(h_status_);
        h_status_ = nullptr;
        biwi_frames_cap_ = (size_t)n + 1;
        dev_alloc(d_offsets_, biwi_frames_cap_);
        dev_alloc(d_status_, biwi_frames_cap_);
        DH_CUDA(cudaHostAlloc((void**)&h_status_, sizeof(uint32_t) * biwi_frames_cap_, cudaHostAllocDefault));
    }
}

void Context::run_batch_encoded(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, const float K[9],
                                const BackEnd& be) {
    // Two streams of chunks meet inside the batch.  FRONT: the workers rewrite chunks 0, 1, 2, .. as
    // run-length files (two chunks in flight, pinned slots 0..2); a finished chunk's bytes go over
    // the first copy stream into device slots 0 / 1 and are expanded and predicted on lane 0.
    // BACK (hybrid, DH_HOST_HYBRID=0 turns it off): chunks n-1, n-2, .. go over RAW on a second copy
    // stream into device slots 2 / 3 and are predicted on lane 1, one after the other as fast as
    // PCIe takes them.  Whoever reaches a chunk first takes it; the call ends where they meet.
    // The host cores and the copy engines therefore work all the time, on different chunks, and
    // the split adapts to how dense the frames are and how many cores the caller gave the workers.
    const bool hybrid = env_flag("DH_HOST_HYBRID", true) && !timing_ && max_lanes_ >= 2;
    uint32_t want_chunk = pick_chunk(n, DH_DEPTH_HOST);
    if (be.image_scratch()) want_chunk = std::min(want_chunk, image_chunk_cap(w, h));
    const int n_lanes = hybrid ? 2 : 1;
    ensure_scratch(hf, w, h, want_chunk, K, n_lanes, be.heads != nullptr);
    if (be.image_scratch()) ensure_image_scratch(n_lanes);
    if (be.heads) ensure_heads_scratch(n_lanes);
    if (be.kind == BackEnd::kPose && be.image && !be.image_on_device) ensure_mask_plane(n_lanes);
    if (be.kind == BackEnd::kBlurred || be.hough.blur) ensure_blur_taps(hf);
    const uint32_t iterations = hf.meanshift_iterations.load();
    const uint32_t F = call_chunk_;
    const uint32_t n_chunks = (n + F - 1) / F;
    const size_t frame_px = (size_t)w * h;
    ensure_results(n, be.hough.from2d != nullptr);
    if (be.heads) ensure_heads_results(n, be.heads->max_heads);
    if (be.args) ensure_frame_args(n);
    ensure_staging(hybrid ? 4 : 2);
    ensure_encode(n, F);
    const size_t bound = enc_frame_bound_;
    const uint32_t M = enc_frames_;  // stride between the begin and end halves of a meta array
    // frames per worker task (and per copy): about two tasks per worker and chunk
    const uint32_t G = std::max<uint32_t>(1u, std::min<uint32_t>(kEncGroup, F / std::max<uint32_t>(1u, 2u * pool_->size())));
    DH_CUDA(cudaMemsetAsync(d_status_, 0, sizeof(uint32_t) * n, stream_));
    DH_CUDA(cudaEventRecord(ev_fork_, stream_));
    for (int i = 1; i < n_lanes; ++i) DH_CUDA(cudaStreamWaitEvent(lanes_[i].stream, ev_fork_, 0));
    DH_CUDA(cudaStreamWaitEvent(copy_stream_, ev_fork_, 0));
    DH_CUDA(cudaStreamWaitEvent(copy_stream2_, ev_fork_, 0));

    std::vector<uint64_t> tickets(n_chunks, 0);
    std::vector<uint32_t> pslot_of(n_chunks, 0);
    std::vector<uint32_t> encq;               // chunks at the workers, oldest first
    uint32_t front = 0, back = n_chunks;      // chunks [front, back) belong to nobody yet
    uint32_t n_submitted = 0, n_front_sent = 0, n_back_sent = 0, done_chunks = 0;
    cudaEvent_t pslot_busy[kEncSlots] = {nullptr, nullptr, nullptr};  // H2D of the slot's previous chunk
    cudaEvent_t last_front_copy = nullptr;                            // after the last copy handed to the front stream
    auto dense = [&](uint32_t c) {
        if (host_encode_ >= 0) return false;
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        // sampled share of 16-pixel groups that would have to travel: above ~60 % the rewrite
        // costs more host time than the copy saves
        const double d = 0.5 * (rle_sample_density(depth + (size_t)f0 * frame_px, frame_px, 61) +
                                rle_sample_density(depth + (size_t)(f0 + nc - 1) * frame_px, frame_px, 61));
        return d >= 0.6;
    };
    auto submit = [&](uint32_t c) {
        const int pslot = (int)(n_submitted % (uint32_t)kEncSlots);
        ++n_submitted;
        pslot_of[c] = (uint32_t)pslot;
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        if (pslot_busy[pslot]) DH_CUDA(cudaEventSynchronize(pslot_busy[pslot]));  // the slot's previous chunk has left the host
        uint8_t* base = h_enc_[pslot];
        unsigned long long* meta = h_enc_meta_[pslot];
        const uint16_t* src = depth + (size_t)f0 * frame_px;
        tickets[c] = pool_->run((nc + G - 1) / G, [=](uint32_t gi) {
            size_t pos = (size_t)gi * G * bound;
            for (uint32_t k = gi * G; k < std::min(nc, (gi + 1) * G); ++k) {
                meta[k] = pos;
                pos += rle_encode_frame(src + (size_t)k * frame_px, w, h, base + pos);
                meta[M + k] = pos;
            }
        });
        encq.push_back(c);
    };
    // the pipeline of one chunk whose frames are (about to be) in device slot `slot`
    auto run_chunk = [&](Lane& L, int slot, uint32_t c) {
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        FrameBuffers b = buffers(L, d_depth_[slot]);
        flush_pending(L);
        run_front(L, b, nc, nullptr, nullptr, 0.0f, be.args, f0);
        run_chunk_back(L, b, f0, nc, iterations, be);
        DH_CUDA(cudaEventRecord(ev_consumed_[slot], L.stream));
        ++done_chunks;
    };
    auto send_encoded = [&](uint32_t c) {
        const int slot = (int)(n_front_sent & 1u), pslot = (int)pslot_of[c];
        Lane& L = lanes_[0];
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        DH_CUDA(cudaStreamWaitEvent(copy_stream_, n_front_sent >= 2 ? ev_consumed_[slot] : ev_fork_, 0));
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        if (timing_) {
            t0 = next_event();
            t1 = next_event();
            DH_CUDA(cudaEventRecord(t0, copy_stream_));
        }
        const unsigned long long* meta = h_enc_meta_[pslot];
        for (uint32_t k0 = 0; k0 < nc; k0 += G) {  // one copy per task: the tasks' bytes are not adjacent
            const uint32_t k1 = std::min(nc, k0 + G) - 1u;
            const size_t b0 = (size_t)meta[k0], b1 = (size_t)meta[M + k1];
            DH_CUDA(cudaMemcpyAsync(d_blob_[slot] + b0, h_enc_[pslot] + b0, b1 - b0, cudaMemcpyHostToDevice, copy_stream_));
            last_h2d_bytes_ += b1 - b0;
        }
        DH_CUDA(cudaMemcpyAsync(d_enc_meta_[slot], meta, sizeof(unsigned long long) * 2 * M, cudaMemcpyHostToDevice, copy_stream_));
        last_h2d_bytes_ += sizeof(unsigned long long) * 2 * M;
        DH_CUDA(cudaEventRecord(ev_enc_copied_[pslot], copy_stream_));
        pslot_busy[pslot] = ev_enc_copied_[pslot];
        ++last_encoded_chunks_;
        if (timing_) {
            DH_CUDA(cudaEventRecord(t1, copy_stream_));
            copy_marks_.push_back({t0, t1});
        }
        DH_CUDA(cudaEventRecord(ev_copied_[slot], copy_stream_));
        last_front_copy = ev_copied_[slot];
        DH_CUDA(cudaStreamWaitEvent(L.stream, ev_copied_[slot], 0));
        mark(DH_STAGE_H2D);  // the expansion counts as input transfer
        DH_CUDA(cudaMemsetAsync(d_depth_[slot], 0, (size_t)nc * frame_px * sizeof(uint16_t), L.stream));
        launch_biwi_decode(d_blob_[slot], d_enc_meta_[slot], d_enc_meta_[slot] + M, 0ull, nc, w, h, d_depth_[slot], d_status_ + f0, L.stream);
        launches_ += 1;
        run_chunk(L, slot, c);
        ++n_front_sent;
    };
    // raw chunk: front stream (a dense chunk met on the way: slots 0 / 1, lane 0) or back stream (slots 2 / 3, lane 1)
    auto send_raw = [&](uint32_t c, bool back_stream) {
        const uint32_t k = back_stream ? n_back_sent : n_front_sent;
        const int slot = (back_stream ? 2 : 0) + (int)(k & 1u);
        cudaStream_t cs = back_stream ? copy_stream2_ : copy_stream_;
        Lane& L = lanes_[back_stream ? 1 : 0];
        const uint32_t f0 = c * F, nc = std::min<uint32_t>(F, n - f0);
        DH_CUDA(cudaStreamWaitEvent(cs, k >= 2 ? ev_consumed_[slot] : ev_fork_, 0));
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        if (timing_) {
            t0 = next_event();
            t1 = next_event();
            DH_CUDA(cudaEventRecord(t0, cs));
        }
        DH_CUDA(cudaMemcpyAsync(d_depth_[slot], depth + (size_t)f0 * frame_px, (size_t)nc * frame_px * sizeof(uint16_t), cudaMemcpyHostToDevice, cs));
        last_h2d_bytes_ += (uint64_t)nc * frame_px * sizeof(uint16_t);
        if (timing_) {
            DH_CUDA(cudaEventRecord(t1, cs));
            copy_marks_.push_back({t0, t1});
        }
        DH_CUDA(cudaEventRecord(ev_copied_[slot], cs));
        if (!back_stream) last_front_copy = ev_copied_[slot];
        DH_CUDA(cudaStreamWaitEvent(L.stream, ev_copied_[slot], 0));
        run_chunk(L, slot, c);
        if (back_stream) ++n_back_sent; else ++n_front_sent;
    };
    // The back stream takes another chunk only while NO copy is in flight on either copy stream.
    // Raw and rewritten bytes compete for the same host memory bandwidth (a rewritten frame costs the
    // host ~870 KB of DRAM traffic, a raw one 614 KB, and this host sustains ~95 GB/s): measured on
    // the 16-core box, a raw stream that is always busy slows the workers by more than it adds
    // (107 k frames/s at 44 % raw against 124 k with no raw chunk at all), while raw chunks that
    // only fill the copy engines' idle time add to the total (134-137 k at ~25 % raw).
    auto back_ready = [&] {
        if (last_front_copy && cudaEventQuery(last_front_copy) == cudaErrorNotReady) return false;
        if (n_back_sent && cudaEventQuery(ev_copied_[2 + (int)((n_back_sent - 1u) & 1u)]) == cudaErrorNotReady) return false;
        return true;
    };
    auto refill = [&] {
        while (encq.size() < 2 && front < back) {
            const uint32_t c = front++;
            if (dense(c)) send_raw(c, false);
            else submit(c);
        }
    };
    auto drain = [&] {
        for (uint32_t c : encq) pool_->wait(tickets[c]);
    };
    try {
        refill();
        while (done_chunks < n_chunks) {
            bool progressed = false;
            if (!encq.empty() && pool_->done(tickets[encq.front()])) {
                const uint32_t c = encq.front();
                encq.erase(encq.begin());
                send_encoded(c);
                refill();
                progressed = true;
            }
            if (hybrid && back > front && back_ready()) {
                send_raw(--back, true);
                progressed = true;
            }
            if (progressed) continue;
            if (!encq.empty()) {
                pool_->wait_for(tickets[encq.front()], hybrid && back > front ? 30u : 1000000u);
            } else if (front < back) {
                refill();  // nothing at the workers (dense chunks only so far)
            } else {
                break;  // everything has been handed out
            }
        }
    } catch (...) {
        drain();  // no worker may still read the caller's frames once this call has returned
        cudaStreamSynchronize(copy_stream_);
        cudaStreamSynchronize(copy_stream2_);
        for (int i = 0; i < n_lanes; ++i) cudaStreamSynchronize(lanes_[i].stream);
        throw;
    }
    for (int i = 0; i < n_lanes; ++i) flush_pending(lanes_[i]);
    if (n_lanes > 1) {
        for (int i = 1; i < n_lanes; ++i) {
            DH_CUDA(cudaEventRecord(lanes_[i].done, lanes_[i].stream));
            DH_CUDA(cudaStreamWaitEvent(stream_, lanes_[i].done, 0));
        }
    }
    mark(-1);
    DH_CUDA(cudaStreamSynchronize(stream_));
    end_call();
    if (last_encoded_chunks_) {
        // the library wrote these files itself: a decode failure is a bug, never the caller's input
        DH_CUDA(cudaMemcpy(h_status_, d_status_, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost));
        for (uint32_t i = 0; i < n; ++i)
            if (h_status_[i]) throw ModelError(DH_E_STATE, "internal error: frame " + std::to_string(i) + " did not survive the compressed host->device path");
    }
    if (be.results) std::memcpy(be.results, h_results_, sizeof(dh_result) * n);
    if (be.hough.from2d) std::memcpy(be.hough.from2d, h_from2d_, sizeof(dh_result) * n);
    if (be.heads) {
        std::memcpy(be.heads_out, h_heads_, sizeof(dh_head) * n * be.heads->max_heads);
        std::memcpy(be.n_heads, h_n_heads_, sizeof(uint32_t) * n);
    }
}

// ------------------------------------------------------------------------------------------------ tracks and seeded sequences
// The reference's real use (examples/live_prediction.rs:75-88) predicts a SEQUENCE: every frame is
// seeded with the pose of the frame before it, which makes a sequence sequential — but separate
// sequences stay independent.  A track is one such sequence from one camera: its own K, optional
// seeds for its first frame, frames t > 0 seeded from frame t - 1 of the same track (centre iff its
// z > min_seed_z, rotation always).  A pass holds up to F frames (the chunk size), one per slot;
// each slot holds the next frame of one track.  The seeds of a pass are written on the device from
// the results of the previous one, and nothing returns to the host between passes but finished
// windows of results.
namespace {
// Where every frame runs: tracks longest first (ties by index), one per slot; when a track ends its
// slot takes the next waiting track in the next pass, so passes stay full while tracks wait, and with
// n_seq <= F there are as many passes as the longest track has frames.  The entries of a pass are
// its occupied slots in slot order; the plan decides only where a frame runs, never what it computes.
struct TrackPlan {
    std::vector<TrackSlot> slots;    // the entries of every pass, pass after pass
    std::vector<uint32_t> pass_off;  // pass p: slots[pass_off[p], pass_off[p + 1])
};
TrackPlan plan_tracks(uint32_t n_seq, const uint64_t* seq_off, uint32_t F) {
    TrackPlan pl;
    std::vector<uint32_t> order;
    for (uint32_t s = 0; s < n_seq; ++s)
        if (seq_off[s + 1] > seq_off[s]) order.push_back(s);
    std::stable_sort(order.begin(), order.end(),
                     [&](uint32_t a, uint32_t b) { return seq_off[a + 1] - seq_off[a] > seq_off[b + 1] - seq_off[b]; });
    struct Slot {
        int32_t track = -1;
        uint64_t t = 0;    // the track's next frame
        int32_t pos = -1;  // the slot's position in the last pass
    };
    std::vector<Slot> sl(std::min<size_t>(F, order.size()));
    size_t next = 0;
    for (Slot& s : sl) s.track = (int32_t)order[next++];
    pl.slots.reserve((size_t)seq_off[n_seq]);
    pl.pass_off.push_back(0);
    for (;;) {
        int32_t pos = 0;
        for (Slot& s : sl) {
            if (s.track < 0) continue;
            pl.slots.push_back(TrackSlot{(int32_t)(seq_off[s.track] + s.t), s.track, s.t ? s.pos : -1});
            s.pos = pos++;
        }
        if (pos == 0) break;
        pl.pass_off.push_back((uint32_t)pl.slots.size());
        for (Slot& s : sl) {
            if (s.track < 0 || ++s.t < seq_off[s.track + 1] - seq_off[s.track]) continue;
            s.t = 0;
            s.track = next < order.size() ? (int32_t)order[next++] : -1;
        }
    }
    return pl;
}

constexpr size_t kTrackWindowResults = 1u << 16;  // results per window of passes (3.7 MB)
// host-bound masks of dh_predict_tracks_mask: a window holds at most this many bytes of masks, or one pass
constexpr size_t kTrackWindowMaskBytes = 64ull << 20;

template <typename T>
void host_alloc(T*& p, size_t n) {
    p = nullptr;
    DH_CUDA(cudaHostAlloc((void**)&p, sizeof(T) * std::max<size_t>(n, 1), cudaHostAllocDefault));
}
template <typename T>
void host_free(T*& p) {
    if (p) cudaFreeHost(p);
    p = nullptr;
}
}  // namespace

void Context::free_track_buffers() {
    for (int i = 0; i < 2; ++i) {
        dev_free(tb_.d_plan[i]);
        host_free(tb_.h_plan[i]);
        host_free(tb_.h_win[i]);
        host_free(tb_.h_blob[i]);
        dev_free(tb_.d_mwin[i]);
        host_free(tb_.h_mwin[i]);
    }
    dev_free(tb_.d_win);
    dev_free(tb_.d_tracks);
    host_free(tb_.h_tracks);
    dev_free(tb_.d_status);
    dev_free(tb_.d_bad);
    host_free(tb_.h_bad);
    tb_.win_cap = tb_.tracks_cap = tb_.blob_cap = tb_.status_cap = tb_.mwin_cap = 0;
}

void Context::predict_tracks(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n_seq,
                             const uint64_t* seq_off, uint32_t w, uint32_t h, int depth_loc, const dh_frame_args* seq_args, float min_seed_z,
                             dh_result* out, uint8_t* mask, int mask_loc) {
    begin_call();
    have_debug_ = false;
    last_encoded_chunks_ = 0;
    last_h2d_bytes_ = 0;
    const uint64_t total = n_seq ? seq_off[n_seq] : 0;
    if (total > 0x7fffffffull) throw ModelError(DH_E_ARG, "more than 2^31 - 1 frames in one call");
    if (total == 0) {
        end_call();
        return;
    }
    if (blob) check_biwi_offsets(offsets, (uint32_t)total);
    ensure_forest(hf);
    // One K, equal lengths, no starting seeds and frames in memory: the operations dh_predict_sequences
    // has always issued (one strided copy per pass, seq_guess_kernel, the one-K kernels).
    bool uniform = !blob;
    uint32_t live = 0;
    for (uint32_t s = 0; s < n_seq; ++s) {
        live += seq_off[s + 1] > seq_off[s] ? 1u : 0u;
        uniform = uniform && seq_off[s + 1] - seq_off[s] == seq_off[1] && seq_args[s].has_guess == 0 &&
                  std::memcmp(seq_args[s].K, seq_args[0].K, sizeof(seq_args[0].K)) == 0;
    }
    const uint32_t want = chunk_frames_ ? std::min(chunk_frames_, live) : std::min<uint32_t>(live, 512u);
    ensure_scratch(hf, w, h, want, seq_args[0].K, 1);
    ensure_staging(2);
    const uint32_t iterations = hf.meanshift_iterations.load();
    const uint32_t F = call_chunk_;
    const TrackPlan pl = plan_tracks(n_seq, seq_off, F);
    const uint32_t n_pass = (uint32_t)pl.pass_off.size() - 1;
    const size_t px = (size_t)w * h;
    // Host-bound masks travel in the windows of the results: a window's passes write their masks to
    // d_mwin in pass order, one copy brings them to h_mwin, and the host scatters them where it scatters
    // the window's results.  Their windows hold at most kTrackWindowMaskBytes of masks, or one pass.
    const bool mask_host = mask && mask_loc != DH_DEPTH_DEVICE;
    const uint32_t W = (uint32_t)std::max<size_t>(
        1, std::min(kTrackWindowResults / F, mask_host ? kTrackWindowMaskBytes / ((size_t)F * px) : kTrackWindowResults));  // passes per window
    const size_t win = (size_t)W * F;

    // buffers (each grows alone; a free waits for the work that may still use it)
    auto drain = [&] {
        DH_CUDA(cudaStreamSynchronize(stream_));
        DH_CUDA(cudaStreamSynchronize(copy_stream_));
    };
    if (win > tb_.win_cap) {
        drain();
        for (int i = 0; i < 2; ++i) {
            dev_free(tb_.d_plan[i]);
            host_free(tb_.h_plan[i]);
            host_free(tb_.h_win[i]);
        }
        dev_free(tb_.d_win);
        for (int i = 0; i < 2; ++i) {
            dev_alloc(tb_.d_plan[i], win);
            host_alloc(tb_.h_plan[i], win);
            host_alloc(tb_.h_win[i], win);
        }
        dev_alloc(tb_.d_win, win);
        tb_.win_cap = win;
    }
    if (!tb_.d_bad) {
        dev_alloc(tb_.d_bad, 1);
        host_alloc(tb_.h_bad, 1);
    }
    if (mask_host && win * px > tb_.mwin_cap) {
        drain();
        for (int i = 0; i < 2; ++i) {
            dev_free(tb_.d_mwin[i]);
            host_free(tb_.h_mwin[i]);
        }
        for (int i = 0; i < 2; ++i) {
            dev_alloc(tb_.d_mwin[i], win * px);
            host_alloc(tb_.h_mwin[i], win * px);
        }
        tb_.mwin_cap = win * px;
    }
    if (!uniform) {
        if (n_seq > tb_.tracks_cap) {
            drain();
            dev_free(tb_.d_tracks);
            host_free(tb_.h_tracks);
            dev_alloc(tb_.d_tracks, n_seq);
            host_alloc(tb_.h_tracks, n_seq);
            tb_.tracks_cap = n_seq;
        }
        // the per-track table, once per call: K, K^-1 (as ensure_scratch computes them for one matrix), first seeds
        for (uint32_t s = 0; s < n_seq; ++s) {
            const dh_frame_args& a = seq_args[s];
            TrackArgs& t = tb_.h_tracks[s];
            std::memset(&t, 0, sizeof(t));
            std::memcpy(t.K, a.K, sizeof(float) * 9);
            mat3_inverse_f32(a.K, t.K + 9);
            t.has_guess = a.has_guess;
            if (a.has_guess & 1u)
                for (int k = 0; k < 3; ++k) t.midp_guess[k] = a.midp_guess[k];
            if (a.has_guess & 2u)
                for (int k = 0; k < 3; ++k) t.rot_guess[k] = a.rot_guess[k];
        }
        DH_CUDA(cudaMemcpyAsync(tb_.d_tracks, tb_.h_tracks, sizeof(TrackArgs) * n_seq, cudaMemcpyHostToDevice, stream_));
    }
    auto file_bytes = [&](int32_t f) { return (size_t)((offsets[f + 1] - offsets[f] + 3) & ~3ull); };
    if (blob) {
        // a pass's (start, end) pairs, then its files at multiples of 4 bytes, then the decode's read-ahead
        size_t need = 0;
        for (uint32_t p = 0; p < n_pass; ++p) {
            size_t b = 16ull * (pl.pass_off[p + 1] - pl.pass_off[p]) + 64;
            for (uint32_t j = pl.pass_off[p]; j < pl.pass_off[p + 1]; ++j) b += file_bytes(pl.slots[j].frame);
            need = std::max(need, b);
        }
        if (need > blob_cap_) {
            drain();
            for (int i = 0; i < 2; ++i) dev_free(d_blob_[i]);
            blob_cap_ = need;
        }
        for (int i = 0; i < 2; ++i)
            if (!d_blob_[i]) dev_alloc(d_blob_[i], blob_cap_);
        if (need > tb_.blob_cap) {
            drain();
            for (int i = 0; i < 2; ++i) host_free(tb_.h_blob[i]);
            for (int i = 0; i < 2; ++i) host_alloc(tb_.h_blob[i], need);
            tb_.blob_cap = need;
        }
        if (F > tb_.status_cap) {
            drain();
            dev_free(tb_.d_status);
            dev_alloc(tb_.d_status, F);
            tb_.status_cap = F;
        }
        DH_CUDA(cudaMemsetAsync(tb_.d_bad, 0xFF, sizeof(unsigned long long), stream_));
    }

    // window wi's results, from pinned memory to `out` in input order
    auto scatter = [&](uint32_t wi) {
        const dh_result* r = tb_.h_win[wi & 1u];
        for (uint32_t p = wi * W; p < std::min(n_pass, (wi + 1) * W); ++p)
            for (uint32_t j = pl.pass_off[p]; j < pl.pass_off[p + 1]; ++j)
                out[pl.slots[j].frame] = r[(size_t)(p - wi * W) * F + (j - pl.pass_off[p])];
    };
    // ... and its masks (host-bound), once tb_.ev_mwin_copied of its parity has passed
    auto scatter_masks = [&](uint32_t wi) {
        const uint8_t* m = tb_.h_mwin[wi & 1u];
        for (uint32_t p = wi * W; p < std::min(n_pass, (wi + 1) * W); ++p)
            for (uint32_t j = pl.pass_off[p]; j < pl.pass_off[p + 1]; ++j)
                std::memcpy(mask + (size_t)pl.slots[j].frame * px, m + ((size_t)(p - wi * W) * F + (j - pl.pass_off[p])) * px, px);
    };
    const cudaMemcpyKind kind = depth_loc == DH_DEPTH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    Lane& L = lanes_[0];
    try {
        DH_CUDA(cudaEventRecord(ev_fork_, stream_));
        DH_CUDA(cudaStreamWaitEvent(copy_stream_, ev_fork_, 0));
        for (uint32_t p = 0; p < n_pass; ++p) {
            const uint32_t wi = p / W, pw = p % W, n = pl.pass_off[p + 1] - pl.pass_off[p];
            const TrackSlot* e = pl.slots.data() + pl.pass_off[p];
            const TrackSlot* d_e = tb_.d_plan[wi & 1u] + (pl.pass_off[p] - pl.pass_off[wi * W]);
            const int slot = (int)(p & 1u);
            if (pw == 0 && wi >= 2) {  // the pinned buffers of this window's parity are free once window wi - 2 is out
                DH_CUDA(cudaEventSynchronize(tb_.ev_win[wi & 1u]));
                scatter(wi - 2);
                if (mask_host) {  // (and d_mwin of this parity: the lane writes it again only after this point)
                    DH_CUDA(cudaEventSynchronize(tb_.ev_mwin_copied[wi & 1u]));
                    scatter_masks(wi - 2);
                }
            }
            if (p >= 2) DH_CUDA(cudaStreamWaitEvent(copy_stream_, ev_consumed_[slot], 0));
            if (pw == 0 && !uniform) {  // the window's slot tables (pass p - 2 consumed: window wi - 2 is done with them)
                const uint32_t e1 = pl.pass_off[std::min(n_pass, p + W)];
                std::memcpy(tb_.h_plan[wi & 1u], e, sizeof(TrackSlot) * (e1 - pl.pass_off[p]));
                DH_CUDA(cudaMemcpyAsync(tb_.d_plan[wi & 1u], tb_.h_plan[wi & 1u], sizeof(TrackSlot) * (e1 - pl.pass_off[p]),
                                        cudaMemcpyHostToDevice, copy_stream_));
            }
            if (uniform) {
                // the same frame of consecutive tracks: rows of one strided copy (row = a frame, pitch = a track)
                const size_t fps = (size_t)seq_off[1];
                DH_CUDA(cudaMemcpy2DAsync(d_depth_[slot], px * sizeof(uint16_t), depth + (size_t)e[0].frame * px,
                                          fps * px * sizeof(uint16_t), px * sizeof(uint16_t), n, kind, copy_stream_));
                if (depth_loc != DH_DEPTH_DEVICE) last_h2d_bytes_ += (uint64_t)n * px * sizeof(uint16_t);
            } else if (blob) {
                DH_CUDA(cudaEventSynchronize(ev_copied_[slot]));  // pass p - 2 has left this pinned slot
                unsigned long long* pairs = reinterpret_cast<unsigned long long*>(tb_.h_blob[slot]);
                uint8_t* files = tb_.h_blob[slot] + 16ull * n;
                size_t o = 0;
                for (uint32_t j = 0; j < n; ++j) {
                    const int32_t f = e[j].frame;
                    const size_t len = (size_t)(offsets[f + 1] - offsets[f]);
                    pairs[j] = o;
                    pairs[n + j] = o + len;
                    std::memcpy(files + o, blob + offsets[f], len);
                    o += file_bytes(f);
                }
                DH_CUDA(cudaMemcpyAsync(d_blob_[slot], tb_.h_blob[slot], 16ull * n + o, cudaMemcpyHostToDevice, copy_stream_));
                last_h2d_bytes_ += 16ull * n + o;
            } else if (depth_loc == DH_DEPTH_DEVICE) {
                launch_track_gather(depth, d_depth_[slot], d_e, n, px, copy_stream_);
                launches_ += 1;
            } else {
                for (uint32_t j = 0; j < n; ++j)
                    DH_CUDA(cudaMemcpyAsync(d_depth_[slot] + (size_t)j * px, depth + (size_t)e[j].frame * px, px * sizeof(uint16_t),
                                            cudaMemcpyHostToDevice, copy_stream_));
                last_h2d_bytes_ += (uint64_t)n * px * sizeof(uint16_t);
            }
            DH_CUDA(cudaEventRecord(ev_copied_[slot], copy_stream_));
            DH_CUDA(cudaStreamWaitEvent(L.stream, ev_copied_[slot], 0));
            FrameBuffers b = buffers(L, d_depth_[slot]);
            if (blob) {
                mark(DH_STAGE_H2D);  // the expansion counts as input transfer
                DH_CUDA(cudaMemsetAsync(d_depth_[slot], 0, (size_t)n * px * sizeof(uint16_t), L.stream));
                const unsigned long long* d_pairs = reinterpret_cast<const unsigned long long*>(d_blob_[slot]);
                launch_biwi_decode(d_blob_[slot] + 16ull * n, d_pairs, d_pairs + n, 0ull, n, w, h, d_depth_[slot], tb_.d_status, L.stream);
                launches_ += 1;
            }
            // the pass's masks, from the leaf words of its traversal: to their frames of `mask` (the slot table, or on the
            // uniform path, which uploads none, the stride of its strided copy), or to the window's plane in pass order
            auto pass_masks = [&] {
                if (!mask) return;
                mark(DH_STAGE_VOTE);  // booked as the 2-D calls book their back end
                if (mask_host)
                    launch_track_mask(b, geom_, fdev_, n, nullptr, 0u, 1u, tb_.d_mwin[wi & 1u] + (size_t)pw * F * px, L.stream);
                else if (uniform)
                    launch_track_mask(b, geom_, fdev_, n, nullptr, (uint32_t)e[0].frame, (uint32_t)seq_off[1], mask, L.stream);
                else
                    launch_track_mask(b, geom_, fdev_, n, d_e, 0u, 0u, mask, L.stream);
                launches_ += 1;
                stage_check("mask");
            };
            if (uniform) {
                run_front(L, b, n, nullptr, e[0].prev >= 0 ? L.results : nullptr, min_seed_z);
                pass_masks();
                run_back(L, b, n, iterations);
            } else {
                launch_track_guess(L.fs, L.frame_k, d_e, tb_.d_tracks, L.results, n, min_seed_z, blob ? tb_.d_status : nullptr,
                                   tb_.d_bad, L.stream);
                launches_ += 1;
                run_front(L, b, n, nullptr, nullptr, 0.0f, nullptr, 0, true);
                pass_masks();
                run_back(L, b, n, iterations, L.frame_k);
            }
            DH_CUDA(cudaMemcpyAsync(tb_.d_win + (size_t)pw * F, L.results, sizeof(dh_result) * n, cudaMemcpyDeviceToDevice, L.stream));
            DH_CUDA(cudaEventRecord(ev_consumed_[slot], L.stream));
            if (pw + 1 == W || p + 1 == n_pass) {
                DH_CUDA(cudaMemcpyAsync(tb_.h_win[wi & 1u], tb_.d_win, sizeof(dh_result) * (size_t)(pw + 1) * F, cudaMemcpyDeviceToHost,
                                        L.stream));
                DH_CUDA(cudaEventRecord(tb_.ev_win[wi & 1u], L.stream));
                if (mask_host) {  // the window's masks leave on the second copy stream while the lane goes on
                    DH_CUDA(cudaEventRecord(tb_.ev_mwin_ready[wi & 1u], L.stream));
                    DH_CUDA(cudaStreamWaitEvent(copy_stream2_, tb_.ev_mwin_ready[wi & 1u], 0));
                    DH_CUDA(cudaMemcpyAsync(tb_.h_mwin[wi & 1u], tb_.d_mwin[wi & 1u], (size_t)(pw + 1) * F * px, cudaMemcpyDeviceToHost,
                                            copy_stream2_));
                    DH_CUDA(cudaEventRecord(tb_.ev_mwin_copied[wi & 1u], copy_stream2_));
                }
            }
        }
        if (blob) DH_CUDA(cudaMemcpyAsync(tb_.h_bad, tb_.d_bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream_));
    } catch (...) {
        cudaStreamSynchronize(copy_stream_);
        cudaStreamSynchronize(copy_stream2_);
        cudaStreamSynchronize(stream_);
        throw;
    }
    mark(-1);
    end_call();
    const uint32_t last = (n_pass - 1) / W;
    if (mask_host) DH_CUDA(cudaStreamSynchronize(copy_stream2_));
    for (uint32_t wi = last >= 1 ? last - 1 : 0; wi <= last; ++wi) {
        scatter(wi);
        if (mask_host) scatter_masks(wi);
    }
    if (blob && *tb_.h_bad != ~0ull) throw_biwi_status((size_t)(*tb_.h_bad >> 2), (uint32_t)(*tb_.h_bad & 3u));
}

// n_seq tracks of frames_per_seq frames with one K and no starting seeds (sequence-major input):
// the pass loop of predict_tracks takes the operations this call has always issued.
void Context::predict_sequences(const HostForest& hf, const uint16_t* depth, uint32_t n_seq, uint32_t frames_per_seq, uint32_t w, uint32_t h,
                                const float K[9], int depth_loc, float min_seed_z, dh_result* out) {
    const uint64_t total = (uint64_t)n_seq * frames_per_seq;
    if (total == 0 || total > 0x7fffffffull) {  // (no per-track tables for a call that does nothing)
        if (total) throw ModelError(DH_E_ARG, "dh_predict_sequences: more than 2^31 frames");
        begin_call();
        have_debug_ = false;
        last_encoded_chunks_ = 0;
        last_h2d_bytes_ = 0;
        end_call();
        return;
    }
    std::vector<uint64_t> seq_off((size_t)n_seq + 1);
    for (uint32_t s = 0; s <= n_seq; ++s) seq_off[s] = (uint64_t)s * frames_per_seq;
    std::vector<dh_frame_args> args(n_seq);
    for (dh_frame_args& a : args) {
        std::memset(&a, 0, sizeof(a));
        std::memcpy(a.K, K, sizeof(a.K));
    }
    predict_tracks(hf, depth, nullptr, nullptr, n_seq, seq_off.data(), w, h, depth_loc, args.data(), min_seed_z, out);
}

// ------------------------------------------------------------------------------------------------ 2-D back ends
// predict_mask, build_hough_image (raw or blurred) and predict_parameter_from2dhough share the
// batch pipeline of the pose path: the same chunks, lanes, staging and front end; only the back
// end of a chunk differs (run_image_back).  The single-frame entry points are batches of one frame.
void Context::predict_mask(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, uint8_t* mask) {
    predict_mask_batch(hf, depth, 1, w, h, DH_DEPTH_HOST, mask, DH_DEPTH_HOST);
}

void Context::hough_image_raw(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                              uint16_t* votes) {
    hough_image(hf, depth, w, h, K, votes, false, nullptr);
}

// build_hough_image (prediction.rs:760-845): vote image (+ gaussian blur with the model's sigma) to
// `votes` (host, may be NULL); from2d != NULL: predict_parameter_from2dhough (prediction.rs:343-367).
void Context::hough_image(const HostForest& hf, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9], uint16_t* votes,
                          bool blur, dh_result* from2d) {
    hough_image_batch(hf, depth, 1, w, h, K, DH_DEPTH_HOST, blur, votes, DH_DEPTH_HOST, from2d);
}

void Context::predict_mask_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                                 uint8_t* mask, int mask_loc) {
    const float K[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};  // predict_mask does not project anything
    BackEnd be;
    be.kind = BackEnd::kMask;
    be.image = mask;
    be.image_on_device = mask_loc == DH_DEPTH_DEVICE;
    run_batch(hf, depth, nullptr, nullptr, n, w, h, K, depth_loc, be);
}

void Context::predict_mask_batch_biwi(const HostForest& hf, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                                      uint32_t h, uint8_t* mask, int mask_loc) {
    const float K[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    BackEnd be;
    be.kind = BackEnd::kMask;
    be.image = mask;
    be.image_on_device = mask_loc == DH_DEPTH_DEVICE;
    run_batch(hf, nullptr, blob, offsets, n, w, h, K, DH_DEPTH_HOST, be);
}

namespace {
BackEnd hough_back_end(bool blur, uint16_t* votes, int votes_loc, dh_result* from2d) {
    if (from2d && !blur) throw ModelError(DH_E_ARG, "predict_parameter_from2dhough takes the arg-max of the BLURRED vote image");
    if (!votes && !from2d) throw ModelError(DH_E_ARG, "neither a vote image nor from2d results are asked for");
    BackEnd be;
    be.kind = blur ? BackEnd::kBlurred : BackEnd::kVotes;
    be.results = from2d;
    be.image = votes;
    be.image_on_device = votes_loc == DH_DEPTH_DEVICE;
    return be;
}
}  // namespace

void Context::hough_image_batch(const HostForest& hf, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, const float K[9],
                                int depth_loc, bool blur, uint16_t* votes, int votes_loc, dh_result* from2d) {
    run_batch(hf, depth, nullptr, nullptr, n, w, h, K, depth_loc, hough_back_end(blur, votes, votes_loc, from2d));
}

// dh_build_hough_image_frames / _biwi: every frame's K reaches the kernels that project through the
// per-frame path of dh_predict_frames (arguments without seeds; run_front packs K and K^-1 per chunk
// into Lane::frame_k).  Geometry holds frame 0's K, which the kFrameK kernels do not read.
void Context::hough_image_frames(const HostForest& hf, const uint16_t* depth, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                                 uint32_t w, uint32_t h, int depth_loc, const float* K, bool blur, uint16_t* votes, int votes_loc,
                                 dh_result* from2d) {
    BackEnd be = hough_back_end(blur, votes, votes_loc, from2d);
    std::vector<dh_frame_args> args(n);
    for (uint32_t i = 0; i < n; ++i) std::memcpy(args[i].K, K + (size_t)9 * i, sizeof(float) * 9);
    be.args = args.data();
    static const float kIdentity[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    run_batch(hf, depth, blob, offsets, n, w, h, n ? K : kIdentity, blob ? DH_DEPTH_HOST : depth_loc, be);
}

// u32 sums + two u16 planes per frame of a chunk, the arg-max keys and their poses, on every lane of the call
void Context::ensure_image_scratch(int n_lanes) {
    const size_t frame_px = (size_t)sk_.w * sk_.h, need = (size_t)call_chunk_ * frame_px;
    for (int i = 0; i < std::max(1, std::min(n_lanes, kMaxLanes)); ++i) {
        Lane& L = lanes_[i];
        if (L.img_px >= need) continue;
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(L.img32);
        dev_free(L.img16);
        dev_free(L.img_keys);
        dev_free(L.img_results);
        L.img_px = 0;
        dev_alloc(L.img32, need);
        dev_alloc(L.img16, 2 * need);
        dev_alloc(L.img_keys, (size_t)call_chunk_);
        dev_alloc(L.img_results, (size_t)call_chunk_);
        L.img_px = need;
    }
}

// taps of the blur (imageproc gaussian_kernel_f32), once per model and sigma
void Context::ensure_blur_taps(const HostForest& hf) {
    const uint64_t sv = hf.sigma_version.load();
    if (d_blur_taps_ && blur_serial_ == hf.serial && blur_sigma_version_ == sv) return;
    const std::vector<float> k = build_gaussian_blur_kernel(hf.gaussian_sigma);
    DH_CUDA(cudaStreamSynchronize(stream_));
    dev_free(d_blur_taps_);
    dev_alloc(d_blur_taps_, k.size());
    DH_CUDA(cudaMemcpy(d_blur_taps_, k.data(), k.size() * sizeof(float), cudaMemcpyHostToDevice));
    blur_radius_ = (int)(k.size() / 2);
    blur_serial_ = hf.serial;
    blur_sigma_version_ = sv;
}

void Context::flush_pending(Lane& L) {
    if (!L.pending_bytes) return;
    DH_CUDA(cudaMemcpyAsync(L.pending_dst, L.pending_src, L.pending_bytes, cudaMemcpyDeviceToHost, L.stream));
    L.pending_bytes = 0;
}

void Context::run_chunk_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, uint32_t iterations, const BackEnd& be) {
    if (be.kind != BackEnd::kPose) {
        run_image_back(L, b, f0, n, be);
        return;
    }
    if (be.image) run_pose_mask(L, b, f0, n, be);
    if (be.hough.wanted()) run_pose_hough(L, b, f0, n, be.hough);
    if (be.heads) {
        FrameBuffers bs = b;
        bs.support = 1;  // head 0's support
        run_back(L, bs, n, iterations, L.frame_k);
        run_heads(L, bs, f0, n, iterations, be);
    } else {
        run_back(L, b, n, iterations, be.args ? L.frame_k : nullptr);
    }
    DH_CUDA(cudaMemcpyAsync(h_results_ + f0, L.results, sizeof(dh_result) * n, cudaMemcpyDeviceToHost, L.stream));
    if (be.hough.from2d) DH_CUDA(cudaMemcpyAsync(h_from2d_ + f0, L.img_results, sizeof(dh_result) * n, cudaMemcpyDeviceToHost, L.stream));
}

// Extra heads of a pose chunk after its back end: round 0 writes head 0 (the chunk's results, the support of
// their centre windows) and starts every frame's search, rounds 1 .. 2 (max_heads - 1) serve one try of every
// frame still searching (launch_heads_round).  The launches do not wait for the GPU: frames that stopped
// leave each kernel at once.
void Context::run_heads(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, uint32_t iterations, const BackEnd& be) {
    const dh_heads_params& p = *be.heads;
    cudaStream_t st = L.stream;
    mark(DH_STAGE_MEANSHIFT);
    HeadsBuffers hb{};
    hb.st = L.heads_st;
    hb.grid = L.heads_grid;
    hb.fs = L.heads_fs;
    hb.res = L.heads_res;
    hb.gated = L.heads_gated;
    hb.cubes = L.heads_cubes;
    hb.out = L.heads_out;
    hb.n_heads = L.heads_n;
    hb.max_heads = p.max_heads;
    hb.min_cell_votes = p.min_cell_votes;
    hb.radius = p.radius_mm;
    DH_CUDA(cudaMemsetAsync(L.heads_out, 0, sizeof(dh_head) * (size_t)n * p.max_heads, st));
    DH_CUDA(cudaMemsetAsync(L.heads_fs, 0, sizeof(FrameState) * n, st));
    const uint32_t rounds = 2u * (p.max_heads - 1u);
    for (uint32_t r = 0; r <= rounds; ++r) {
        launches_ += (uint64_t)launch_heads_round(b, hb, geom_, fdev_, n, r, iterations, n_sms_, L.frame_k, st);
        stage_check("extra heads");
    }
    mark(DH_STAGE_D2H);
    DH_CUDA(cudaMemcpyAsync(h_heads_ + (size_t)f0 * p.max_heads, L.heads_out, sizeof(dh_head) * (size_t)n * p.max_heads,
                            cudaMemcpyDeviceToHost, st));
    DH_CUDA(cudaMemcpyAsync(h_n_heads_ + f0, L.heads_n, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
    DH_CUDA(cudaGetLastError());
}

void Context::ensure_heads_scratch(int n_lanes) {
    const uint32_t F = sk_.frames;
    const size_t P = std::max<uint32_t>(geom_.P, 1u);
    for (int i = 0; i < std::max(1, std::min(n_lanes, kMaxLanes)); ++i) {
        Lane& L = lanes_[i];
        if (L.heads_frames >= F) continue;
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(L.heads_st);
        dev_free(L.heads_grid);
        dev_free(L.heads_fs);
        dev_free(L.heads_res);
        dev_free(L.heads_gated);
        dev_free(L.heads_cubes);
        dev_free(L.heads_out);
        dev_free(L.heads_n);
        L.heads_frames = 0;
        dev_alloc(L.heads_st, F);
        dev_alloc(L.heads_grid, (size_t)F * kPosGridCells);
        dev_alloc(L.heads_fs, F);
        dev_alloc(L.heads_res, F);
        dev_alloc(L.heads_gated, (size_t)F * P);
        dev_alloc(L.heads_cubes, (size_t)F * 2 * vote_box_cells());
        DH_CUDA(cudaMemset(L.heads_cubes, 0, sizeof(uint32_t) * (size_t)F * 2 * vote_box_cells()));
        dev_alloc(L.heads_out, (size_t)F * kMaxHeads);
        dev_alloc(L.heads_n, F);
        L.heads_frames = F;
    }
}

void Context::ensure_heads_results(uint32_t n, uint32_t max_heads) {
    const size_t need = (size_t)n * max_heads;
    if (h_heads_cap_ < need) {
        if (h_heads_) cudaFreeHost(h_heads_);
        h_heads_ = nullptr;
        h_heads_cap_ = 0;
        DH_CUDA(cudaHostAlloc((void**)&h_heads_, sizeof(dh_head) * need, cudaHostAllocDefault));
        h_heads_cap_ = need;
    }
    if (h_n_heads_cap_ < n) {
        if (h_n_heads_) cudaFreeHost(h_n_heads_);
        h_n_heads_ = nullptr;
        h_n_heads_cap_ = 0;
        DH_CUDA(cudaHostAlloc((void**)&h_n_heads_, sizeof(uint32_t) * n, cudaHostAllocDefault));
        h_n_heads_cap_ = n;
    }
}

// The Hough image of a pose chunk, between its traversal and its patch gate as run_pose_mask: run_hough
// as the 2-D calls run it (it reads the leaf words, the depth and the frames' K, none of which the pose
// back end writes), without their counters launch (run_back counts every frame once).  Its from2d poses
// go to the lane's img_results, since L.results is the pose back end's.  Device-bound images are written
// in place; a host-bound image leaves through the lane's one deferred copy: the poses of both kinds go
// to pinned memory with copies issued in stream order, so the image is the only deferred copy of the chunk.
void Context::run_pose_hough(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd::Hough& hb) {
    mark(DH_STAGE_VOTE);  // booked as the 2-D calls book their back end
    uint16_t* image = run_hough(L, b, f0, n, hb.blur, hb.image, hb.image_on_device, hb.from2d ? L.img_results : nullptr, L.frame_k);
    stage_check("2-D back end");
    if (image && !hb.image_on_device) {
        const size_t frame_px = (size_t)geom_.w * geom_.h;
        L.pending_dst = hb.image + (size_t)f0 * frame_px;
        L.pending_src = image;
        L.pending_bytes = frame_px * n * sizeof(uint16_t);
    }
}

// The Hough image of a chunk (frames f0 .. f0 + n - 1 of the batch) from the leaf words of its traversal:
// the votes, then the raw image or its blur; with poses != nullptr the blurred image's arg-max and its pose
// (predict_parameter_from2dhough) to poses [n] on the device.  The image goes to image + f0 frames when it
// is on the device, else to the lane's second u16 plane.  Returns where the chunk's image is (nullptr:
// image is nullptr, blurred from2d only).
uint16_t* Context::run_hough(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, bool blur, uint16_t* image, bool image_on_device,
                             dh_result* poses, const float* frame_k) {
    const Geometry& g = geom_;
    cudaStream_t st = L.stream;
    const size_t frame_px = (size_t)g.w * g.h, px = frame_px * n;
    uint16_t* out = image ? (image_on_device ? image + (size_t)f0 * frame_px : L.img16 + L.img_px) : nullptr;
    DH_CUDA(cudaMemsetAsync(L.img32, 0, px * sizeof(uint32_t), st));
    if (g.P) {
        launch_hough_votes(b, g, fdev_, n, L.img32, st, frame_k);
        launches_ += 1;
    }
    if (!blur) {
        launch_narrow_u16(L.img32, out, px, st);
        launches_ += 1;
        return out;
    }
    if (poses) DH_CUDA(cudaMemsetAsync(L.img_keys, 0, sizeof(unsigned long long) * n, st));
    launches_ += (uint64_t)launch_gaussian_blur(L.img32, L.img16, out, poses ? L.img_keys : nullptr, g.w, g.h, n, d_blur_taps_,
                                                blur_radius_, st);
    if (poses) {
        launch_hough2d_pose(L.img_keys, b.depth, g, n, poses, st, frame_k);
        launches_ += 1;
    }
    return out;
}

// The masks of a pose chunk, between its traversal and its patch gate (nothing after the traversal
// writes the leaf words, and the lane's next chunk rewrites them only after this launch in stream
// order).  mask_kernel as in run_image_back: it reads ids through b.leaf_mask whether or not the words
// carry probability codes, and decides background on the tree-0 slice.  Device-bound masks are
// written in place; host-bound ones go to the lane's plane and out through the deferred copy.
void Context::run_pose_mask(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd& be) {
    const Geometry& g = geom_;
    const size_t frame_px = (size_t)g.w * g.h, px = frame_px * n;
    mark(DH_STAGE_VOTE);  // booked as the 2-D calls book their back end
    uint8_t* mask = be.image_on_device ? static_cast<uint8_t*>(be.image) + (size_t)f0 * frame_px : L.mask_plane;
    DH_CUDA(cudaMemsetAsync(mask, 0, px, L.stream));
    if (g.P) {
        launch_mask(b, g, fdev_, n, mask, L.stream);
        launches_ += 1;
    }
    stage_check("mask");
    if (!be.image_on_device) {
        L.pending_dst = static_cast<uint8_t*>(be.image) + (size_t)f0 * frame_px;
        L.pending_src = mask;
        L.pending_bytes = px;
    }
}

// one u8 plane per frame of a chunk, on every lane of the call (host-bound masks of the pose back end)
void Context::ensure_mask_plane(int n_lanes) {
    const size_t need = (size_t)call_chunk_ * sk_.w * sk_.h;
    for (int i = 0; i < std::max(1, std::min(n_lanes, kMaxLanes)); ++i) {
        Lane& L = lanes_[i];
        if (L.mask_px >= need) continue;
        DH_CUDA(cudaStreamSynchronize(stream_));
        dev_free(L.mask_plane);
        L.mask_px = 0;
        dev_alloc(L.mask_plane, need);
        L.mask_px = need;
    }
}

// The 2-D back end of one chunk; the launches do not depend on the number of frames.  Images the
// caller wants in device memory are written there by the kernels; host-bound images are left in
// the lane's scratch and copied out before the lane's next chunk (flush_pending).
void Context::run_image_back(Lane& L, const FrameBuffers& b, uint32_t f0, uint32_t n, const BackEnd& be) {
    const Geometry& g = geom_;
    cudaStream_t st = L.stream;
    const size_t frame_px = (size_t)g.w * g.h, px = frame_px * n;
    const float* frame_k = be.args ? L.frame_k : nullptr;  // masks project nothing
    mark(DH_STAGE_VOTE);  // the whole 2-D back end is booked here
    void* image = nullptr;  // this chunk's image in device memory
    size_t elem = sizeof(uint16_t);
    if (be.kind == BackEnd::kMask) {
        elem = 1;
        uint8_t* mask = be.image_on_device ? static_cast<uint8_t*>(be.image) + (size_t)f0 * frame_px : reinterpret_cast<uint8_t*>(L.img16 + L.img_px);
        DH_CUDA(cudaMemsetAsync(mask, 0, px, st));
        if (g.P) {
            launch_mask(b, g, fdev_, n, mask, st);
            launches_ += 1;
        }
        image = mask;
    } else {
        image = run_hough(L, b, f0, n, be.kind == BackEnd::kBlurred, static_cast<uint16_t*>(be.image), be.image_on_device,
                          be.results ? L.results : nullptr, frame_k);
    }
    stage_check("2-D back end");
    mark(DH_STAGE_D2H);
    launch_counters(b, g, n, d_counters_, st);
    launches_ += 1;
    if (be.results) DH_CUDA(cudaMemcpyAsync(h_results_ + f0, L.results, sizeof(dh_result) * n, cudaMemcpyDeviceToHost, st));
    if (image && !be.image_on_device) {
        L.pending_dst = static_cast<char*>(be.image) + (size_t)f0 * frame_px * elem;
        L.pending_src = image;
        L.pending_bytes = px * elem;
    }
    DH_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------ debug exports
void Context::require_debug() const {
    if (!have_debug_) throw ModelError(DH_E_STATE, "no debug state: call dh_ctx_enable_debug(ctx, 1) and then dh_predict");
}
void Context::debug_dims(uint32_t* npx, uint32_t* npy, uint32_t* n_trees) const {
    require_debug();
    if (npx) *npx = geom_.npx;
    if (npy) *npy = geom_.npy;
    if (n_trees) *n_trees = geom_.n_trees;
}
void Context::debug_leaf(int32_t* leaf) {
    require_debug();
    const size_t P = geom_.P, T = geom_.n_trees;
    std::vector<int32_t> tmp(P * T);
    DH_CUDA(cudaMemcpy(tmp.data(), lanes_[0].leaf, P * T * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (size_t t = 0; t < T; ++t)  // device layout [T][P] -> exported [P][T]
        for (size_t p = 0; p < P; ++p) {
            const int32_t w = tmp[t * P + p];  // leaf word: id | probability code << 23 when codes ride along
            leaf[p * T + t] = (w >= 0 && leaf_codes_) ? (int32_t)((uint32_t)w & kLeafIdMask) : w;
        }
}
void Context::debug_patches(float* p3, uint8_t* gate) {
    require_debug();
    const size_t P = geom_.P;
    if (gate) DH_CUDA(cudaMemcpy(gate, lanes_[0].gate, P, cudaMemcpyDeviceToHost));
    if (p3) DH_CUDA(cudaMemcpy(p3, lanes_[0].p3, P * 3 * sizeof(float), cudaMemcpyDeviceToHost));
}
void Context::debug_seeds(uint32_t* guess_pos, uint32_t* guess_rot, int32_t* seed_mid, int32_t* seed_rot) {
    require_debug();
    if (guess_pos) DH_CUDA(cudaMemcpy(guess_pos, lanes_[0].grids, kPosGridCells * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (guess_rot) DH_CUDA(cudaMemcpy(guess_rot, lanes_[0].grids + kPosGridCells, kRotGridCells * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    FrameState fs;
    DH_CUDA(cudaMemcpy(&fs, lanes_[0].fs, sizeof(fs), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 3; ++k) {
        if (seed_mid) seed_mid[k] = fs.seed_mid[k];
        if (seed_rot) seed_rot[k] = fs.seed_rot[k];
    }
}
void Context::debug_votes(int which, int32_t* keys, uint32_t* vals, uint64_t* n, int32_t* box_origin, int32_t* box_dim) {
    require_debug();
    if (which < 0 || which > 1) throw ModelError(DH_E_ARG, "which must be 0 (centre) or 1 (rotation)");
    unsigned long long* d_count = nullptr;
    dev_alloc(d_count, 1);
    DH_CUDA(cudaMemset(d_count, 0, sizeof(unsigned long long)));
    int32_t* d_keys = nullptr;
    uint32_t* d_vals = nullptr;
    FrameState fs;
    DH_CUDA(cudaMemcpy(&fs, lanes_[0].fs, sizeof(fs), cudaMemcpyDeviceToHost));
    const size_t cells = vote_box_cells();
    if (keys) {
        dev_alloc(d_keys, cells * 3);
        dev_alloc(d_vals, cells);
    }
    FrameBuffers b = buffers(lanes_[0], d_depth_[0]);
    launch_box_dump(b, 0, which, d_keys, d_vals, d_count, stream_);
    DH_CUDA(cudaStreamSynchronize(stream_));
    unsigned long long cnt = 0;
    DH_CUDA(cudaMemcpy(&cnt, d_count, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (keys && cnt) {
        DH_CUDA(cudaMemcpy(keys, d_keys, cnt * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost));
        DH_CUDA(cudaMemcpy(vals, d_vals, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    }
    dev_free(d_keys);
    dev_free(d_vals);
    dev_free(d_count);
    if (n) *n = cnt;
    if (box_origin)
        for (int k = 0; k < 3; ++k) box_origin[k] = fs.box_org[which][k];
    if (box_dim) *box_dim = fs.box_valid[which] ? (int32_t)vote_box_dim() : 0;
}
void Context::debug_meanshift(int which, int32_t* pos, uint32_t* n_iter) {
    require_debug();
    if (which < 0 || which > 1) throw ModelError(DH_E_ARG, "which must be 0 (centre) or 1 (rotation)");
    FrameState fs;
    DH_CUDA(cudaMemcpy(&fs, lanes_[0].fs, sizeof(fs), cudaMemcpyDeviceToHost));
    const uint32_t ran = std::min<uint32_t>(fs.ms_iters[which], sk_.trace_iters);
    const uint32_t room = n_iter ? *n_iter : 0;
    const uint32_t cnt = std::min(ran, room);
    if (pos && cnt && lanes_[0].ms_trace)
        DH_CUDA(cudaMemcpy(pos, lanes_[0].ms_trace + (size_t)which * sk_.trace_iters * 3, (size_t)cnt * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (n_iter) *n_iter = ran;
    last_ms_flags_[which] = fs.ms_flags[which];
}
void Context::debug_leaf_static(const HostForest& hf, uint32_t* valtoadd, uint8_t* rot_ok, uint8_t* off_ok) {
    DH_CUDA(cudaSetDevice(device_));
    ensure_forest(hf);
    std::vector<LeafInfo> li(df_n_leaves_);
    DH_CUDA(cudaMemcpy(li.data(), df_leaf_info_, li.size() * sizeof(LeafInfo), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < li.size(); ++i) {
        if (valtoadd) valtoadd[i] = li[i].valtoadd;
        if (rot_ok) rot_ok[i] = (li[i].flags & kLeafRotOk) ? 1 : 0;
        if (off_ok) off_ok[i] = (li[i].flags & kLeafOffOk) ? 1 : 0;
    }
}

}  // namespace dh
