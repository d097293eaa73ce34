// dh_capi.cu — the extern "C" boundary declared in include/depthhead_cuda.h.
// Every entry point catches everything (nothing unwinds across the ABI) and records a
// thread-local message for dh_last_error().
#include <cstring>
#include <memory>
#include <new>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/depthhead_cuda.h"
#include "dh_ctx.hpp"
#include "dh_forest.hpp"
#include "dh_json.hpp"

struct dh_forest {
    std::unique_ptr<dh::HostForest> hf;
};
struct dh_ctx {
    std::unique_ptr<dh::Context> cx;
};

namespace {

thread_local std::string g_last_error = "";

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

template <typename F>
int guarded(F&& body) {
    try {
        body();
        return DH_OK;
    } catch (const dh::JsonError& e) {
        return fail(DH_E_JSON, std::string("json: ") + e.what());
    } catch (const dh::ModelError& e) {
        return fail(e.code, e.what());
    } catch (const std::bad_alloc&) {
        return fail(DH_E_ARG, "out of host memory");
    } catch (const std::exception& e) {
        return fail(DH_E_ARG, e.what());
    } catch (...) {
        return fail(DH_E_ARG, "unknown error");
    }
}

#define REQUIRE(cond, msg) \
    do {                   \
        if (!(cond)) throw dh::ModelError(DH_E_ARG, msg); \
    } while (0)

static_assert(sizeof(dh_frame_args) == 80 && offsetof(dh_frame_args, K) == 0 && offsetof(dh_frame_args, midp_guess) == 36 &&
                  offsetof(dh_frame_args, rot_guess) == 48 && offsetof(dh_frame_args, has_guess) == 72 &&
                  offsetof(dh_frame_args, _pad) == 76,
              "dh_frame_args layout (mirrored by capi.FRAME_ARGS_DTYPE and the Rust shim)");

static_assert(sizeof(dh_heads_params) == 16 && offsetof(dh_heads_params, max_heads) == 0 &&
                  offsetof(dh_heads_params, min_cell_votes) == 4 && offsetof(dh_heads_params, radius_mm) == 8 &&
                  offsetof(dh_heads_params, _pad) == 12,
              "dh_heads_params layout (mirrored by capi.HEADS_PARAMS_DTYPE)");
static_assert(sizeof(dh_head) == 72 && offsetof(dh_head, pose) == 0 && offsetof(dh_head, support) == 56 &&
                  offsetof(dh_head, n_patches) == 64 && offsetof(dh_head, seed_cell) == 68,
              "dh_head layout (mirrored by capi.HEAD_DTYPE)");
static_assert(dh::kMaxHeads == 8, "dh_heads_params.max_heads allows 1..8");

void check_frame_args(const char* fn, const dh_frame_args* args, uint32_t n, const char* what = "frame") {
    for (uint32_t i = 0; i < n; ++i)
        if (args[i].has_guess & ~3u)
            throw dh::ModelError(DH_E_ARG, std::string(fn) + ": " + what + " " + std::to_string(i) + " has has_guess " +
                                               std::to_string(args[i].has_guess) + " (only bits 0 and 1 are defined)");
}

// seq_off of dh_predict_tracks: n_seq + 1 offsets from 0, monotone, at most 2^31 - 1 frames
void check_seq_off(const char* fn, const uint64_t* seq_off, uint32_t n_seq) {
    if (seq_off[0] != 0) throw dh::ModelError(DH_E_ARG, std::string(fn) + ": seq_off[0] is not 0");
    for (uint32_t s = 0; s < n_seq; ++s)
        if (seq_off[s + 1] < seq_off[s])
            throw dh::ModelError(DH_E_ARG, std::string(fn) + ": seq_off is not monotone at track " + std::to_string(s));
    if (seq_off[n_seq] > 0x7fffffffull) throw dh::ModelError(DH_E_ARG, std::string(fn) + ": more than 2^31 - 1 frames");
}

// check_biwi_offsets with the entry point named in the message
void check_offsets(const char* fn, const uint64_t* offsets, uint32_t n) {
    try {
        dh::check_biwi_offsets(offsets, n);
    } catch (const dh::ModelError& e) {
        throw dh::ModelError(e.code, std::string(fn) + ": " + e.what());
    }
}

}  // namespace

extern "C" {

const char* dh_last_error(void) { return g_last_error.c_str(); }
int dh_abi_version(void) { return DH_ABI_VERSION; }
#ifndef DH_BUILD_ID
#define DH_BUILD_ID "unknown"
#endif
const char* dh_build_id(void) { return DH_BUILD_ID; }

int dh_forest_from_json(const char* json, size_t len, dh_forest** out) {
    return guarded([&] {
        REQUIRE(json && out, "dh_forest_from_json: NULL argument");
        *out = nullptr;
        dh::RawForest raw = dh::parse_hough_prediction_json(json, len);
        std::unique_ptr<dh_forest> f(new dh_forest());
        f->hf.reset(dh::flatten_forest(raw));
        *out = f.release();
    });
}

int dh_forest_from_arrays(const dh_forest_arrays* a, dh_forest** out) {
    return guarded([&] {
        REQUIRE(a && out, "dh_forest_from_arrays: NULL argument");
        *out = nullptr;
        REQUIRE(a->n_trees >= 1 && a->tree_node_off && a->tree_leaf_off && a->prob && a->vote_off,
                "dh_forest_from_arrays: missing arrays");
        dh::RawForest raw;
        raw.stepwidth = a->stepwidth;
        raw.subimage_width = a->subimage_width;
        raw.subimage_height = a->subimage_height;
        raw.meanshift_iterations = a->meanshift_iterations;
        raw.gaussian_sigma = a->gaussian_sigma;
        raw.n_trees = a->n_trees;
        const int T = a->n_trees;
        raw.tree_node_off.assign(a->tree_node_off, a->tree_node_off + T + 1);
        raw.tree_leaf_off.assign(a->tree_leaf_off, a->tree_leaf_off + T + 1);
        const int64_t NN = raw.tree_node_off[T], NL = raw.tree_leaf_off[T];
        REQUIRE(NN >= 0 && NL >= 1, "dh_forest_from_arrays: bad offsets");
        if (NN) {
            REQUIRE(a->rects && a->threshold && a->child, "dh_forest_from_arrays: missing node arrays");
            raw.rects.assign(a->rects, a->rects + NN * 8);
            raw.threshold.assign(a->threshold, a->threshold + NN);
            raw.child.assign(a->child, a->child + NN * 2);
        }
        raw.prob.assign(a->prob, a->prob + NL);
        raw.vote_off.assign(a->vote_off, a->vote_off + NL + 1);
        const int64_t NV = raw.vote_off[NL];
        REQUIRE(NV >= 0, "dh_forest_from_arrays: bad vote offsets");
        if (NV) {
            REQUIRE(a->offsets && a->rotations, "dh_forest_from_arrays: missing vote arrays");
            raw.offsets.assign(a->offsets, a->offsets + NV * 3);
            raw.rotations.assign(a->rotations, a->rotations + NV * 3);
        }
        std::unique_ptr<dh_forest> f(new dh_forest());
        f->hf.reset(dh::flatten_forest(raw));
        *out = f.release();
    });
}

void dh_forest_free(dh_forest* f) { delete f; }

uint32_t dh_forest_get_stepwidth(const dh_forest* f) { return f ? f->hf->stepwidth.load() : 0; }
int dh_forest_set_stepwidth(dh_forest* f, uint32_t v) {
    return guarded([&] {
        REQUIRE(f, "NULL forest");
        if (v == 0) throw dh::ModelError(DH_E_SHAPE, "stepwidth 0: the reference's sliding window never advances (prediction.rs:684)");
        f->hf->stepwidth.store(v);
    });
}
uint32_t dh_forest_get_meanshift_iterations(const dh_forest* f) { return f ? f->hf->meanshift_iterations.load() : 0; }
int dh_forest_set_meanshift_iterations(dh_forest* f, uint32_t v) {
    return guarded([&] {
        REQUIRE(f, "NULL forest");
        REQUIRE(v <= 65535, "meanshift_iterations > 65535 is not supported");
        f->hf->meanshift_iterations.store(v);
    });
}
float dh_forest_get_sigma(const dh_forest* f) { return f ? f->hf->gaussian_sigma : 0.0f; }
int dh_forest_set_sigma(dh_forest* f, float v) {
    return guarded([&] {
        REQUIRE(f, "NULL forest");
        // update_sigma (prediction.rs:320-326): ignored if unchanged or <= 0 (NaN compares false
        // on both tests in the reference and would be stored; it is rejected here)
        REQUIRE(v == v, "sigma is NaN");
        if (v == f->hf->gaussian_sigma || v <= 0.0f) return;
        f->hf->gaussian_sigma = v;
        f->hf->sigma_version.fetch_add(1);
    });
}
uint32_t dh_forest_get_subimage_width(const dh_forest* f) { return f ? f->hf->subimage_width : 0; }
uint32_t dh_forest_get_subimage_height(const dh_forest* f) { return f ? f->hf->subimage_height : 0; }
int32_t dh_forest_n_trees(const dh_forest* f) { return f ? f->hf->n_trees : 0; }
int64_t dh_forest_n_nodes(const dh_forest* f) { return f ? (int64_t)f->hf->n_nodes() : 0; }
int64_t dh_forest_n_leaves(const dh_forest* f) { return f ? (int64_t)f->hf->n_leaves() : 0; }
int64_t dh_forest_n_votes(const dh_forest* f) { return f ? (int64_t)f->hf->n_votes() : 0; }

int dh_ctx_create(int device, dh_ctx** out) {
    return guarded([&] {
        REQUIRE(out, "dh_ctx_create: NULL out");
        *out = nullptr;
        std::unique_ptr<dh_ctx> c(new dh_ctx());
        c->cx.reset(new dh::Context(device));
        *out = c.release();
    });
}
void dh_ctx_free(dh_ctx* c) {
    try {
        delete c;
    } catch (...) {
    }
}
int dh_ctx_set_stream(dh_ctx* c, void* s) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->set_stream(s);
    });
}
int dh_ctx_set_chunk_frames(dh_ctx* c, uint32_t frames) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->set_chunk_frames(frames);
    });
}
int dh_ctx_set_encode_threads(dh_ctx* c, uint32_t n) {
    return guarded([&] {
        REQUIRE(c, "NULL context");
        REQUIRE(n <= 256, "dh_ctx_set_encode_threads: more than 256 threads");
        c->cx->set_encode_threads(n);
    });
}
int dh_ctx_transfer_info(dh_ctx* c, uint64_t info[4]) {
    return guarded([&] {
        REQUIRE(c && info, "NULL argument");
        info[0] = c->cx->last_h2d_bytes();
        info[1] = c->cx->last_encoded_chunks();
        info[2] = c->cx->encode_threads();
        info[3] = 0;
    });
}
int dh_ctx_synchronize(dh_ctx* c) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->synchronize();
    });
}

int dh_predict(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
               const float* midp_guess, const double* rot_guess, dh_result* out) {
    return guarded([&] {
        REQUIRE(c && f && depth && K && out, "dh_predict: NULL argument");
        c->cx->predict(*f->hf, depth, w, h, K, midp_guess, rot_guess, out);
    });
}
int dh_predict_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                     const float K[9], int depth_loc, dh_result* out) {
    return guarded([&] {
        REQUIRE(c && f && K && (n == 0 || (depth && out)), "dh_predict_batch: NULL argument");
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_batch: bad depth_loc");
        c->cx->predict_batch(*f->hf, depth, n, w, h, K, depth_loc, out);
    });
}
int dh_biwi_depth_dims(const uint8_t* file, size_t len, uint32_t* w, uint32_t* h) {
    return guarded([&] {
        REQUIRE(file && w && h, "dh_biwi_depth_dims: NULL argument");
        dh::biwi_depth_dims(file, len, w, h);
    });
}
int dh_biwi_decode_depth(dh_ctx* c, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h,
                         uint16_t* out, int out_loc) {
    return guarded([&] {
        REQUIRE(c && (n == 0 || (blob && offsets && out)), "dh_biwi_decode_depth: NULL argument");
        REQUIRE(out_loc == DH_DEPTH_HOST || out_loc == DH_DEPTH_DEVICE, "dh_biwi_decode_depth: bad out_loc");
        c->cx->biwi_decode(blob, offsets, n, w, h, out, out_loc);
    });
}
int dh_predict_batch_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                          uint32_t w, uint32_t h, const float K[9], dh_result* out) {
    return guarded([&] {
        REQUIRE(c && f && K && (n == 0 || (blob && offsets && out)), "dh_predict_batch_biwi: NULL argument");
        c->cx->predict_batch_biwi(*f->hf, blob, offsets, n, w, h, K, out);
    });
}
int dh_predict_frames(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                      const dh_frame_args* args, dh_result* out) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_frames: bad depth_loc");
        if (args) check_frame_args("dh_predict_frames", args, n);
        REQUIRE(c && f && (n == 0 || (depth && args && out)), "dh_predict_frames: NULL argument");
        c->cx->predict_frames(*f->hf, depth, nullptr, nullptr, n, w, h, depth_loc, args, out);
    });
}
int dh_predict_frames_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                           uint32_t h, const dh_frame_args* args, dh_result* out) {
    return guarded([&] {
        if (args) check_frame_args("dh_predict_frames_biwi", args, n);
        REQUIRE(c && f && (n == 0 || (blob && offsets && args && out)), "dh_predict_frames_biwi: NULL argument");
        c->cx->predict_frames(*f->hf, nullptr, blob, offsets, n, w, h, DH_DEPTH_HOST, args, out);
    });
}

int dh_predict_tracks(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n_seq, const uint64_t* seq_off, uint32_t w,
                      uint32_t h, int depth_loc, const dh_frame_args* seq_args, float min_seed_z, dh_result* out) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_tracks: bad depth_loc");
        if (seq_off) check_seq_off("dh_predict_tracks", seq_off, n_seq);
        if (seq_args) check_frame_args("dh_predict_tracks", seq_args, n_seq, "track");
        REQUIRE(c && f && seq_off && (n_seq == 0 || seq_args) && (seq_off[n_seq] == 0 || (depth && out)), "dh_predict_tracks: NULL argument");
        c->cx->predict_tracks(*f->hf, depth, nullptr, nullptr, n_seq, seq_off, w, h, depth_loc, seq_args, min_seed_z, out);
    });
}

int dh_predict_tracks_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n_seq,
                           const uint64_t* seq_off, uint32_t w, uint32_t h, const dh_frame_args* seq_args, float min_seed_z,
                           dh_result* out) {
    return guarded([&] {
        if (seq_off) check_seq_off("dh_predict_tracks_biwi", seq_off, n_seq);
        if (seq_args) check_frame_args("dh_predict_tracks_biwi", seq_args, n_seq, "track");
        if (seq_off && offsets) dh::check_biwi_offsets(offsets, (uint32_t)seq_off[n_seq]);
        REQUIRE(c && f && seq_off && (n_seq == 0 || seq_args) && (seq_off[n_seq] == 0 || (blob && offsets && out)),
                "dh_predict_tracks_biwi: NULL argument");
        c->cx->predict_tracks(*f->hf, nullptr, blob, offsets, n_seq, seq_off, w, h, DH_DEPTH_HOST, seq_args, min_seed_z, out);
    });
}

// Pose and head mask from one traversal: the pose call's argument rules, then the two outputs named
int dh_predict_frames_mask(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                           const dh_frame_args* args, dh_result* out, uint8_t* mask, int mask_loc) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_frames_mask: bad depth_loc");
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_frames_mask: bad mask_loc");
        if (args) check_frame_args("dh_predict_frames_mask", args, n);
        REQUIRE(n == 0 || out, "dh_predict_frames_mask: NULL out");
        REQUIRE(n == 0 || mask, "dh_predict_frames_mask: NULL mask");
        REQUIRE(c && f && (n == 0 || (depth && args)), "dh_predict_frames_mask: NULL argument");
        c->cx->predict_frames(*f->hf, depth, nullptr, nullptr, n, w, h, depth_loc, args, out, mask, mask_loc);
    });
}
int dh_predict_frames_mask_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                                uint32_t h, const dh_frame_args* args, dh_result* out, uint8_t* mask, int mask_loc) {
    return guarded([&] {
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_frames_mask_biwi: bad mask_loc");
        if (args) check_frame_args("dh_predict_frames_mask_biwi", args, n);
        if (offsets) check_offsets("dh_predict_frames_mask_biwi", offsets, n);
        REQUIRE(n == 0 || out, "dh_predict_frames_mask_biwi: NULL out");
        REQUIRE(n == 0 || mask, "dh_predict_frames_mask_biwi: NULL mask");
        REQUIRE(c && f && (n == 0 || (blob && offsets && args)), "dh_predict_frames_mask_biwi: NULL argument");
        c->cx->predict_frames(*f->hf, nullptr, blob, offsets, n, w, h, DH_DEPTH_HOST, args, out, mask, mask_loc);
    });
}
int dh_predict_tracks_mask(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n_seq, const uint64_t* seq_off, uint32_t w,
                           uint32_t h, int depth_loc, const dh_frame_args* seq_args, float min_seed_z, dh_result* out, uint8_t* mask,
                           int mask_loc) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_tracks_mask: bad depth_loc");
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_tracks_mask: bad mask_loc");
        if (seq_off) check_seq_off("dh_predict_tracks_mask", seq_off, n_seq);
        if (seq_args) check_frame_args("dh_predict_tracks_mask", seq_args, n_seq, "track");
        const bool work = seq_off && seq_off[n_seq] > 0;
        REQUIRE(!work || out, "dh_predict_tracks_mask: NULL out");
        REQUIRE(!work || mask, "dh_predict_tracks_mask: NULL mask");
        REQUIRE(c && f && seq_off && (n_seq == 0 || seq_args) && (!work || depth), "dh_predict_tracks_mask: NULL argument");
        c->cx->predict_tracks(*f->hf, depth, nullptr, nullptr, n_seq, seq_off, w, h, depth_loc, seq_args, min_seed_z, out, mask, mask_loc);
    });
}
int dh_predict_tracks_mask_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n_seq,
                                const uint64_t* seq_off, uint32_t w, uint32_t h, const dh_frame_args* seq_args, float min_seed_z,
                                dh_result* out, uint8_t* mask, int mask_loc) {
    return guarded([&] {
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_tracks_mask_biwi: bad mask_loc");
        if (seq_off) check_seq_off("dh_predict_tracks_mask_biwi", seq_off, n_seq);
        if (seq_args) check_frame_args("dh_predict_tracks_mask_biwi", seq_args, n_seq, "track");
        if (seq_off && offsets) check_offsets("dh_predict_tracks_mask_biwi", offsets, (uint32_t)seq_off[n_seq]);
        const bool work = seq_off && seq_off[n_seq] > 0;
        REQUIRE(!work || out, "dh_predict_tracks_mask_biwi: NULL out");
        REQUIRE(!work || mask, "dh_predict_tracks_mask_biwi: NULL mask");
        REQUIRE(c && f && seq_off && (n_seq == 0 || seq_args) && (!work || (blob && offsets)), "dh_predict_tracks_mask_biwi: NULL argument");
        c->cx->predict_tracks(*f->hf, nullptr, blob, offsets, n_seq, seq_off, w, h, DH_DEPTH_HOST, seq_args, min_seed_z, out, mask,
                              mask_loc);
    });
}

// Pose and Hough image from one traversal: the argument rules of the pose call and of the 2-D call
int dh_predict_frames_hough(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                            const dh_frame_args* args, dh_result* out, int blur, uint16_t* hough, int hough_loc, dh_result* from2d) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_frames_hough: bad depth_loc");
        REQUIRE(hough_loc == DH_DEPTH_HOST || hough_loc == DH_DEPTH_DEVICE, "dh_predict_frames_hough: bad hough_loc");
        REQUIRE(blur == 0 || blur == 1, "dh_predict_frames_hough: blur must be 0 or 1");
        REQUIRE(hough || from2d, "dh_predict_frames_hough: hough and from2d are both NULL");
        REQUIRE(blur || !from2d, "dh_predict_frames_hough: from2d needs blur = 1 (the arg-max of the blurred image)");
        if (args) check_frame_args("dh_predict_frames_hough", args, n);
        REQUIRE(n == 0 || out, "dh_predict_frames_hough: NULL out");
        REQUIRE(c && f && (n == 0 || (depth && args)), "dh_predict_frames_hough: NULL argument");
        c->cx->predict_frames_hough(*f->hf, depth, nullptr, nullptr, n, w, h, depth_loc, args, out, blur != 0, hough, hough_loc, from2d);
    });
}
int dh_predict_frames_hough_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                                 uint32_t h, const dh_frame_args* args, dh_result* out, int blur, uint16_t* hough, int hough_loc,
                                 dh_result* from2d) {
    return guarded([&] {
        REQUIRE(hough_loc == DH_DEPTH_HOST || hough_loc == DH_DEPTH_DEVICE, "dh_predict_frames_hough_biwi: bad hough_loc");
        REQUIRE(blur == 0 || blur == 1, "dh_predict_frames_hough_biwi: blur must be 0 or 1");
        REQUIRE(hough || from2d, "dh_predict_frames_hough_biwi: hough and from2d are both NULL");
        REQUIRE(blur || !from2d, "dh_predict_frames_hough_biwi: from2d needs blur = 1 (the arg-max of the blurred image)");
        if (args) check_frame_args("dh_predict_frames_hough_biwi", args, n);
        if (offsets) check_offsets("dh_predict_frames_hough_biwi", offsets, n);
        REQUIRE(n == 0 || out, "dh_predict_frames_hough_biwi: NULL out");
        REQUIRE(c && f && (n == 0 || (blob && offsets && args)), "dh_predict_frames_hough_biwi: NULL argument");
        c->cx->predict_frames_hough(*f->hf, nullptr, blob, offsets, n, w, h, DH_DEPTH_HOST, args, out, blur != 0, hough, hough_loc, from2d);
    });
}
int dh_predict_frames_heads(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h, int depth_loc,
                            const dh_frame_args* args, const dh_heads_params* params, dh_head* out, uint32_t* n_heads) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_frames_heads: bad depth_loc");
        REQUIRE(params, "dh_predict_frames_heads: NULL params");
        REQUIRE(params->max_heads >= 1 && params->max_heads <= dh::kMaxHeads,
                "dh_predict_frames_heads: max_heads must be 1..8, got " + std::to_string(params->max_heads));
        REQUIRE(params->radius_mm > 0.0f, "dh_predict_frames_heads: radius_mm must be > 0 (and not NaN)");
        REQUIRE(params->min_cell_votes >= 1, "dh_predict_frames_heads: min_cell_votes must be >= 1");
        if (args) check_frame_args("dh_predict_frames_heads", args, n);
        REQUIRE(n == 0 || (out && n_heads), "dh_predict_frames_heads: NULL out or n_heads");
        REQUIRE(c && f && (n == 0 || (depth && args)), "dh_predict_frames_heads: NULL argument");
        c->cx->predict_frames_heads(*f->hf, depth, n, w, h, depth_loc, args, *params, out, n_heads);
    });
}
size_t dh_biwi_encode_bound(uint32_t w, uint32_t h) { return dh::rle_frame_bound(w, h); }
int dh_biwi_encode_depth(const uint16_t* frames, uint32_t n, uint32_t w, uint32_t h, uint32_t threads, uint8_t* blob, size_t cap,
                         uint64_t* offsets, size_t* needed) {
    return guarded([&] {
        REQUIRE(needed && (n == 0 || frames), "dh_biwi_encode_depth: NULL argument");
        REQUIRE((uint64_t)w * h <= 0x3fffffffull, "dh_biwi_encode_depth: frame of more than 2^30 pixels");
        const size_t px = (size_t)w * h, bound = dh::rle_frame_bound(w, h);
        // pass 1 (parallel): every frame into its own slot of an uninitialised scratch area;
        // pass 2 (parallel): the files move to their packed places
        std::unique_ptr<uint8_t[]> scratch(new uint8_t[(size_t)std::max<uint32_t>(n, 1u) * bound]);
        std::vector<size_t> len(n), start(n + 1, 0);
        dh::WorkerPool pool(threads ? threads : dh::default_encode_threads());
        uint8_t* sc = scratch.get();
        pool.wait(pool.run(n, [&](uint32_t i) { len[i] = dh::rle_encode_frame(frames + (size_t)i * px, w, h, sc + (size_t)i * bound); }));
        for (uint32_t i = 0; i < n; ++i) start[i + 1] = start[i] + ((len[i] + 15) & ~(size_t)15);
        if (offsets)
            for (uint32_t i = 0; i < n; ++i) offsets[i] = start[i];
        if (blob)
            pool.wait(pool.run(n, [&](uint32_t i) {
                if (start[i + 1] > cap) return;
                std::memcpy(blob + start[i], sc + (size_t)i * bound, len[i]);
                std::memset(blob + start[i] + len[i], 0, start[i + 1] - start[i] - len[i]);
            }));
        const size_t pos = start[n];
        if (offsets) offsets[n] = pos;
        *needed = pos + 16;  // the decoder reads whole 4-byte words; a little slack after the last file
    });
}
int dh_biwi_parse_cal(const char* text, size_t len, float K[9]) {
    return guarded([&] {
        REQUIRE(text && K, "dh_biwi_parse_cal: NULL argument");
        dh::biwi_parse_cal(text, len, K);
    });
}
int dh_biwi_parse_pose(const uint8_t* file, size_t len, const float K[9], float pos3d[3], float pos2d[2], float rot[3]) {
    return guarded([&] {
        REQUIRE(file && K && pos3d && pos2d && rot, "dh_biwi_parse_pose: NULL argument");
        dh::biwi_parse_pose(file, len, K, pos3d, pos2d, rot);
    });
}
struct dh_trainset {
    dh::TrainSet* ts;
};
int dh_trainset_create(dh_ctx* c, const uint16_t* patches, uint64_t n, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh,
                       const uint8_t* is_object, const float* offsets, const double* rotations, dh_trainset** out) {
    return guarded([&] {
        REQUIRE(c && patches && is_object && offsets && rotations && out, "dh_trainset_create: NULL argument");
        *out = nullptr;
        dh::TrainSet* ts = c->cx->trainset_create(patches, n, sw, sh, rw, rh, is_object, offsets, rotations);
        *out = new dh_trainset{ts};
    });
}
void dh_trainset_free(dh_trainset* t) {
    if (!t) return;
    dh::trainset_free(t->ts);
    delete t;
}
int dh_train_score_level(dh_ctx* c, const dh_trainset* t, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                         const int32_t* cand_rects, const double* cand_thr, uint32_t m, uint64_t depth, double steepness,
                         dh_split_stats* out) {
    return guarded([&] {
        REQUIRE(c && t && node_off && (n_nodes == 0 || m == 0 || (sample_idx && cand_rects && cand_thr && out)),
                "dh_train_score_level: NULL argument");
        REQUIRE(steepness == steepness && steepness != 0.0, "dh_train_score_level: steepness must be a non-zero number");
        c->cx->train_score_level(*t->ts, sample_idx, node_off, n_nodes, cand_rects, cand_thr, m, depth, steepness, out);
    });
}
int dh_train_split_level(dh_ctx* c, const dh_trainset* t, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                         const int32_t* rects, const double* thr, uint8_t* bits) {
    return guarded([&] {
        REQUIRE(c && t && node_off && (n_nodes == 0 || (sample_idx && rects && thr && bits)), "dh_train_split_level: NULL argument");
        c->cx->train_split_level(*t->ts, sample_idx, node_off, n_nodes, rects, thr, bits);
    });
}
int dh_debug_tile_plan(dh_ctx* c, uint32_t plan[8]) {
    return guarded([&] {
        REQUIRE(c && plan, "dh_debug_tile_plan: NULL argument");
        const dh::TilePlan& t = c->cx->tile_plan();
        const uint32_t v[8] = {t.tpx, t.tpy, t.tiles_x, t.tiles_y, t.tw, t.th, t.smem_bytes, t.threads};
        std::memcpy(plan, v, sizeof(v));
    });
}
int dh_train_forest(dh_ctx* c, const dh_train_params* p, const uint16_t* patches, uint64_t n, const uint8_t* is_object,
                    const float* offsets, const double* rotations, dh_forest** out) {
    return guarded([&] {
        REQUIRE(c && p && patches && is_object && offsets && rotations && out, "dh_train_forest: NULL argument");
        *out = nullptr;
        std::unique_ptr<dh::HostForest> hf(c->cx->train_forest(*p, patches, n, is_object, offsets, rotations));
        *out = new dh_forest{std::move(hf)};
    });
}
int dh_train_learn(dh_ctx* c, const dh_train_params* p, uint32_t n_frames, uint32_t w, uint32_t h, const uint16_t* depth,
                   const uint8_t* mask, const float* K, const float* pos3d, const float* rot, dh_forest** out) {
    return guarded([&] {
        REQUIRE(c && p && out && (n_frames == 0 || (depth && mask && K && pos3d && rot)), "dh_train_learn: NULL argument");
        *out = nullptr;
        std::unique_ptr<dh::HostForest> hf(c->cx->train_learn(*p, n_frames, w, h, depth, mask, K, pos3d, rot));
        *out = new dh_forest{std::move(hf)};
    });
}
int dh_forest_to_json(const dh_forest* f, char* buf, size_t cap, size_t* needed) {
    return guarded([&] {
        REQUIRE(f && needed && (cap == 0 || buf), "dh_forest_to_json: NULL argument");
        const std::string js = dh::forest_to_json(*f->hf);
        *needed = js.size();
        if (cap) std::memcpy(buf, js.data(), std::min(cap, js.size()));
    });
}
int dh_predict_mask(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, uint8_t* mask) {
    return guarded([&] {
        REQUIRE(c && f && depth && mask, "dh_predict_mask: NULL argument");
        c->cx->predict_mask(*f->hf, depth, w, h, mask);
    });
}
int dh_hough_image_raw(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h,
                       const float K[9], uint16_t* votes) {
    return guarded([&] {
        REQUIRE(c && f && depth && K && votes, "dh_hough_image_raw: NULL argument");
        c->cx->hough_image_raw(*f->hf, depth, w, h, K, votes);
    });
}

int dh_predict_sequences(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n_seq, uint32_t frames_per_seq,
                         uint32_t w, uint32_t h, const float K[9], int depth_loc, float min_seed_z, dh_result* out) {
    return guarded([&] {
        REQUIRE(c && f && K && ((uint64_t)n_seq * frames_per_seq == 0 || (depth && out)), "dh_predict_sequences: NULL argument");
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_sequences: bad depth_loc");
        c->cx->predict_sequences(*f->hf, depth, n_seq, frames_per_seq, w, h, K, depth_loc, min_seed_z, out);
    });
}
int dh_build_hough_image(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                         uint16_t* hough) {
    return guarded([&] {
        REQUIRE(c && f && depth && K && hough, "dh_build_hough_image: NULL argument");
        c->cx->hough_image(*f->hf, depth, w, h, K, hough, true, nullptr);
    });
}
int dh_predict_from2dhough(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                           dh_result* out) {
    return guarded([&] {
        REQUIRE(c && f && depth && K && out, "dh_predict_from2dhough: NULL argument");
        c->cx->hough_image(*f->hf, depth, w, h, K, nullptr, true, out);
    });
}

int dh_predict_mask_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                          int depth_loc, uint8_t* mask, int mask_loc) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_predict_mask_batch: bad depth_loc");
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_mask_batch: bad mask_loc");
        REQUIRE(c && f && (n == 0 || (depth && mask)), "dh_predict_mask_batch: NULL argument");
        c->cx->predict_mask_batch(*f->hf, depth, n, w, h, depth_loc, mask, mask_loc);
    });
}
int dh_build_hough_image_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                               const float K[9], int depth_loc, int blur, uint16_t* hough, int hough_loc, dh_result* from2d) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_build_hough_image_batch: bad depth_loc");
        REQUIRE(hough_loc == DH_DEPTH_HOST || hough_loc == DH_DEPTH_DEVICE, "dh_build_hough_image_batch: bad hough_loc");
        REQUIRE(blur == 0 || blur == 1, "dh_build_hough_image_batch: blur must be 0 or 1");
        REQUIRE(hough || from2d, "dh_build_hough_image_batch: hough and from2d are both NULL");
        REQUIRE(blur || !from2d, "dh_build_hough_image_batch: from2d needs blur = 1 (the arg-max of the blurred image)");
        REQUIRE(c && f && K && (n == 0 || depth), "dh_build_hough_image_batch: NULL argument");
        c->cx->hough_image_batch(*f->hf, depth, n, w, h, K, depth_loc, blur != 0, hough, hough_loc, from2d);
    });
}
int dh_build_hough_image_frames(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                                int depth_loc, const float* K, int blur, uint16_t* hough, int hough_loc, dh_result* from2d) {
    return guarded([&] {
        REQUIRE(depth_loc == DH_DEPTH_HOST || depth_loc == DH_DEPTH_DEVICE, "dh_build_hough_image_frames: bad depth_loc");
        REQUIRE(hough_loc == DH_DEPTH_HOST || hough_loc == DH_DEPTH_DEVICE, "dh_build_hough_image_frames: bad hough_loc");
        REQUIRE(blur == 0 || blur == 1, "dh_build_hough_image_frames: blur must be 0 or 1");
        REQUIRE(hough || from2d, "dh_build_hough_image_frames: hough and from2d are both NULL");
        REQUIRE(blur || !from2d, "dh_build_hough_image_frames: from2d needs blur = 1 (the arg-max of the blurred image)");
        REQUIRE(c && f && (n == 0 || (depth && K)), "dh_build_hough_image_frames: NULL argument");
        c->cx->hough_image_frames(*f->hf, depth, nullptr, nullptr, n, w, h, depth_loc, K, blur != 0, hough, hough_loc, from2d);
    });
}
int dh_build_hough_image_frames_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                                     uint32_t w, uint32_t h, const float* K, int blur, uint16_t* hough, int hough_loc,
                                     dh_result* from2d) {
    return guarded([&] {
        REQUIRE(hough_loc == DH_DEPTH_HOST || hough_loc == DH_DEPTH_DEVICE, "dh_build_hough_image_frames_biwi: bad hough_loc");
        REQUIRE(blur == 0 || blur == 1, "dh_build_hough_image_frames_biwi: blur must be 0 or 1");
        REQUIRE(hough || from2d, "dh_build_hough_image_frames_biwi: hough and from2d are both NULL");
        REQUIRE(blur || !from2d, "dh_build_hough_image_frames_biwi: from2d needs blur = 1 (the arg-max of the blurred image)");
        if (offsets) check_offsets("dh_build_hough_image_frames_biwi", offsets, n);
        REQUIRE(c && f && (n == 0 || (blob && offsets && K)), "dh_build_hough_image_frames_biwi: NULL argument");
        c->cx->hough_image_frames(*f->hf, nullptr, blob, offsets, n, w, h, DH_DEPTH_HOST, K, blur != 0, hough, hough_loc, from2d);
    });
}
int dh_predict_mask_batch_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w,
                               uint32_t h, uint8_t* mask, int mask_loc) {
    return guarded([&] {
        REQUIRE(mask_loc == DH_DEPTH_HOST || mask_loc == DH_DEPTH_DEVICE, "dh_predict_mask_batch_biwi: bad mask_loc");
        if (offsets) check_offsets("dh_predict_mask_batch_biwi", offsets, n);
        REQUIRE(c && f && (n == 0 || (blob && offsets && mask)), "dh_predict_mask_batch_biwi: NULL argument");
        c->cx->predict_mask_batch_biwi(*f->hf, blob, offsets, n, w, h, mask, mask_loc);
    });
}

int dh_ctx_enable_stage_timing(dh_ctx* c, int on) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->enable_timing(on != 0);
    });
}
int dh_ctx_stage_ms(dh_ctx* c, float ms[DH_N_STAGES]) {
    return guarded([&] {
        REQUIRE(c && ms, "NULL argument");
        std::memcpy(ms, c->cx->stage_ms(), sizeof(float) * DH_N_STAGES);
    });
}
int dh_ctx_counters(dh_ctx* c, uint64_t counters[DH_N_COUNTERS]) {
    return guarded([&] {
        REQUIRE(c && counters, "NULL argument");
        std::memcpy(counters, c->cx->counters(), sizeof(uint64_t) * DH_N_COUNTERS);
    });
}

int dh_ctx_enable_debug(dh_ctx* c, int on) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->enable_debug(on != 0);
    });
}
int dh_debug_dims(dh_ctx* c, uint32_t* npx, uint32_t* npy, uint32_t* n_trees) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->debug_dims(npx, npy, n_trees);
    });
}
int dh_debug_leaf_indices(dh_ctx* c, int32_t* leaf) {
    return guarded([&] {
        REQUIRE(c && leaf, "NULL argument");
        c->cx->debug_leaf(leaf);
    });
}
int dh_debug_patches(dh_ctx* c, float* p3, uint8_t* gate) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->debug_patches(p3, gate);
    });
}
int dh_debug_seeds(dh_ctx* c, uint32_t* guess_pos, uint32_t* guess_rot, int32_t seed_mid[3], int32_t seed_rot[3]) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        c->cx->debug_seeds(guess_pos, guess_rot, seed_mid, seed_rot);
    });
}
int dh_debug_votes(dh_ctx* c, int which, int32_t* keys, uint32_t* vals, uint64_t* n, int32_t box_origin[3],
                   int32_t* box_dim) {
    return guarded([&] {
        REQUIRE(c, "NULL ctx");
        REQUIRE((keys == nullptr) == (vals == nullptr), "keys and vals must both be NULL or both be set");
        c->cx->debug_votes(which, keys, vals, n, box_origin, box_dim);
    });
}
int dh_debug_meanshift(dh_ctx* c, int which, int32_t* pos, uint32_t* n_iter) {
    return guarded([&] {
        REQUIRE(c && n_iter, "NULL argument");
        c->cx->debug_meanshift(which, pos, n_iter);
    });
}
int dh_debug_meanshift_flags(dh_ctx* c, uint32_t flags[2]) {
    return guarded([&] {
        REQUIRE(c && flags, "NULL argument");
        uint32_t n = 0;
        c->cx->debug_meanshift(0, nullptr, &n);
        n = 0;
        c->cx->debug_meanshift(1, nullptr, &n);
        flags[0] = c->cx->last_ms_flags(0);
        flags[1] = c->cx->last_ms_flags(1);
    });
}
int dh_debug_leaf_static(dh_ctx* c, const dh_forest* f, uint32_t* valtoadd, uint8_t* rot_ok, uint8_t* off_ok) {
    return guarded([&] {
        REQUIRE(c && f, "NULL argument");
        c->cx->debug_leaf_static(*f->hf, valtoadd, rot_ok, off_ok);
    });
}

}  // extern "C"
