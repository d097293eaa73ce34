/* depthhead_cuda.h — C ABI of libdepthhead_cuda.so: the B200 (sm_100a) replacement for
 * depthhead's Hough-forest prediction path.
 *
 * These are the entry points a thin Rust crate (`depthhead-cuda`, see INTEGRATION.md) binds with
 * an `extern "C"` block to stand in for `HoughPrediction::predict_parameter_parallel` and its
 * siblings.  Plain pointers and sizes only; nothing here unwinds across the boundary; there is
 * NO CPU fallback — without a usable CUDA device every compute call returns DH_E_CUDA.
 *
 * Reference interfaces replaced (paths relative to the depthhead repository):
 *   src/hough/prediction.rs:239-256   struct HoughPrediction (serde JSON)      -> dh_forest_*
 *   src/hough/prediction.rs:320-331   update_sigma / sigma                     -> dh_forest_{set,get}_sigma
 *   src/hough/prediction.rs:242,255   pub stepwidth, pub meanshift_iterations  -> dh_forest_{get,set}_*
 *   src/types.rs:405-446              IntrinsicMatrix                          -> `const float K[9]`
 *   src/hough/prediction.rs:376-409   predict_parameter{,_parallel}            -> dh_predict, dh_predict_batch
 *   src/hough/prediction.rs:259-267   struct PredictionResult                  -> dh_result
 *   examples/live_prediction.rs:75-88 frame-to-frame seeding of a sequence     -> dh_predict_sequences
 *   predict_parameter_parallel over n frames, each with its own K and seeds    -> dh_predict_frames,
 *                                                                                 dh_predict_frames_biwi
 *   src/hough/prediction.rs:850-905   predict_mask                             -> dh_predict_mask
 *   src/hough/prediction.rs:760-841   build_hough_image (votes, before blur)   -> dh_hough_image_raw
 *   src/hough/prediction.rs:760-845   build_hough_image (with its blur)        -> dh_build_hough_image
 *   src/hough/prediction.rs:343-367   predict_parameter_from2dhough            -> dh_predict_from2dhough
 *   the three above over n frames                                              -> dh_predict_mask_batch,
 *                                                                                 dh_build_hough_image_batch
 *   src/db_reader/biwi.rs:81-103      read_depth (run-length coded depth file)  -> dh_biwi_depth_dims,
 *                                                                                 dh_biwi_decode_depth, dh_predict_batch_biwi
 *   src/db_reader/biwi.rs:27-60       read_cal (depth.cal -> IntrinsicMatrix)   -> dh_biwi_parse_cal
 *   src/db_reader/biwi.rs:63-77       read_gt (ground-truth pose file)          -> dh_biwi_parse_pose
 *   src/hough/houghforest.rs:250-295  HoughTreeFunctions::impurity (training)   -> dh_train_score_level
 *   src/hough/houghforest.rs:185-193  binarize of the chosen split (training)   -> dh_train_split_level
 */
#ifndef DEPTHHEAD_CUDA_H
#define DEPTHHEAD_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DH_ABI_VERSION 1

/* error codes (0 = ok) */
#define DH_OK 0
#define DH_E_JSON (-1)   /* malformed document / forest the reference itself would panic on */
#define DH_E_SHAPE (-2)  /* image smaller than the sub-image, zero stride, unsupported sizes */
#define DH_E_CUDA (-3)   /* no device, wrong architecture, CUDA runtime failure */
#define DH_E_ARG (-4)    /* NULL / out-of-range argument */
#define DH_E_STATE (-5)  /* debug query without a preceding debug-enabled predict */

typedef struct dh_forest dh_forest; /* immutable model: shareable across threads and GPUs */
typedef struct dh_ctx dh_ctx;       /* one per GPU per host thread: stream, scratch, device copy */

/* prediction.rs:259-267 PredictionResult.  mid_point: whole millimetres; rotation: radians
 * (multiples of 3 degrees, pi = 3.14159 as in the reference); bounding_box: always 0,0,0,0
 * (topleft x,y, bottomright x,y) because the reference never predicts it. */
typedef struct dh_result {
    float mid_point[3];
    uint32_t _pad;
    double rotation[3];
    uint32_t bounding_box[4];
} dh_result;

/* Thread-local description of the last failure in this thread (never NULL). */
const char* dh_last_error(void);
int dh_abi_version(void);
/* Identifies the build: a hash of the library's sources, fixed at compile time (profiles recorded
 * under profiles/ carry it, so a number is only ever quoted for the build it was measured on). */
const char* dh_build_id(void);

/* ------------------------------------------------------------------ model (HoughPrediction) */
/* serde_json::from_str::<HoughPrediction>(json)  (Readme.md:82-86, prediction.rs:239-256).
 * Parses the document, flattens the forest into structure-of-arrays node/leaf/vote tables and
 * validates everything the reference would panic on at prediction time.  Host-only. */
int dh_forest_from_json(const char* json, size_t len, dh_forest** out);

/* Same model from already-flat arrays (the binary SoA form; skips JSON for very large forests).
 * tree_node_off/tree_leaf_off: n_trees+1 prefix offsets; rects: int32[n_nodes][8] =
 * r1.topleft x,y, r1.bottomright x,y, r2...; child: int32[n_nodes][2], >=0 = node index local to
 * the tree (root = 0), <0 = ~(leaf index local to the tree); vote_off: n_leaves+1. */
typedef struct dh_forest_arrays {
    uint32_t stepwidth, subimage_width, subimage_height, meanshift_iterations;
    float gaussian_sigma;
    int32_t n_trees;
    const int64_t* tree_node_off;
    const int64_t* tree_leaf_off;
    const int32_t* rects;
    const double* threshold;
    const int32_t* child;
    const double* prob;
    const int64_t* vote_off;
    const float* offsets;     /* [n_votes][3] mm  */
    const double* rotations;  /* [n_votes][3] deg */
} dh_forest_arrays;
int dh_forest_from_arrays(const dh_forest_arrays* a, dh_forest** out);
void dh_forest_free(dh_forest* f);

uint32_t dh_forest_get_stepwidth(const dh_forest* f);
int dh_forest_set_stepwidth(dh_forest* f, uint32_t v);              /* pub field, prediction.rs:242 */
uint32_t dh_forest_get_meanshift_iterations(const dh_forest* f);
int dh_forest_set_meanshift_iterations(dh_forest* f, uint32_t v);   /* pub field, prediction.rs:255 */
float dh_forest_get_sigma(const dh_forest* f);                      /* sigma(), prediction.rs:329 */
int dh_forest_set_sigma(dh_forest* f, float v);                     /* update_sigma, prediction.rs:320-326:
                                                                       ignored if v<=0 or unchanged */
uint32_t dh_forest_get_subimage_width(const dh_forest* f);
uint32_t dh_forest_get_subimage_height(const dh_forest* f);
int32_t dh_forest_n_trees(const dh_forest* f);
int64_t dh_forest_n_nodes(const dh_forest* f);
int64_t dh_forest_n_leaves(const dh_forest* f);
int64_t dh_forest_n_votes(const dh_forest* f);
/* Leaf numbering used by the debug exports: global leaf id = tree_leaf_off[t] + index in file order. */

/* ------------------------------------------------------------------ context */
int dh_ctx_create(int device, dh_ctx** out);
void dh_ctx_free(dh_ctx* c);
/* Run on a caller-owned CUDA stream (cudaStream_t as void*; NULL = the context's own stream). */
int dh_ctx_set_stream(dh_ctx* c, void* cuda_stream);
/* Frames processed per pipeline pass (scratch is sized for this many); 0 = default. */
int dh_ctx_set_chunk_frames(dh_ctx* c, uint32_t frames);
int dh_ctx_synchronize(dh_ctx* c);
/* dh_predict_batch with HOST frames: the frames are mostly background (0), so worker threads of the
 * context rewrite every chunk as run-length files (the Biwi format, see dh_biwi_encode_depth) in
 * pinned memory, only those bytes cross PCIe, and the GPU expands them again bit for bit; chunks
 * that are too dense to gain are copied raw.  n = number of worker threads (0 = default: the cores
 * this process may run on, at most 16; DH_ENCODE_THREADS overrides).  DH_HOST_ENCODE=0 turns the
 * rewrite off, =1 forces it for every chunk. */
int dh_ctx_set_encode_threads(dh_ctx* c, uint32_t n);
/* Host->device traffic of the LAST dh_predict_batch / dh_predict_batch_biwi call:
 * [0] bytes copied host->device, [1] chunks that went through the run-length rewrite,
 * [2] worker threads of the context (0 = none started yet), [3] reserved. */
int dh_ctx_transfer_info(dh_ctx* c, uint64_t info[4]);

/* ------------------------------------------------------------------ prediction */
#define DH_DEPTH_HOST 0   /* depth points to host memory (pinned preferred) */
#define DH_DEPTH_DEVICE 1 /* depth points to device memory on the context's GPU */

/* predict_parameter_parallel (prediction.rs:397-409).  depth: w*h u16 millimetres, row-major,
 * 0 = invalid (types.rs:10).  K: row-major 3x3 intrinsic matrix.  midp_guess (mm) and rot_guess
 * (radians) may be NULL = None.  Synchronous: *out is valid on return. */
int dh_predict(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
               const float* midp_guess, const double* rot_guess, dh_result* out);

/* n independent frames [n][h][w] with seeds = None, results to out[n] (host).  depth_loc says
 * where `depth` lives.  Synchronous. */
int dh_predict_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                     const float K[9], int depth_loc, dh_result* out);

/* The reference's real use predicts SEQUENCES (examples/live_prediction.rs:75-88): frame t is seeded
 * with the pose of frame t - 1 — midp_guess = the previous mid_point if its z exceeds min_seed_z
 * (500.0 there; the first frame has none), rot_guess = the previous rotation (none for the first
 * frame).  That makes one sequence sequential, but separate sequences are independent: depth holds
 * n_seq sequences of frames_per_seq frames, sequence-major ([n_seq][frames_per_seq][h][w]); frame t
 * of every sequence runs as one pass on the GPU, seeded on the device from pass t - 1.  Results in
 * input order: out[s * frames_per_seq + t], equal to calling dh_predict frame by frame with those
 * seeds.  Synchronous. */
int dh_predict_sequences(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n_seq, uint32_t frames_per_seq,
                         uint32_t w, uint32_t h, const float K[9], int depth_loc, float min_seed_z, dh_result* out);

/* The arguments of dh_predict for one frame of dh_predict_frames: its own intrinsics and seeds. */
typedef struct dh_frame_args {
    float K[9];            /* row-major intrinsics of this frame */
    float midp_guess[3];   /* mm; used iff has_guess bit 0 */
    double rot_guess[3];   /* radians; used iff has_guess bit 1 */
    uint32_t has_guess;    /* bit 0 midp_guess, bit 1 rot_guess; 0 = (None, None) */
    uint32_t _pad;
} dh_frame_args;           /* 80 bytes */

/* predict_parameter_parallel(img, K_i, midp_i, rot_i) for n independent frames [n][h][w] at
 * depth_loc, frame i with args[i] (host memory); results to out[n] (host).  Results are equal,
 * bit for bit, to calling dh_predict frame by frame with the same arguments, through the chunked
 * pipeline of dh_predict_batch (device-resident or host frames, the run-length host path).  K is
 * not validated, as in dh_predict.  A has_guess with bits other than 0-1 is DH_E_ARG naming the
 * frame.  Synchronous; n = 0 is a successful no-op. */
int dh_predict_frames(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                      int depth_loc, const dh_frame_args* args, dh_result* out);

/* predict_mask (prediction.rs:850-905): mask[h][w] u8 to host memory. */
int dh_predict_mask(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, uint8_t* mask);
/* build_hough_image before its gaussian blur (prediction.rs:760-841): votes[h][w] u16 to host. */
int dh_hough_image_raw(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h,
                       const float K[9], uint16_t* votes);

/* build_hough_image (prediction.rs:760-845): the vote image blurred with the model's gaussian_sigma
 * (imageproc::gaussian_blur_f32, an external crate: its kernel — radius ceil(2 sigma), unnormalised
 * pdf taps —, edge-clamped borders and u16 truncation after each of the two passes are restated
 * from its published source, see DESIGN.md): hough[h][w] u16 to host. */
int dh_build_hough_image(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                         uint16_t* hough);
/* predict_parameter_from2dhough (prediction.rs:343-367): arg-max of that image (the LAST of equal
 * maxima, as Iterator::max_by_key), z = depth at the pixel, mid_point = back-projection; rotation and
 * bounding box are 0. */
int dh_predict_from2dhough(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t w, uint32_t h, const float K[9],
                           dh_result* out);

/* The three calls above over n independent frames [n][h][w] at depth_loc, through the same chunked
 * pipeline as dh_predict_batch (device-resident or host frames; results equal to calling the
 * single-frame entry points frame by frame).  Images go to [n][h][w] at mask_loc / hough_loc
 * (DH_DEPTH_HOST or DH_DEPTH_DEVICE).  Synchronous; n = 0 is a successful no-op. */
int dh_predict_mask_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                          int depth_loc, uint8_t* mask, int mask_loc);
/* blur = 0: the raw vote image (dh_hough_image_raw); blur = 1: build_hough_image.  hough may be NULL
 * (no image copied out); from2d (n results, host memory) may be NULL: predict_parameter_from2dhough
 * per frame.  from2d needs blur = 1; hough and from2d both NULL is DH_E_ARG. */
int dh_build_hough_image_batch(dh_ctx* c, const dh_forest* f, const uint16_t* depth, uint32_t n, uint32_t w, uint32_t h,
                               const float K[9], int depth_loc, int blur, uint16_t* hough, int hough_loc, dh_result* from2d);

/* ------------------------------------------------------------------ Biwi Kinect Head Pose wire formats */
/* read_depth (biwi.rs:81-103): u32 width, u32 height, then until width*height pixels are covered
 * [u32 n_empty][u32 n_full][n_full x u16], all little-endian; pixels of empty runs are 0.  The
 * compressed files of n frames are handed over as ONE blob: frame i occupies bytes
 * [offsets[i], offsets[i+1]) (offsets: n+1 entries, each a multiple of 4; padding between files is
 * fine), so that the COMPRESSED bytes cross PCIe and the runs are expanded on the GPU.
 * A file the reference would fail on (truncated: UnexpectedEof; a run past the last pixel: panic)
 * or whose header differs from w x h gives DH_E_ARG naming the first bad frame. */

/* header of one file: width and height (host-only, no GPU needed) */
int dh_biwi_depth_dims(const uint8_t* file, size_t len, uint32_t* w, uint32_t* h);
/* Expand n frames to out[n][h][w] u16; blob and offsets in host memory; out_loc says whether `out`
 * is host or device memory (DH_DEPTH_HOST / DH_DEPTH_DEVICE). */
int dh_biwi_decode_depth(dh_ctx* c, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t w, uint32_t h,
                         uint16_t* out, int out_loc);
/* read_depth + predict_parameter_parallel(img, K, None, None) for n frames: what
 * examples/db_evaluate.rs:296 does per file, with the decode on the GPU. */
int dh_predict_batch_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                          uint32_t w, uint32_t h, const float K[9], dh_result* out);
/* The same with the arguments of every frame (dh_predict_frames): a whole database, whose sequence
 * folders each have their own depth.cal, in one call. */
int dh_predict_frames_biwi(dh_ctx* c, const dh_forest* f, const uint8_t* blob, const uint64_t* offsets, uint32_t n,
                           uint32_t w, uint32_t h, const dh_frame_args* args, dh_result* out);
/* The writer for that format (the reference only reads it): n raw frames [n][h][w] u16 become n
 * files in ONE blob, file i at [offsets[i], offsets[i+1]) (offsets: n+1 entries, multiples of 16).
 * Runs are found at a granularity of 16 pixels: a group of 16 pixels with any non-zero pixel is
 * stored verbatim (isolated zeros inside it travel as literal zeros, which the format allows), so
 * read_depth gives back exactly the input.  This is the encoder dh_predict_batch runs on its own
 * worker threads for host frames (see dh_ctx_set_encode_threads).  Host-only, `threads` workers
 * (0 = the default).  Copies at most cap bytes and reports the full length in *needed (call with
 * cap = 0 to size the buffer; dh_biwi_encode_bound(w, h) * n + 16 always suffices). */
size_t dh_biwi_encode_bound(uint32_t w, uint32_t h);
int dh_biwi_encode_depth(const uint16_t* frames, uint32_t n, uint32_t w, uint32_t h, uint32_t threads, uint8_t* blob, size_t cap,
                         uint64_t* offsets, size_t* needed);
/* read_cal (biwi.rs:27-60): the first three lines of depth.cal, three numbers each (tokens
 * matching \d+[\.\d+]* exactly as the reference's regex, so a sign is not part of a number), to
 * a row-major 3x3 matrix.  Host-only. */
int dh_biwi_parse_cal(const char* text, size_t len, float K[9]);
/* read_gt (biwi.rs:63-77): six little-endian f32 (position mm, rotation), plus the position
 * projected with K (space_to_img_coord).  Host-only. */
int dh_biwi_parse_pose(const uint8_t* file, size_t len, const float K[9], float pos3d[3], float pos2d[2], float rot[3]);

/* ------------------------------------------------------------------ training: split scoring */
/* The reference grows its trees with stamm's train_forest_parallel (an external crate), which
 * calls HoughTreeFunctions::impurity (houghforest.rs:250-295) for every candidate NodeParam of
 * every node.  These entry points evaluate that for all nodes of one tree level on the GPU; the
 * loop that grows the tree stays with the caller (depthhead_b200/train.py mirrors HoughLearning). */
typedef struct dh_trainset dh_trainset;  /* training samples resident on one GPU */
/* n samples: patches[n][sh][sw] u16 (the cropped sub-images of prediction.rs:223-226),
 * is_object[n] (Truth::Object or NoObject), offsets[n][3] f32 mm and rotations[n][3] f64 of the
 * Object samples (ignored for the others).  rw x rh: the one rectangle size every candidate
 * feature will have (subrect_feature_scale of hough_tree_trainer.rs:165 applied to the sub-image). */
int dh_trainset_create(dh_ctx* c, const uint16_t* patches, uint64_t n, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh,
                       const uint8_t* is_object, const float* offsets, const double* rotations, dh_trainset** out);
void dh_trainset_free(dh_trainset* t);
/* per candidate: side 0 = binarize Zero, side 1 = One.  det_*: determinants of the covariance
 * matrices of the side's Object offsets / rotations (NaN with fewer than two of them); impurity:
 * houghforest.rs:250-295, NaN where the reference itself aborts (an empty side: its
 * assert!(res.is_finite()); a determinant sum below -0.001: its unreachable!()). */
typedef struct dh_split_stats {
    uint32_t n[2], n_pos[2];
    double det_off[2], det_rot[2];
    double impurity;
} dh_split_stats;
/* One tree level: node k owns sample_idx[node_off[k] .. node_off[k+1]) (indices into the training
 * set, in set order); cand_rects[n_nodes][m][8] (r1 x0,y0,x1,y1, r2 ..; bottomright exclusive) and
 * cand_thr[n_nodes][m] are its m candidates; out[n_nodes][m]. */
int dh_train_score_level(dh_ctx* c, const dh_trainset* t, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                         const int32_t* cand_rects, const double* cand_thr, uint32_t m, uint64_t depth, double steepness,
                         dh_split_stats* out);
/* binarize (houghforest.rs:185-193) of ONE chosen NodeParam per node over the node's samples:
 * bits[node_off[n_nodes]] (1 = One). */
int dh_train_split_level(dh_ctx* c, const dh_trainset* t, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                         const int32_t* rects, const double* thr, uint8_t* bits);

/* HoughLearning::new + learn (prediction.rs:106-143, 145-234) on an already extracted sample set
 * (the windows the per-image loop of learn collects, in training order): grows n_trees trees with
 * the callbacks of houghforest.rs:196-311 scored on the GPU and returns the model, ready for
 * dh_predict* and dh_forest_to_json.  The tree-growing loop and the random numbers are this
 * library's (stamm 0.2.0 and rand::thread_rng cannot be reproduced, see DESIGN.md section 9);
 * the same seed and samples always give the same forest. */
typedef struct dh_train_params {
    uint32_t stepwidth, subimage_width, subimage_height;   /* HoughLearning::new arguments, in order */
    uint32_t max_depth, n_trees, subset_per_tree;
    double subrect_feature_scale;
    uint32_t features_per_node, min_subset_size;
    double steepness;
    float gaussian_sigma;                                  /* learn(gaussian_sigma, ..) */
    uint32_t _pad;
    uint64_t seed;
} dh_train_params;
int dh_train_forest(dh_ctx* c, const dh_train_params* p, const uint16_t* patches, uint64_t n, const uint8_t* is_object,
                    const float* offsets, const double* rotations, dh_forest** out);
/* HoughLearning::learn (prediction.rs:145-234) from annotated frames (db_reader DepthTrue): depth
 * [n][h][w] u16, head mask [n][h][w] u8 (non-zero = head), per-frame intrinsics K[n][9], head
 * centre pos3d[n][3] (mm) and rotation rot[n][3].  Extracts the windows exactly as the reference
 * (sliding window at p->stepwidth, background test, truth from the mask at the window centre,
 * offset = back-projected centre - pos3d; 20 negatives and 20 positives per frame after a random
 * permutation), then dh_train_forest with seed + 1. */
int dh_train_learn(dh_ctx* c, const dh_train_params* p, uint32_t n_frames, uint32_t w, uint32_t h, const uint16_t* depth,
                   const uint8_t* mask, const float* K, const float* pos3d, const float* rot, dh_forest** out);
/* serde_json::to_string(&HoughPrediction) — what hough_tree_trainer.rs:182 writes.  Copies at most
 * cap bytes (no terminator) and reports the full length in *needed; call with cap = 0 to size the buffer. */
int dh_forest_to_json(const dh_forest* f, char* buf, size_t cap, size_t* needed);

/* ------------------------------------------------------------------ measurement */
/* Per-stage device time (CUDA events on the context's stream) of the LAST dh_predict_batch call,
 * summed over its chunks, in milliseconds.  Order of stages: see DH_STAGE_*.  After the 2-D calls
 * (dh_predict_mask*, dh_hough_image_raw, dh_build_hough_image*, dh_predict_from2dhough) H2D, SAT,
 * TRAVERSE and D2H mean the same, and their whole back end (mask or vote image, blur, arg-max) is
 * booked under DH_STAGE_VOTE; GATE and MEANSHIFT stay 0. */
#define DH_STAGE_H2D 0
#define DH_STAGE_SAT 1
#define DH_STAGE_TRAVERSE 2
#define DH_STAGE_GATE 3      /* patch gate, hit list, coarse seed grids */
#define DH_STAGE_VOTE 4      /* seeds + accumulator cubes */
#define DH_STAGE_MEANSHIFT 5
#define DH_STAGE_D2H 6
#define DH_N_STAGES 7
int dh_ctx_enable_stage_timing(dh_ctx* c, int on);
int dh_ctx_stage_ms(dh_ctx* c, float ms[DH_N_STAGES]);
/* Work counters of the last dh_predict/dh_predict_batch call:
 * [0] frames, [1] patches (all), [2] valid (non-background) patches, [3] patch*tree evals,
 * [4] node visits, [5] gate-passing patches, [6] hits (voting patch*tree pairs, both lists), [7] centre
 * votes cast, [8] rotation votes cast, [9] kernel launches, [10] mean-shift rounds run (both
 * accumulators), [11] accumulator-cube rebuilds.  After a 2-D call [0]-[4] and [9] are filled and
 * the others are 0. */
#define DH_N_COUNTERS 12
int dh_ctx_counters(dh_ctx* c, uint64_t counters[DH_N_COUNTERS]);

/* ------------------------------------------------------------------ debug exports (parity tests) */
/* Keep the intermediates of the last dh_predict call (single frame) on the device. */
int dh_ctx_enable_debug(dh_ctx* c, int on);
/* patches per row / column of the sliding window of the last call */
int dh_debug_dims(dh_ctx* c, uint32_t* npx, uint32_t* npy, uint32_t* n_trees);
/* leaf[P][T] global leaf id, -1 = background patch; visited may be NULL */
int dh_debug_leaf_indices(dh_ctx* c, int32_t* leaf /*[P*T]*/);
/* p3[P][3] back-projected patch centres; gate[P] = 1 iff mean prob > 0.7 */
int dh_debug_patches(dh_ctx* c, float* p3, uint8_t* gate);
/* coarse seed grids (400 + 8000 u32) and the seeds handed to mean-shift */
int dh_debug_seeds(dh_ctx* c, uint32_t* guess_pos, uint32_t* guess_rot, int32_t seed_mid[3], int32_t seed_rot[3]);
/* Accumulator contents as unsorted (key, value) lists.  which: 0 = centre, 1 = rotation.
 * The device keeps the cells of a dense cube of box_dim^3 cells starting at box_origin (the cube
 * around the last mean-shift position, see DESIGN.md); only its non-zero cells are returned.
 * Call with keys == NULL to get the count (at most box_dim^3). */
int dh_debug_votes(dh_ctx* c, int which, int32_t* keys /*[n][3]*/, uint32_t* vals, uint64_t* n,
                   int32_t box_origin[3], int32_t* box_dim);
/* mean-shift trajectory: positions after each executed iteration; *n_iter in/out */
int dh_debug_meanshift(dh_ctx* c, int which, int32_t* pos /*[n_iter][3]*/, uint32_t* n_iter);
/* flags of the last mean-shift runs: bit0 = zero-sum break (meanshift.rs:385-388) */
int dh_debug_meanshift_flags(dh_ctx* c, uint32_t flags[2]);
/* tile plan of the traversal kernel for the last call's shape: patches per tile x, y; tiles per
 * frame x, y; tile extent in elements x, y; dynamic shared memory bytes; threads per CTA */
int dh_debug_tile_plan(dh_ctx* c, uint32_t plan[8]);
/* per-leaf static quantities computed by the leaf-gate kernel: valtoadd, rot_ok, off_ok */
int dh_debug_leaf_static(dh_ctx* c, const dh_forest* f, uint32_t* valtoadd, uint8_t* rot_ok, uint8_t* off_ok);

#ifdef __cplusplus
}
#endif
#endif /* DEPTHHEAD_CUDA_H */
