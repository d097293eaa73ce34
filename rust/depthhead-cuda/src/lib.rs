//! Drop-in for the prediction path of depthhead's `HoughPrediction` on an NVIDIA B200: the same
//! type names, fields and method signatures as `src/hough/prediction.rs` and `src/types.rs` of
//! the reference, on top of the C ABI of `libdepthhead_cuda.so` (`include/depthhead_cuda.h`).
//!
//! What the reference's own caller does compiles unchanged against this crate
//! (`examples/live_prediction.rs:76,86,108,166-173`):
//!
//! ```ignore
//! let forest: HoughPrediction = serde_json::from_str(&json)?;            // Deserialize
//! let res = forest.predict_parameter_parallel(img, &intrinsic, None, None);   // img: Arc<DepthImage>
//! let res = forest.predict_parameter_parallel(img, &intrinsic, Some(mid), Some(rot));
//! let mask = forest.predict_mask(img.clone());
//! ```
//!
//! NOT compiled in the build image of this repository (no cargo / rustc there): the same C ABI
//! is exercised from C (`tests/test_capi_c.py`) and from Python (`depthhead_b200/capi.py`).
//! The model FILE format is this library's (the `forest` member is not stamm 0.2.0's serde
//! layout, whose source is not available): see INTEGRATION.md.
extern crate image;
extern crate serde;
extern crate serde_json;

use std::cell::Cell;
use std::ffi::CStr;
use std::os::raw::{c_char, c_int};
use std::sync::Arc;

use image::{ImageBuffer, Luma};
use serde::de::{Deserialize, Deserializer, Error as DeError};
use serde::ser::{Error as SerError, Serialize, Serializer};

#[repr(C)] pub struct DhForest { _p: [u8; 0] }
#[repr(C)] pub struct DhCtx { _p: [u8; 0] }

/// include/depthhead_cuda.h: dh_result
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct DhResult {
    pub mid_point: [f32; 3],
    pub _pad: u32,
    pub rotation: [f64; 3],
    pub bounding_box: [u32; 4],
}

/// HoughLearning::new arguments (prediction.rs:106-116), learn's sigma, and a seed (the reference
/// draws from thread_rng; here the same seed always gives the same forest)
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct DhTrainParams {
    pub stepwidth: u32, pub subimage_width: u32, pub subimage_height: u32,
    pub max_depth: u32, pub n_trees: u32, pub subset_per_tree: u32,
    pub subrect_feature_scale: f64, pub features_per_node: u32, pub min_subset_size: u32,
    pub steepness: f64, pub gaussian_sigma: f32, pub _pad: u32, pub seed: u64,
}

/// include/depthhead_cuda.h: dh_frame_args, the arguments of dh_predict for one frame of
/// dh_predict_frames (80 bytes)
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct DhFrameArgs {
    pub k: [f32; 9],
    pub midp_guess: [f32; 3],
    pub rot_guess: [f64; 3],
    pub has_guess: u32,
    pub _pad: u32,
}
const _: () = assert!(std::mem::size_of::<DhFrameArgs>() == 80);

extern "C" {
    fn dh_last_error() -> *const c_char;
    fn dh_forest_from_json(json: *const c_char, len: usize, out: *mut *mut DhForest) -> c_int;
    fn dh_forest_to_json(f: *const DhForest, buf: *mut c_char, cap: usize, needed: *mut usize) -> c_int;
    fn dh_forest_free(f: *mut DhForest);
    fn dh_forest_get_stepwidth(f: *const DhForest) -> u32;
    fn dh_forest_set_stepwidth(f: *mut DhForest, v: u32) -> c_int;
    fn dh_forest_get_meanshift_iterations(f: *const DhForest) -> u32;
    fn dh_forest_set_meanshift_iterations(f: *mut DhForest, v: u32) -> c_int;
    fn dh_forest_get_sigma(f: *const DhForest) -> f32;
    fn dh_forest_set_sigma(f: *mut DhForest, v: f32) -> c_int;
    fn dh_ctx_create(device: c_int, out: *mut *mut DhCtx) -> c_int;
    fn dh_ctx_free(c: *mut DhCtx);
    fn dh_predict(c: *mut DhCtx, f: *const DhForest, depth: *const u16, w: u32, h: u32, k: *const f32,
                  midp_guess: *const f32, rot_guess: *const f64, out: *mut DhResult) -> c_int;
    fn dh_predict_batch(c: *mut DhCtx, f: *const DhForest, depth: *const u16, n: u32, w: u32, h: u32,
                        k: *const f32, depth_loc: c_int, out: *mut DhResult) -> c_int;
    fn dh_predict_frames(c: *mut DhCtx, f: *const DhForest, depth: *const u16, n: u32, w: u32, h: u32, depth_loc: c_int,
                         args: *const DhFrameArgs, out: *mut DhResult) -> c_int;
    fn dh_predict_sequences(c: *mut DhCtx, f: *const DhForest, depth: *const u16, n_seq: u32, frames_per_seq: u32,
                            w: u32, h: u32, k: *const f32, depth_loc: c_int, min_seed_z: f32, out: *mut DhResult) -> c_int;
    fn dh_predict_mask(c: *mut DhCtx, f: *const DhForest, depth: *const u16, w: u32, h: u32, mask: *mut u8) -> c_int;
    fn dh_build_hough_image(c: *mut DhCtx, f: *const DhForest, depth: *const u16, w: u32, h: u32, k: *const f32,
                            hough: *mut u16) -> c_int;
    fn dh_predict_from2dhough(c: *mut DhCtx, f: *const DhForest, depth: *const u16, w: u32, h: u32, k: *const f32,
                              out: *mut DhResult) -> c_int;
    fn dh_predict_mask_batch(c: *mut DhCtx, f: *const DhForest, depth: *const u16, n: u32, w: u32, h: u32,
                             depth_loc: c_int, mask: *mut u8, mask_loc: c_int) -> c_int;
    fn dh_build_hough_image_batch(c: *mut DhCtx, f: *const DhForest, depth: *const u16, n: u32, w: u32, h: u32, k: *const f32,
                                  depth_loc: c_int, blur: c_int, hough: *mut u16, hough_loc: c_int, from2d: *mut DhResult) -> c_int;
    // Biwi wire formats (src/db_reader/biwi.rs:27-103)
    fn dh_biwi_depth_dims(file: *const u8, len: usize, w: *mut u32, h: *mut u32) -> c_int;
    fn dh_biwi_decode_depth(c: *mut DhCtx, blob: *const u8, offsets: *const u64, n: u32, w: u32, h: u32,
                            out: *mut u16, out_loc: c_int) -> c_int;
    fn dh_predict_batch_biwi(c: *mut DhCtx, f: *const DhForest, blob: *const u8, offsets: *const u64, n: u32,
                             w: u32, h: u32, k: *const f32, out: *mut DhResult) -> c_int;
    fn dh_predict_frames_biwi(c: *mut DhCtx, f: *const DhForest, blob: *const u8, offsets: *const u64, n: u32,
                              w: u32, h: u32, args: *const DhFrameArgs, out: *mut DhResult) -> c_int;
    fn dh_biwi_parse_cal(text: *const c_char, len: usize, k: *mut f32) -> c_int;
    fn dh_biwi_parse_pose(file: *const u8, len: usize, k: *const f32, pos3d: *mut f32, pos2d: *mut f32,
                          rot: *mut f32) -> c_int;
    // training (src/hough/prediction.rs:106-234, src/hough/houghforest.rs:196-311)
    fn dh_train_learn(c: *mut DhCtx, p: *const DhTrainParams, n_frames: u32, w: u32, h: u32, depth: *const u16,
                      mask: *const u8, k: *const f32, pos3d: *const f32, rot: *const f32, out: *mut *mut DhForest) -> c_int;
}

#[derive(Debug)]
pub struct Error { pub code: i32, pub message: String }
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter) -> std::fmt::Result { write!(f, "{} (code {})", self.message, self.code) }
}
impl std::error::Error for Error { fn description(&self) -> &str { &self.message } }
fn check(rc: c_int) -> Result<(), Error> {
    if rc == 0 { return Ok(()); }
    let message = unsafe { CStr::from_ptr(dh_last_error()) }.to_string_lossy().into_owned();
    Err(Error { code: rc, message })
}

/// types.rs:10
pub type DepthImage = ImageBuffer<Luma<u16>, Vec<u16>>;

/// types.rs:28-62 (the part PredictionResult needs)
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct Rect { topleft: [u32; 2], bottomright: [u32; 2] }
impl Rect {
    pub fn new(x: u32, y: u32, width: u32, height: u32) -> Rect { Rect { topleft: [x, y], bottomright: [x + width, y + height] } }
    pub fn width(&self) -> u32 { self.bottomright[0] - self.topleft[0] }
    pub fn height(&self) -> u32 { self.bottomright[1] - self.topleft[1] }
    pub fn x(&self) -> u32 { self.topleft[0] }
    pub fn y(&self) -> u32 { self.topleft[1] }
}

/// types.rs:405-446.  `.0` is the row-major 3x3 matrix (the reference's `Mat3<f32>` converts from
/// and to `[[f32; 3]; 3]`); the inverse is computed inside the library (adjugate / det, f32, the
/// formula of meancov_estimation.rs:344-352).
#[derive(Clone, Debug)]
pub struct IntrinsicMatrix(pub [[f32; 3]; 3]);
impl IntrinsicMatrix {
    pub fn new<T: Into<[[f32; 3]; 3]>>(mat: T) -> IntrinsicMatrix { IntrinsicMatrix(mat.into()) }
    /// types.rs:418-420
    pub fn default_kinect_intrinsic() -> IntrinsicMatrix {
        IntrinsicMatrix::new([[560.0, 0.0, 320.0], [0.0, 560.0, 240.0], [0.0, 0.0, 1.0]])
    }
    fn ptr(&self) -> *const f32 { self.0.as_ptr() as *const f32 }
}

/// prediction.rs:259-267
pub struct PredictionResult {
    pub mid_point: [f32; 3],
    pub rotation: [f64; 3],
    pub bounding_box: Rect,
}
impl PredictionResult {
    fn from_c(r: &DhResult) -> PredictionResult {
        PredictionResult { mid_point: r.mid_point, rotation: r.rotation,
                           bounding_box: Rect::new(r.bounding_box[0], r.bounding_box[1], r.bounding_box[2], r.bounding_box[3]) }
    }
}

/// prediction.rs:239-256.  The two fields the reference makes `pub` are `pub` here and are read at
/// every prediction; the model itself lives behind the C ABI.  Like the reference (a `RefCell`
/// inside) the type is Send but not Sync: one predictor per thread.  The GPU context is created at
/// the first prediction, on the device named by the environment variable DEPTHHEAD_CUDA_DEVICE
/// (default 0).
pub struct HoughPrediction {
    /// stepwidth use for sliding window (prediction.rs:242)
    pub stepwidth: u32,
    /// number of iteration used for meanshifting (prediction.rs:255)
    pub meanshift_iterations: u32,
    forest: *mut DhForest,
    ctx: Cell<*mut DhCtx>,
}
unsafe impl Send for HoughPrediction {}

impl HoughPrediction {
    fn from_handle(forest: *mut DhForest) -> HoughPrediction {
        HoughPrediction {
            stepwidth: unsafe { dh_forest_get_stepwidth(forest) },
            meanshift_iterations: unsafe { dh_forest_get_meanshift_iterations(forest) },
            forest,
            ctx: Cell::new(std::ptr::null_mut()),
        }
    }
    /// the document `serde_json::from_str::<HoughPrediction>` reads (Readme.md:82-86)
    pub fn from_json(text: &str) -> Result<HoughPrediction, Error> {
        let mut f = std::ptr::null_mut();
        check(unsafe { dh_forest_from_json(text.as_ptr() as *const c_char, text.len(), &mut f) })?;
        Ok(HoughPrediction::from_handle(f))
    }
    /// what `tojson(&tree, filename)` writes (examples/hough_tree_trainer.rs:182)
    pub fn to_json(&self) -> Result<String, Error> {
        self.push_fields()?;
        let mut need = 0usize;
        check(unsafe { dh_forest_to_json(self.forest, std::ptr::null_mut(), 0, &mut need) })?;
        let mut buf = vec![0u8; need];
        check(unsafe { dh_forest_to_json(self.forest, buf.as_mut_ptr() as *mut c_char, need, &mut need) })?;
        Ok(String::from_utf8_lossy(&buf).into_owned())
    }
    fn context(&self) -> *mut DhCtx {
        if self.ctx.get().is_null() {
            let device = std::env::var("DEPTHHEAD_CUDA_DEVICE").ok().and_then(|s| s.parse::<c_int>().ok()).unwrap_or(0);
            let mut c = std::ptr::null_mut();
            check(unsafe { dh_ctx_create(device, &mut c) }).expect("depthhead-cuda: no usable CUDA device (there is no CPU fallback)");
            self.ctx.set(c);
        }
        self.ctx.get()
    }
    /// the public fields may have been changed since the last call (prediction.rs:242,255)
    fn push_fields(&self) -> Result<(), Error> {
        unsafe {
            if dh_forest_get_stepwidth(self.forest) != self.stepwidth { check(dh_forest_set_stepwidth(self.forest, self.stepwidth))?; }
            if dh_forest_get_meanshift_iterations(self.forest) != self.meanshift_iterations {
                check(dh_forest_set_meanshift_iterations(self.forest, self.meanshift_iterations))?;
            }
        }
        Ok(())
    }

    /// Update sigma value used for mean shifting (prediction.rs:320-326): ignored if unchanged or <= 0
    pub fn update_sigma(&mut self, val: f32) { unsafe { dh_forest_set_sigma(self.forest, val); } }
    /// prediction.rs:329-331
    pub fn sigma(&self) -> f32 { unsafe { dh_forest_get_sigma(self.forest) } }

    /// prediction.rs:397-409.  `DepthImage` is contiguous row-major u16 (types.rs:10), so its
    /// buffer is passed as is.  The reference's signature is infallible and panics on degenerate
    /// input (prediction.rs:565,716); so does this one, with the library's message.
    pub fn predict_parameter_parallel(&self, img: Arc<DepthImage>, intrinsic: &IntrinsicMatrix,
                                      midp_guess: Option<[f32; 3]>, rot_guess: Option<[f64; 3]>) -> PredictionResult {
        self.push_fields().expect("depthhead-cuda: invalid stepwidth / meanshift_iterations");
        let mut out = DhResult::default();
        let mg = midp_guess.as_ref().map_or(std::ptr::null(), |g| g.as_ptr());
        let rg = rot_guess.as_ref().map_or(std::ptr::null(), |g| g.as_ptr());
        check(unsafe { dh_predict(self.context(), self.forest, img.as_ptr(), img.width(), img.height(), intrinsic.ptr(), mg, rg, &mut out) })
            .expect("depthhead-cuda: prediction failed");
        PredictionResult::from_c(&out)
    }
    /// prediction.rs:376-388: the single-core variant returns identical results (same leaves in
    /// tree order, all later accumulation sequential); on the GPU both are the same call
    pub fn predict_parameter(&self, img: Arc<DepthImage>, intrinsic: &IntrinsicMatrix,
                             midp_guess: Option<[f32; 3]>, rot_guess: Option<[f64; 3]>) -> PredictionResult {
        self.predict_parameter_parallel(img, intrinsic, midp_guess, rot_guess)
    }
    /// prediction.rs:343-367
    pub fn predict_parameter_from2dhough(&self, img: Arc<DepthImage>, intrinsic: &IntrinsicMatrix) -> PredictionResult {
        self.push_fields().expect("depthhead-cuda: invalid stepwidth");
        let mut out = DhResult::default();
        check(unsafe { dh_predict_from2dhough(self.context(), self.forest, img.as_ptr(), img.width(), img.height(), intrinsic.ptr(), &mut out) })
            .expect("depthhead-cuda: predict_parameter_from2dhough failed");
        PredictionResult::from_c(&out)
    }
    /// prediction.rs:760-845
    pub fn build_hough_image(&self, img: Arc<DepthImage>, intrinsic: &IntrinsicMatrix) -> ImageBuffer<Luma<u16>, Vec<u16>> {
        self.push_fields().expect("depthhead-cuda: invalid stepwidth");
        let mut buf = vec![0u16; (img.width() * img.height()) as usize];
        check(unsafe { dh_build_hough_image(self.context(), self.forest, img.as_ptr(), img.width(), img.height(), intrinsic.ptr(), buf.as_mut_ptr()) })
            .expect("depthhead-cuda: build_hough_image failed");
        ImageBuffer::from_raw(img.width(), img.height(), buf).unwrap()
    }
    /// prediction.rs:850-905
    pub fn predict_mask(&self, img: Arc<DepthImage>) -> ImageBuffer<Luma<u8>, Vec<u8>> {
        self.push_fields().expect("depthhead-cuda: invalid stepwidth");
        let mut buf = vec![0u8; (img.width() * img.height()) as usize];
        check(unsafe { dh_predict_mask(self.context(), self.forest, img.as_ptr(), img.width(), img.height(), buf.as_mut_ptr()) })
            .expect("depthhead-cuda: predict_mask failed");
        ImageBuffer::from_raw(img.width(), img.height(), buf).unwrap()
    }

    // ---- beyond the reference's surface: what a GPU is for
    /// n independent frames back to back, seeds None; results in frame order
    pub fn predict_batch(&self, frames: &[u16], n: u32, w: u32, h: u32, k: &IntrinsicMatrix) -> Result<Vec<DhResult>, Error> {
        assert_eq!(frames.len(), (n as usize) * (w as usize) * (h as usize));
        self.push_fields()?;
        let mut out = vec![DhResult::default(); n as usize];
        check(unsafe { dh_predict_batch(self.context(), self.forest, frames.as_ptr(), n, w, h, k.ptr(), 0 /* DH_DEPTH_HOST */, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// predict_parameter_parallel(img_i, &intrinsics[i], midp_guess[i], rot_guess[i]) for n independent
    /// frames back to back in one call (a camera and seeds per frame: trackers, multi-camera rigs,
    /// seeds from a detector); equal to calling predict_parameter_parallel frame by frame
    pub fn predict_frames(&self, frames: &[u16], n: u32, w: u32, h: u32, intrinsics: &[IntrinsicMatrix],
                          midp_guess: &[Option<[f32; 3]>], rot_guess: &[Option<[f64; 3]>]) -> Vec<PredictionResult> {
        assert_eq!(frames.len(), (n as usize) * (w as usize) * (h as usize));
        let args = frame_args(n, intrinsics, midp_guess, rot_guess);
        self.push_fields().expect("depthhead-cuda: invalid stepwidth / meanshift_iterations");
        let mut out = vec![DhResult::default(); n as usize];
        check(unsafe { dh_predict_frames(self.context(), self.forest, frames.as_ptr(), n, w, h, 0 /* DH_DEPTH_HOST */,
                                         args.as_ptr(), out.as_mut_ptr()) })
            .expect("depthhead-cuda: prediction failed");
        out.iter().map(PredictionResult::from_c).collect()
    }
    /// predict_mask of n independent frames back to back: masks [n][h][w] in frame order
    pub fn predict_mask_batch(&self, frames: &[u16], n: u32, w: u32, h: u32) -> Result<Vec<u8>, Error> {
        let px = (n as usize) * (w as usize) * (h as usize);
        assert_eq!(frames.len(), px);
        self.push_fields()?;
        let mut out = vec![0u8; px];
        check(unsafe { dh_predict_mask_batch(self.context(), self.forest, frames.as_ptr(), n, w, h, 0 /* DH_DEPTH_HOST */,
                                             out.as_mut_ptr(), 0) })?;
        Ok(out)
    }
    /// build_hough_image of n independent frames back to back: blurred vote images [n][h][w] in frame
    /// order (blur = false: the vote images before the blur)
    pub fn build_hough_image_batch(&self, frames: &[u16], n: u32, w: u32, h: u32, k: &IntrinsicMatrix, blur: bool)
                                   -> Result<Vec<u16>, Error> {
        let px = (n as usize) * (w as usize) * (h as usize);
        assert_eq!(frames.len(), px);
        self.push_fields()?;
        let mut out = vec![0u16; px];
        check(unsafe { dh_build_hough_image_batch(self.context(), self.forest, frames.as_ptr(), n, w, h, k.ptr(), 0 /* DH_DEPTH_HOST */,
                                                  blur as c_int, out.as_mut_ptr(), 0, std::ptr::null_mut()) })?;
        Ok(out)
    }
    /// predict_parameter_from2dhough of n independent frames back to back; results in frame order
    pub fn predict_parameter_from2dhough_batch(&self, frames: &[u16], n: u32, w: u32, h: u32, k: &IntrinsicMatrix)
                                               -> Result<Vec<DhResult>, Error> {
        assert_eq!(frames.len(), (n as usize) * (w as usize) * (h as usize));
        self.push_fields()?;
        let mut out = vec![DhResult::default(); n as usize];
        check(unsafe { dh_build_hough_image_batch(self.context(), self.forest, frames.as_ptr(), n, w, h, k.ptr(), 0 /* DH_DEPTH_HOST */,
                                                  1, std::ptr::null_mut(), 0, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// n_seq independent sequences of frames_per_seq frames each (sequence-major): frame t of every
    /// sequence is seeded with the pose of frame t - 1 exactly as examples/live_prediction.rs:75-88
    /// does (a centre seed only if its z exceeds min_seed_z, 500.0 there)
    pub fn predict_sequences(&self, frames: &[u16], n_seq: u32, frames_per_seq: u32, w: u32, h: u32, k: &IntrinsicMatrix,
                             min_seed_z: f32) -> Result<Vec<DhResult>, Error> {
        let n = (n_seq as usize) * (frames_per_seq as usize);
        assert_eq!(frames.len(), n * (w as usize) * (h as usize));
        self.push_fields()?;
        let mut out = vec![DhResult::default(); n];
        check(unsafe { dh_predict_sequences(self.context(), self.forest, frames.as_ptr(), n_seq, frames_per_seq, w, h, k.ptr(), 0, min_seed_z,
                                            out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// HoughLearning::learn (prediction.rs:145-234) on the GPU: `depth`/`mask` are n frames back to
    /// back, `k` one row-major 3x3 matrix per frame, `pos3d`/`rot` the annotated head pose per frame.
    pub fn learn(params: &DhTrainParams, n: u32, w: u32, h: u32, depth: &[u16], mask: &[u8], k: &[f32],
                 pos3d: &[f32], rot: &[f32]) -> Result<HoughPrediction, Error> {
        let device = std::env::var("DEPTHHEAD_CUDA_DEVICE").ok().and_then(|s| s.parse::<c_int>().ok()).unwrap_or(0);
        let (mut f, mut c) = (std::ptr::null_mut(), std::ptr::null_mut());
        check(unsafe { dh_ctx_create(device, &mut c) })?;
        if let Err(e) = check(unsafe { dh_train_learn(c, params, n, w, h, depth.as_ptr(), mask.as_ptr(), k.as_ptr(),
                                                      pos3d.as_ptr(), rot.as_ptr(), &mut f) }) {
            unsafe { dh_ctx_free(c) };
            return Err(e);
        }
        let hp = HoughPrediction::from_handle(f);
        hp.ctx.set(c);
        Ok(hp)
    }
}
impl Drop for HoughPrediction {
    fn drop(&mut self) {
        unsafe {
            if !self.ctx.get().is_null() { dh_ctx_free(self.ctx.get()); }
            dh_forest_free(self.forest);
        }
    }
}

/// one DhFrameArgs per frame; every slice has n entries
fn frame_args(n: u32, intrinsics: &[IntrinsicMatrix], midp_guess: &[Option<[f32; 3]>], rot_guess: &[Option<[f64; 3]>])
              -> Vec<DhFrameArgs> {
    let n = n as usize;
    assert!(intrinsics.len() == n && midp_guess.len() == n && rot_guess.len() == n, "one matrix and one pair of seeds per frame");
    (0..n).map(|i| {
        let mut a = DhFrameArgs::default();
        for r in 0..3 { a.k[3 * r..3 * r + 3].copy_from_slice(&intrinsics[i].0[r]); }
        if let Some(m) = midp_guess[i] { a.midp_guess = m; a.has_guess |= 1; }
        if let Some(r) = rot_guess[i] { a.rot_guess = r; a.has_guess |= 2; }
        a
    }).collect()
}

/// `#[derive(Deserialize)]` of the reference (prediction.rs:238): any serde deserializer works; the
/// document is captured as a `serde_json::Value`, written back as text and parsed by the library
/// (the flattening into device tables happens there, once).
impl<'de> Deserialize<'de> for HoughPrediction {
    fn deserialize<D: Deserializer<'de>>(deserializer: D) -> Result<HoughPrediction, D::Error> {
        let doc = serde_json::Value::deserialize(deserializer)?;
        let text = serde_json::to_string(&doc).map_err(D::Error::custom)?;
        HoughPrediction::from_json(&text).map_err(D::Error::custom)
    }
}
/// `#[derive(Serialize)]` of the reference: the library writes the document, serde carries it on.
impl Serialize for HoughPrediction {
    fn serialize<S: Serializer>(&self, serializer: S) -> Result<S::Ok, S::Error> {
        let text = self.to_json().map_err(S::Error::custom)?;
        let doc: serde_json::Value = serde_json::from_str(&text).map_err(S::Error::custom)?;
        doc.serialize(serializer)
    }
}

/// src/db_reader/biwi.rs: the three file formats on the way to the prediction path.
pub mod biwi {
    use super::*;
    /// Compressed depth files of one sequence, packed for the GPU: every file starts at a multiple
    /// of 16 bytes of `blob`; `offsets` has one more entry than there are files.
    pub struct PackedFiles { pub blob: Vec<u8>, pub offsets: Vec<u64>, pub width: u32, pub height: u32 }
    impl PackedFiles {
        pub fn new(files: &[Vec<u8>]) -> Result<Self, Error> {
            let (mut w, mut h) = (0u32, 0u32);
            if let Some(first) = files.first() {
                check(unsafe { dh_biwi_depth_dims(first.as_ptr(), first.len(), &mut w, &mut h) })?;
            }
            let (mut blob, mut offsets) = (Vec::new(), Vec::with_capacity(files.len() + 1));
            for f in files {
                offsets.push(blob.len() as u64);
                blob.extend_from_slice(f);
                while blob.len() % 16 != 0 { blob.push(0); }
            }
            offsets.push(blob.len() as u64);
            blob.extend_from_slice(&[0u8; 16]);
            Ok(PackedFiles { blob, offsets, width: w, height: h })
        }
    }
    /// read_cal (biwi.rs:27-60)
    pub fn read_cal(text: &str) -> Result<IntrinsicMatrix, Error> {
        let mut k = [[0f32; 3]; 3];
        check(unsafe { dh_biwi_parse_cal(text.as_ptr() as *const c_char, text.len(), k.as_mut_ptr() as *mut f32) })?;
        Ok(IntrinsicMatrix(k))
    }
    /// read_gt (biwi.rs:63-77): (pos3d, pos2d, rot)
    pub fn read_gt(file: &[u8], k: &IntrinsicMatrix) -> Result<([f32; 3], [f32; 2], [f32; 3]), Error> {
        let (mut p3, mut p2, mut rot) = ([0f32; 3], [0f32; 2], [0f32; 3]);
        check(unsafe { dh_biwi_parse_pose(file.as_ptr(), file.len(), k.0.as_ptr() as *const f32, p3.as_mut_ptr(),
                                          p2.as_mut_ptr(), rot.as_mut_ptr()) })?;
        Ok((p3, p2, rot))
    }
    impl HoughPrediction {
        /// read_depth (biwi.rs:81-103) for every file, expanded on the GPU: n images back to back
        pub fn read_depth(&self, files: &PackedFiles) -> Result<Vec<u16>, Error> {
            let n = (files.offsets.len() - 1) as u32;
            let mut out = vec![0u16; n as usize * files.width as usize * files.height as usize];
            check(unsafe { dh_biwi_decode_depth(self.context(), files.blob.as_ptr(), files.offsets.as_ptr(), n, files.width,
                                                files.height, out.as_mut_ptr(), 0 /* DH_DEPTH_HOST */) })?;
            Ok(out)
        }
        /// what examples/db_evaluate.rs:296 does per file — read_depth + predict_parameter(img, K, None,
        /// None) — for a whole sequence, the compressed bytes crossing PCIe
        pub fn predict_files(&self, files: &PackedFiles, k: &IntrinsicMatrix) -> Result<Vec<DhResult>, Error> {
            let n = (files.offsets.len() - 1) as u32;
            self.push_fields()?;
            let mut out = vec![DhResult::default(); n as usize];
            check(unsafe { dh_predict_batch_biwi(self.context(), self.forest, files.blob.as_ptr(), files.offsets.as_ptr(), n,
                                                 files.width, files.height, k.0.as_ptr() as *const f32, out.as_mut_ptr()) })?;
            Ok(out)
        }
        /// predict_files with the arguments of every file: a whole database, whose sequence folders
        /// each have their own depth.cal, in one call
        pub fn predict_files_frames(&self, files: &PackedFiles, intrinsics: &[IntrinsicMatrix], midp_guess: &[Option<[f32; 3]>],
                                    rot_guess: &[Option<[f64; 3]>]) -> Result<Vec<DhResult>, Error> {
            let n = (files.offsets.len() - 1) as u32;
            let args = frame_args(n, intrinsics, midp_guess, rot_guess);
            self.push_fields()?;
            let mut out = vec![DhResult::default(); n as usize];
            check(unsafe { dh_predict_frames_biwi(self.context(), self.forest, files.blob.as_ptr(), files.offsets.as_ptr(), n,
                                                  files.width, files.height, args.as_ptr(), out.as_mut_ptr()) })?;
            Ok(out)
        }
    }
}
