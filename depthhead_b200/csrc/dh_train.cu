// dh_train.cu — split scoring for Hough-forest TRAINING (SURVEY.md section 8 f4).
//
// The reference trains with stamm's `train_forest_parallel` (a crate that is not vendored), which
// calls back into depthhead's HoughTreeFunctions (src/hough/houghforest.rs:196-311).  What costs
// the time there is, per tree node, `impurity` (:250-295) of every candidate NodeParam: binarize
// (:185-193) every sample of the node, then entropy and the covariance determinants of the
// offsets and rotations on either side.  These kernels do that for all nodes of one tree level
// at once; the tree-growing loop above them is host code (depthhead_b200/train.py).
//
// Exactness: the covariance sums run over the samples IN SET ORDER with separate multiplications
// and additions, exactly estimate_mean_cov (meancov_estimation.rs:359-378) and Mat3::det
// (:339-343) in f64, so the per-side statistics equal the CPU restatement bit for bit; ln/exp of
// the final combination are taken on the host with the same libm the reference's f64::ln uses.
#include <cmath>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "dh_ctx.hpp"

namespace dh {

#define DH_CUDA_T(expr)                                                                                 \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            throw ModelError(DH_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));            \
    } while (0)

struct TrainSet {
    int device = 0;
    uint64_t n = 0;
    uint32_t sw = 0, sh = 0, rw = 0, rh = 0, bw = 0, bh = 0, bpitch = 0;
    uint32_t* box = nullptr;      // [n][bh][bpitch] box sums of every sample patch
    uint8_t* is_obj = nullptr;    // [n]
    double* off = nullptr;        // [n][3] offsets widened to f64 (`x.0[k] as f64`, houghforest.rs:268-269)
    double* rot = nullptr;        // [n][3]
    ~TrainSet() {
        cudaSetDevice(device);
        if (box) cudaFree(box);
        if (is_obj) cudaFree(is_obj);
        if (off) cudaFree(off);
        if (rot) cudaFree(rot);
    }
};

namespace dev {

struct Cand {  // one candidate NodeParam: box-table offsets of its two rectangles + threshold
    uint32_t tap1, tap2;
    double threshold;
};

// binarize (houghforest.rs:185-193) from two box sums: avg = sum as f64 / count as f64
__device__ __forceinline__ bool train_bit(const uint32_t* __restrict__ tbl, const Cand& c, double count) {
    const double a1 = __ddiv_rn((double)__ldg(tbl + c.tap1), count), a2 = __ddiv_rn((double)__ldg(tbl + c.tap2), count);
    return __dsub_rn(a1, a2) > c.threshold;
}

// One thread per (node, candidate).  Pass 1: side sizes, positives and the sums for the two
// means; pass 2: the two covariance matrices per side; then the four determinants.
__global__ void __launch_bounds__(128) train_score_kernel(const uint32_t* __restrict__ box, uint32_t tbl_words,
                                                          const uint8_t* __restrict__ is_obj, const double* __restrict__ off,
                                                          const double* __restrict__ rot, const uint32_t* __restrict__ idx,
                                                          const unsigned long long* __restrict__ node_off,
                                                          const Cand* __restrict__ cands, uint32_t m, double count,
                                                          dh_split_stats* __restrict__ out) {
    const uint32_t node = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    const Cand cd = cands[(size_t)node * m + c];
    const unsigned long long s0 = node_off[node], s1 = node_off[node + 1];
    uint32_t n[2] = {0, 0}, np[2] = {0, 0};
    double mo[2][3], mr[2][3];
    for (unsigned long long s = s0; s < s1; ++s) {
        const uint32_t j = __ldg(idx + s);
        const int side = train_bit(box + (size_t)j * tbl_words, cd, count) ? 1 : 0;
        ++n[side];
        if (__ldg(is_obj + j)) {
            const double* o = off + (size_t)j * 3;
            const double* r = rot + (size_t)j * 3;
            if (np[side] == 0) {  // mean starts from the first element (meancov_estimation.rs:363-366)
                for (int k = 0; k < 3; ++k) { mo[side][k] = __ldg(o + k); mr[side][k] = __ldg(r + k); }
            } else {
                for (int k = 0; k < 3; ++k) { mo[side][k] = __dadd_rn(mo[side][k], __ldg(o + k)); mr[side][k] = __dadd_rn(mr[side][k], __ldg(r + k)); }
            }
            ++np[side];
        }
    }
    for (int sd = 0; sd < 2; ++sd)
        if (np[sd])
            for (int k = 0; k < 3; ++k) {
                mo[sd][k] = __ddiv_rn(mo[sd][k], (double)np[sd]);
                mr[sd][k] = __ddiv_rn(mr[sd][k], (double)np[sd]);
            }
    // covariance: upper triangle (d[a]*d[b] == d[b]*d[a] exactly), entries 00 01 02 11 12 22
    double co[2][6], cr[2][6];
    uint32_t seen[2] = {0, 0};
    for (unsigned long long s = s0; s < s1; ++s) {
        const uint32_t j = __ldg(idx + s);
        if (!__ldg(is_obj + j)) continue;
        const int side = train_bit(box + (size_t)j * tbl_words, cd, count) ? 1 : 0;
        double d[3], e[3];
        for (int k = 0; k < 3; ++k) {
            d[k] = __dsub_rn(__ldg(off + (size_t)j * 3 + k), mo[side][k]);
            e[k] = __dsub_rn(__ldg(rot + (size_t)j * 3 + k), mr[side][k]);
        }
        const double po[6] = {__dmul_rn(d[0], d[0]), __dmul_rn(d[0], d[1]), __dmul_rn(d[0], d[2]),
                              __dmul_rn(d[1], d[1]), __dmul_rn(d[1], d[2]), __dmul_rn(d[2], d[2])};
        const double pr[6] = {__dmul_rn(e[0], e[0]), __dmul_rn(e[0], e[1]), __dmul_rn(e[0], e[2]),
                              __dmul_rn(e[1], e[1]), __dmul_rn(e[1], e[2]), __dmul_rn(e[2], e[2])};
        if (seen[side] == 0) {
            for (int k = 0; k < 6; ++k) { co[side][k] = po[k]; cr[side][k] = pr[k]; }
        } else {
            for (int k = 0; k < 6; ++k) { co[side][k] = __dadd_rn(co[side][k], po[k]); cr[side][k] = __dadd_rn(cr[side][k], pr[k]); }
        }
        ++seen[side];
    }
    dh_split_stats st;
    for (int sd = 0; sd < 2; ++sd) {
        st.n[sd] = n[sd];
        st.n_pos[sd] = np[sd];
        double det_o = __longlong_as_double(0x7ff8000000000000ll), det_r = det_o;
        if (np[sd]) {
            const double dn1 = (double)(np[sd] - 1u);  // n == 1: 0/0 = NaN entries, NaN determinant
            double a[6], b[6];
            for (int k = 0; k < 6; ++k) { a[k] = __ddiv_rn(co[sd][k], dn1); b[k] = __ddiv_rn(cr[sd][k], dn1); }
            // Mat3::det (meancov_estimation.rs:339-343) with m10 = m01, m20 = m02, m21 = m12:
            // m00*(m11*m22 - m12*m21) - m10*(m01*m22 - m02*m21) + m20*(m01*m12 - m02*m11)
            auto det = [](const double* q) {
                const double t0 = __dmul_rn(q[0], __dsub_rn(__dmul_rn(q[3], q[5]), __dmul_rn(q[4], q[4])));
                const double t1 = __dmul_rn(q[1], __dsub_rn(__dmul_rn(q[1], q[5]), __dmul_rn(q[2], q[4])));
                const double t2 = __dmul_rn(q[2], __dsub_rn(__dmul_rn(q[1], q[4]), __dmul_rn(q[2], q[3])));
                return __dadd_rn(__dsub_rn(t0, t1), t2);
            };
            det_o = det(a);
            det_r = det(b);
        }
        st.det_off[sd] = det_o;
        st.det_rot[sd] = det_r;
    }
    st.impurity = 0.0;
    out[(size_t)node * m + c] = st;
}

// bits of ONE chosen candidate per node over the node's samples
__global__ void __launch_bounds__(256) train_split_kernel(const uint32_t* __restrict__ box, uint32_t tbl_words,
                                                          const uint32_t* __restrict__ idx,
                                                          const unsigned long long* __restrict__ node_off,
                                                          const Cand* __restrict__ chosen, uint32_t n_nodes, double count,
                                                          uint8_t* __restrict__ bits) {
    const unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= node_off[n_nodes]) return;
    uint32_t lo = 0, hi = n_nodes;  // node of sample slot s: last k with node_off[k] <= s
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (node_off[mid] <= s) lo = mid; else hi = mid;
    }
    bits[s] = train_bit(box + (size_t)__ldg(idx + s) * tbl_words, chosen[lo], count) ? 1 : 0;
}

}  // namespace dev

// ---------------------------------------------------------------------------------------------- host
namespace {
template <typename T>
struct DevBuf {
    T* p = nullptr;
    explicit DevBuf(size_t n) { if (cudaMalloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T)) != cudaSuccess) { p = nullptr; throw ModelError(DH_E_CUDA, "cudaMalloc failed (training scratch)"); } }
    ~DevBuf() { if (p) cudaFree(p); }
};

// `ln!` (houghforest.rs:18-20)
inline double rs_ln(double x) { return x == 0.0 ? 0.0 : std::log(x); }

// impurity (houghforest.rs:250-295) from the per-side statistics; NaN where the reference itself
// aborts: an empty side (rel!(0, 0) is NaN and assert!(res.is_finite()) fires, :293) or a
// covariance determinant sum below -0.001 (unreachable!(), :281 — rounding of a rank-deficient
// covariance of widely spread samples can get there)
double impurity_from_stats(const dh_split_stats& s, uint64_t depth, double steepness, bool* unreachable) {
    if (s.n[0] == 0 || s.n[1] == 0) return std::numeric_limits<double>::quiet_NaN();
    auto entropy = [](uint32_t pos, uint32_t n) {
        const double prob = (double)pos / (double)n;
        return prob * rs_ln(prob) + (1.0 - prob) * rs_ln(1.0 - prob);
    };
    auto reglog = [&](int sd) {
        if (s.n_pos[sd] == 0) return 0.0;
        const double x = s.det_off[sd] + s.det_rot[sd];
        if (x > 0.0) return std::log(x);
        if (x < -0.001) *unreachable = true;  // houghforest.rs:281
        return 0.0;
    };
    const uint64_t count = (uint64_t)s.n[0] + s.n[1];
    const double lf = (double)s.n[0] / (double)count, rf = (double)s.n[1] / (double)count;
    const double impurity = -(lf * entropy(s.n_pos[0], s.n[0]) + rf * entropy(s.n_pos[1], s.n[1]));
    const double reg = lf * reglog(0) + rf * reglog(1);
    const double f = std::exp(-((double)depth / steepness));
    return impurity + (1.0 - f) * reg;
}

void make_cands(const TrainSet& ts, const int32_t* rects, const double* thr, size_t n, std::vector<dev::Cand>& out) {
    out.resize(n);
    for (size_t i = 0; i < n; ++i) {
        const int32_t* r = rects + i * 8;
        for (int k = 0; k < 2; ++k) {
            const int32_t x0 = r[k * 4], y0 = r[k * 4 + 1], x1 = r[k * 4 + 2], y1 = r[k * 4 + 3];
            if (x0 < 0 || y0 < 0 || x1 - x0 != (int32_t)ts.rw || y1 - y0 != (int32_t)ts.rh || x1 > (int32_t)ts.sw || y1 > (int32_t)ts.sh)
                throw ModelError(DH_E_ARG, "candidate " + std::to_string(i) + ": rectangle is not " + std::to_string(ts.rw) + "x" +
                                               std::to_string(ts.rh) + " inside the sub-image (this training set was built for one rectangle size)");
            (k ? out[i].tap2 : out[i].tap1) = (uint32_t)y0 * ts.bpitch + (uint32_t)x0;
        }
        out[i].threshold = thr[i];
    }
}
}  // namespace

TrainSet* Context::trainset_create(const uint16_t* patches, uint64_t n, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh,
                                   const uint8_t* is_object, const float* offsets, const double* rotations) {
    DH_CUDA_T(cudaSetDevice(device_));
    if (n == 0 || n > 0x7fffffffull) throw ModelError(DH_E_ARG, "training set must hold 1 .. 2^31-1 samples");
    // What box_image_kernel needs of a training table: sides of 1..128 inside the sub-image and
    // rw * rh <= 16383.  The prediction path's further limit on how many rectangles cover a patch
    // (box_image_supported) belongs to its background test, which training does not run.
    if (!rw || !rh || rw > sw || rh > sh || rw > 128u || rh > 128u || (uint64_t)rw * rh > 16383u)
        throw ModelError(DH_E_SHAPE, "feature rectangle size not supported by the box-sum tables: sides of 1 .. 128 inside the "
                                     "sub-image, rw * rh <= 16383 (see DESIGN.md)");
    std::unique_ptr<TrainSet> ts(new TrainSet());
    ts->device = device_;
    ts->n = n; ts->sw = sw; ts->sh = sh; ts->rw = rw; ts->rh = rh;
    ts->bw = sw - rw + 1; ts->bh = sh - rh + 1; ts->bpitch = (ts->bw + 3) & ~3u;
    DH_CUDA_T(cudaMalloc((void**)&ts->box, n * (size_t)ts->bh * ts->bpitch * sizeof(uint32_t)));
    DH_CUDA_T(cudaMalloc((void**)&ts->is_obj, n));
    DH_CUDA_T(cudaMalloc((void**)&ts->off, n * 3 * sizeof(double)));
    DH_CUDA_T(cudaMalloc((void**)&ts->rot, n * 3 * sizeof(double)));
    std::vector<double> off64(n * 3);
    for (size_t i = 0; i < n * 3; ++i) off64[i] = (double)offsets[i];
    DH_CUDA_T(cudaMemcpyAsync(ts->is_obj, is_object, n, cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(ts->off, off64.data(), n * 3 * sizeof(double), cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(ts->rot, rotations, n * 3 * sizeof(double), cudaMemcpyHostToDevice, stream_));
    // box-sum table of every patch: the prediction path's front-end kernel with frame = patch
    const size_t patch_px = (size_t)sw * sh;
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(n, (256ull << 20) / (patch_px * 2)));
    DevBuf<uint16_t> d_px(chunk * patch_px);
    Geometry g{};
    g.w = sw; g.h = sh; g.sw = sw; g.sh = sh; g.rw = rw; g.rh = rh;
    g.box_w = ts->bw; g.box_h = ts->bh; g.box_pitch = ts->bpitch;
    for (uint64_t f0 = 0; f0 < n; f0 += chunk) {
        const uint64_t nc = std::min(chunk, n - f0);
        DH_CUDA_T(cudaMemcpyAsync(d_px.p, patches + f0 * patch_px, nc * patch_px * sizeof(uint16_t), cudaMemcpyHostToDevice, stream_));
        FrameBuffers b{};
        b.depth = d_px.p;
        b.box = ts->box + f0 * (size_t)ts->bh * ts->bpitch;
        launch_box_image(b, g, (uint32_t)nc, n_sms_, box_whole_, box_bands_, stream_);
        DH_CUDA_T(cudaGetLastError());
        DH_CUDA_T(cudaStreamSynchronize(stream_));
    }
    return ts.release();
}

void Context::train_score_level(const TrainSet& ts, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                                const int32_t* cand_rects, const double* cand_thr, uint32_t m, uint64_t depth, double steepness,
                                dh_split_stats* out) {
    DH_CUDA_T(cudaSetDevice(device_));
    if (ts.device != device_) throw ModelError(DH_E_ARG, "the training set lives on another GPU than this context");
    if (n_nodes == 0 || m == 0) return;
    const uint64_t total = node_off[n_nodes];
    for (uint32_t k = 0; k < n_nodes; ++k)
        if (node_off[k + 1] < node_off[k]) throw ModelError(DH_E_ARG, "dh_train_score_level: node_off is not monotone");
    for (uint64_t s = 0; s < total; ++s)
        if (sample_idx[s] >= ts.n) throw ModelError(DH_E_ARG, "sample index out of range");
    std::vector<dev::Cand> cands;
    make_cands(ts, cand_rects, cand_thr, (size_t)n_nodes * m, cands);
    DevBuf<uint32_t> d_idx(total);
    DevBuf<unsigned long long> d_off(n_nodes + 1);
    DevBuf<dev::Cand> d_c(cands.size());
    DevBuf<dh_split_stats> d_out(cands.size());
    DH_CUDA_T(cudaMemcpyAsync(d_idx.p, sample_idx, total * sizeof(uint32_t), cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(d_off.p, node_off, (n_nodes + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(d_c.p, cands.data(), cands.size() * sizeof(dev::Cand), cudaMemcpyHostToDevice, stream_));
    // the node is blockIdx.y, at most 65535 per launch: wider levels go in slices of nodes (node_off
    // holds offsets into the whole sample_idx, so a slice only moves the node_off, cands and out bases)
    constexpr uint32_t kMaxNodesPerLaunch = 65535u;
    for (uint32_t k0 = 0; k0 < n_nodes; k0 += kMaxNodesPerLaunch) {
        const uint32_t nk = std::min(kMaxNodesPerLaunch, n_nodes - k0);
        dim3 gr((m + 127) / 128, nk);
        dev::train_score_kernel<<<gr, 128, 0, stream_>>>(ts.box, ts.bh * ts.bpitch, ts.is_obj, ts.off, ts.rot, d_idx.p, d_off.p + k0,
                                                         d_c.p + (size_t)k0 * m, m, (double)((uint64_t)ts.rw * ts.rh),
                                                         d_out.p + (size_t)k0 * m);
        DH_CUDA_T(cudaGetLastError());
    }
    DH_CUDA_T(cudaMemcpyAsync(out, d_out.p, cands.size() * sizeof(dh_split_stats), cudaMemcpyDeviceToHost, stream_));
    DH_CUDA_T(cudaStreamSynchronize(stream_));
    for (size_t i = 0; i < cands.size(); ++i) {
        bool unreachable = false;
        out[i].impurity = impurity_from_stats(out[i], depth, steepness, &unreachable);
        if (unreachable) out[i].impurity = std::numeric_limits<double>::quiet_NaN();
    }
}

void Context::train_split_level(const TrainSet& ts, const uint32_t* sample_idx, const uint64_t* node_off, uint32_t n_nodes,
                                const int32_t* rects, const double* thr, uint8_t* bits) {
    DH_CUDA_T(cudaSetDevice(device_));
    if (ts.device != device_) throw ModelError(DH_E_ARG, "the training set lives on another GPU than this context");
    if (n_nodes == 0) return;
    const uint64_t total = node_off[n_nodes];
    for (uint32_t k = 0; k < n_nodes; ++k)
        if (node_off[k + 1] < node_off[k]) throw ModelError(DH_E_ARG, "dh_train_split_level: node_off is not monotone");
    if (total == 0) return;
    for (uint64_t s = 0; s < total; ++s)
        if (sample_idx[s] >= ts.n) throw ModelError(DH_E_ARG, "sample index out of range");
    std::vector<dev::Cand> cands;
    make_cands(ts, rects, thr, n_nodes, cands);
    DevBuf<uint32_t> d_idx(total);
    DevBuf<unsigned long long> d_off(n_nodes + 1);
    DevBuf<dev::Cand> d_c(cands.size());
    DevBuf<uint8_t> d_bits(total);
    DH_CUDA_T(cudaMemcpyAsync(d_idx.p, sample_idx, total * sizeof(uint32_t), cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(d_off.p, node_off, (n_nodes + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, stream_));
    DH_CUDA_T(cudaMemcpyAsync(d_c.p, cands.data(), cands.size() * sizeof(dev::Cand), cudaMemcpyHostToDevice, stream_));
    dev::train_split_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream_>>>(ts.box, ts.bh * ts.bpitch, d_idx.p, d_off.p, d_c.p, n_nodes,
                                                                                 (double)((uint64_t)ts.rw * ts.rh), d_bits.p);
    DH_CUDA_T(cudaGetLastError());
    DH_CUDA_T(cudaMemcpyAsync(bits, d_bits.p, total, cudaMemcpyDeviceToHost, stream_));
    DH_CUDA_T(cudaStreamSynchronize(stream_));
}

// ---------------------------------------------------------------------------------------------- tree growing
// Stand-in for stamm 0.2.0's `train_forest_parallel` (not vendored), stated in DESIGN.md section 9 and
// mirrored line by line by depthhead_b200/train.py: counter-based random numbers, subsets drawn
// without replacement in drawn order, breadth-first growth from depth 0, candidates on which the
// reference's impurity aborts are skipped, the smallest impurity wins (first of equals), samples
// keep their order through a split, children[bit] receives the side with binarize == bit.
namespace {
struct CounterRng {  // draw k = splitmix64(seed + k * golden), k = 1, 2, ..; uniform [0,1) = top 53 bits
    uint64_t seed, k = 0;
    explicit CounterRng(uint64_t s) : seed(s) {}
    double next() {
        ++k;
        uint64_t z = seed + k * 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        return (double)(z >> 11) * (1.0 / 9007199254740992.0);
    }
    std::vector<uint32_t> permutation(uint64_t n) {  // Fisher-Yates from the back
        std::vector<uint32_t> a(n);
        for (uint64_t i = 0; i < n; ++i) a[i] = (uint32_t)i;
        for (uint64_t i = n; i-- > 1;) {
            const uint64_t j = (uint64_t)(next() * (double)(i + 1));
            std::swap(a[i], a[j]);
        }
        return a;
    }
};

// Rect::scale_and_replace (types.rs:82-91) of Rect(0, 0, w, h): x0, y0, x1, y1
void scale_and_replace(uint32_t w, uint32_t h, double scale, double rx, double ry, int32_t out[4]) {
    if (scale > 1.0) { out[0] = 0; out[1] = 0; out[2] = (int32_t)w; out[3] = (int32_t)h; return; }
    const double nw = (double)w * scale, nh = (double)h * scale;
    const double nx = 0.0 + rx * ((double)w - nw), ny = 0.0 + ry * ((double)h - nh);
    const uint32_t x = (uint32_t)nx, y = (uint32_t)ny;  // `as u32`: truncation (values are in range)
    out[0] = (int32_t)x; out[1] = (int32_t)y; out[2] = (int32_t)(x + (uint32_t)nw); out[3] = (int32_t)(y + (uint32_t)nh);
}
}  // namespace

HostForest* Context::train_forest(const dh_train_params& tp, const uint16_t* patches, uint64_t n, const uint8_t* is_object,
                                  const float* offsets, const double* rotations) {
    // HoughTreeFunctions::new returns None for these (houghforest.rs:143-147); a factor of 0 makes
    // random_subrect_iterator(..).unwrap() panic (types.rs:106-110)
    const double sc = tp.subrect_feature_scale;
    if (!(sc > 0.0) || sc > 1.0 || tp.features_per_node == 0 || !(tp.steepness > 0.0))
        throw ModelError(DH_E_ARG, "Bad parameter for learning Houghforest");
    if (tp.n_trees == 0 || tp.subimage_width == 0 || tp.subimage_height == 0 || tp.stepwidth == 0)
        throw ModelError(DH_E_ARG, "dh_train_forest: zero trees / sub-image / stepwidth");
    const uint32_t sw = tp.subimage_width, sh = tp.subimage_height;
    const uint32_t rw = (uint32_t)((double)sw * sc), rh = (uint32_t)((double)sh * sc);
    std::unique_ptr<TrainSet, void (*)(TrainSet*)> ts(trainset_create(patches, n, sw, sh, rw, rh, is_object, offsets, rotations), trainset_free);
    CounterRng rng(tp.seed);
    const uint32_t M = tp.features_per_node;

    RawForest raw;
    raw.stepwidth = tp.stepwidth; raw.subimage_width = sw; raw.subimage_height = sh;
    raw.meanshift_iterations = 20;  // prediction.rs:232
    raw.gaussian_sigma = tp.gaussian_sigma;
    raw.n_trees = (int32_t)tp.n_trees;

    struct Slot { int32_t rect[8]; double thr; int32_t child[2]; bool is_node = false; int64_t leaf = -1; };
    for (uint32_t t = 0; t < tp.n_trees; ++t) {
        std::vector<uint32_t> subset = rng.permutation(n);
        if (subset.size() > tp.subset_per_tree) subset.resize(tp.subset_per_tree);
        std::vector<Slot> slots(1);
        std::vector<std::pair<uint32_t, std::vector<uint32_t>>> frontier;
        frontier.emplace_back(0u, std::move(subset));
        std::vector<std::pair<uint32_t, std::vector<uint32_t>>> leaf_sets;  // (slot, samples) in creation order
        for (uint64_t depth = 0; !frontier.empty(); ++depth) {
            // early_stop (houghforest.rs:302-311), else param_set (:227-246): five draws per candidate
            std::vector<size_t> split;            // indices into frontier
            std::vector<int32_t> cand_rects;
            std::vector<double> cand_thr;
            for (size_t f = 0; f < frontier.size(); ++f) {
                const std::vector<uint32_t>& idx = frontier[f].second;
                bool any_obj = false;
                for (uint32_t j : idx) any_obj = any_obj || is_object[j];
                if (!any_obj || depth >= tp.max_depth || idx.size() < tp.min_subset_size) continue;
                split.push_back(f);
                for (uint32_t c = 0; c < M; ++c) {
                    const double u0 = rng.next(), u1 = rng.next(), u2 = rng.next(), u3 = rng.next(), u4 = rng.next();
                    int32_t r[8];
                    scale_and_replace(sw, sh, sc, u0, u1, r);
                    scale_and_replace(sw, sh, sc, u2, u3, r + 4);
                    cand_rects.insert(cand_rects.end(), r, r + 8);
                    cand_thr.push_back(-256.0 + u4 * (256.0 - -256.0));
                }
            }
            std::vector<int> chosen(frontier.size(), -1);  // candidate index per frontier node
            if (!split.empty()) {
                std::vector<uint32_t> all_idx;
                std::vector<uint64_t> node_off(1, 0);
                for (size_t f : split) {
                    all_idx.insert(all_idx.end(), frontier[f].second.begin(), frontier[f].second.end());
                    node_off.push_back(all_idx.size());
                }
                std::vector<dh_split_stats> st(split.size() * (size_t)M);
                train_score_level(*ts, all_idx.data(), node_off.data(), (uint32_t)split.size(), cand_rects.data(), cand_thr.data(), M,
                                  depth, tp.steepness, st.data());
                std::vector<size_t> deciding;       // positions in `split` that found a candidate
                std::vector<int32_t> ch_rects;
                std::vector<double> ch_thr;
                for (size_t k = 0; k < split.size(); ++k) {
                    int best = -1;
                    for (uint32_t c = 0; c < M; ++c) {
                        const double v = st[k * M + c].impurity;
                        if (v != v) continue;                                   // the reference aborts on this candidate
                        if (best < 0 || v < st[k * M + (size_t)best].impurity) best = (int)c;  // smallest, first of equals
                    }
                    if (best < 0) continue;
                    chosen[split[k]] = best;
                    deciding.push_back(k);
                    ch_rects.insert(ch_rects.end(), cand_rects.begin() + (k * M + (size_t)best) * 8, cand_rects.begin() + (k * M + (size_t)best + 1) * 8);
                    ch_thr.push_back(cand_thr[k * M + (size_t)best]);
                }
                if (!deciding.empty()) {
                    std::vector<uint32_t> sub_idx;
                    std::vector<uint64_t> sub_off(1, 0);
                    for (size_t k : deciding) {
                        const auto& v = frontier[split[k]].second;
                        sub_idx.insert(sub_idx.end(), v.begin(), v.end());
                        sub_off.push_back(sub_idx.size());
                    }
                    std::vector<uint8_t> bits(sub_idx.size());
                    train_split_level(*ts, sub_idx.data(), sub_off.data(), (uint32_t)deciding.size(), ch_rects.data(), ch_thr.data(), bits.data());
                    std::vector<std::pair<uint32_t, std::vector<uint32_t>>> next;
                    // children are created in frontier order, like the Python mirror (slots numbered as they appear)
                    size_t d = 0;
                    std::vector<std::pair<size_t, size_t>> where(frontier.size(), {SIZE_MAX, 0});  // frontier node -> position in deciding
                    for (size_t q = 0; q < deciding.size(); ++q) where[split[deciding[q]]] = {q, 0};
                    for (size_t f = 0; f < frontier.size(); ++f) {
                        if (chosen[f] < 0) { leaf_sets.emplace_back(frontier[f].first, std::move(frontier[f].second)); continue; }
                        const size_t q = where[f].first;
                        const uint32_t slot = frontier[f].first;
                        std::vector<uint32_t> side[2];
                        const auto& v = frontier[f].second;
                        for (size_t i = 0; i < v.size(); ++i) side[bits[sub_off[q] + i] ? 1 : 0].push_back(v[i]);
                        slots[slot].is_node = true;
                        std::memcpy(slots[slot].rect, &ch_rects[q * 8], sizeof(int32_t) * 8);
                        slots[slot].thr = ch_thr[q];
                        for (int b = 0; b < 2; ++b) {
                            slots[slot].child[b] = (int32_t)slots.size();
                            next.emplace_back((uint32_t)slots.size(), std::move(side[b]));
                            slots.emplace_back();
                        }
                        (void)d;
                    }
                    frontier.swap(next);
                    continue;
                }
            }
            for (auto& fr : frontier) leaf_sets.emplace_back(fr.first, std::move(fr.second));
            frontier.clear();
        }
        // leaves in creation order; slots that became leaves drop out of the node table
        for (size_t i = 0; i < leaf_sets.size(); ++i) slots[leaf_sets[i].first].leaf = (int64_t)i;
        std::vector<int32_t> node_of(slots.size(), -1);
        int32_t nn = 0;
        for (size_t s2 = 0; s2 < slots.size(); ++s2)
            if (slots[s2].is_node) node_of[s2] = nn++;
        for (size_t s2 = 0; s2 < slots.size(); ++s2) {
            if (!slots[s2].is_node) continue;
            raw.rects.insert(raw.rects.end(), slots[s2].rect, slots[s2].rect + 8);
            raw.threshold.push_back(slots[s2].thr);
            for (int b = 0; b < 2; ++b) {
                const int32_t c = slots[s2].child[b];
                raw.child.push_back(slots[(size_t)c].is_node ? node_of[(size_t)c] : ~(int32_t)slots[(size_t)c].leaf);
            }
        }
        // comp_leaf_data (houghforest.rs:204-225)
        for (auto& ls : leaf_sets) {
            uint64_t pos = 0;
            for (uint32_t j : ls.second)
                if (is_object[j]) {
                    ++pos;
                    raw.offsets.insert(raw.offsets.end(), offsets + (size_t)j * 3, offsets + (size_t)j * 3 + 3);
                    raw.rotations.insert(raw.rotations.end(), rotations + (size_t)j * 3, rotations + (size_t)j * 3 + 3);
                }
            raw.prob.push_back((double)pos / (double)ls.second.size());
            raw.vote_off.push_back((int64_t)(raw.offsets.size() / 3));
        }
        raw.tree_node_off.push_back((int64_t)raw.threshold.size());
        raw.tree_leaf_off.push_back((int64_t)raw.prob.size());
    }
    HostForest* hf = flatten_forest(raw);
    hf->fn_min_subrect_factor = hf->fn_max_subrect_factor = sc;
    hf->fn_steepness = tp.steepness;
    hf->fn_number_of_gen_features = M;
    hf->fn_max_depth = tp.max_depth;
    hf->fn_min_subset_size = tp.min_subset_size;
    return hf;
}

// HoughLearning::learn (prediction.rs:145-234): per annotated frame, every non-background window
// with its truth; 20 negatives then 20 positives per frame after a random permutation; one more
// permutation of the whole set; then the trees.  Random numbers: CounterRng(seed) for the sample
// selection, CounterRng(seed + 1) for the trees (the Python mirror does the same).
HostForest* Context::train_learn(const dh_train_params& tp, uint32_t n_frames, uint32_t w, uint32_t h, const uint16_t* depth,
                                 const uint8_t* mask, const float* K, const float* pos3d, const float* rot) {
    const uint32_t sw = tp.subimage_width, sh = tp.subimage_height, step = tp.stepwidth;
    if (!sw || !sh || !step) throw ModelError(DH_E_ARG, "dh_train_learn: zero sub-image / stepwidth");
    if (w < sw || h < sh) throw ModelError(DH_E_SHAPE, "image smaller than the sub-image (the reference underflows u32 at types.rs:371-373)");
    const uint32_t left_w = sw / 2, left_h = sh / 2, right_w = sw - left_w, right_h = sh - left_h;  // types.rs:365-368
    CounterRng rng(tp.seed);
    std::vector<uint16_t> patches;
    std::vector<uint8_t> is_obj;
    std::vector<float> offs;
    std::vector<double> rots;
    std::vector<uint32_t> nz((size_t)(w + 1) * (h + 1));
    struct Cand { uint32_t x, y; };
    for (uint32_t f = 0; f < n_frames; ++f) {
        const uint16_t* d = depth + (size_t)f * w * h;
        const uint8_t* m = mask + (size_t)f * w * h;
        // count of non-zero pixels: average_value_in_rect(whole window) > 0.0 <=> any non-zero pixel (prediction.rs:189-190)
        std::fill(nz.begin(), nz.begin() + (w + 1), 0u);
        for (uint32_t y = 0; y < h; ++y) {
            uint32_t row = 0;
            nz[(size_t)(y + 1) * (w + 1)] = 0;
            for (uint32_t x = 0; x < w; ++x) {
                row += d[(size_t)y * w + x] != 0;
                nz[(size_t)(y + 1) * (w + 1) + x + 1] = nz[(size_t)y * (w + 1) + x + 1] + row;
            }
        }
        std::vector<Cand> neg, pos;
        for (uint32_t y = left_h; y < h - right_h; y += step)          // iterate_subimage, types.rs:369-383
            for (uint32_t x = left_w; x < w - right_w; x += step) {
                const uint32_t x0 = x - left_w, y0 = y - left_h;
                const uint32_t cnt = nz[(size_t)(y0 + sh) * (w + 1) + x0 + sw] - nz[(size_t)y0 * (w + 1) + x0 + sw] -
                                     nz[(size_t)(y0 + sh) * (w + 1) + x0] + nz[(size_t)y0 * (w + 1) + x0];
                if (!cnt) continue;
                (m[(size_t)y * w + x] ? pos : neg).push_back(Cand{x, y});   // mask[(x, y)], prediction.rs:191
            }
        float inv[9];
        mat3_inverse_f32(K + (size_t)f * 9, inv);
        const std::vector<Cand>* parts[2] = {&neg, &pos};                 // negatives first (prediction.rs:222-226)
        for (int part = 0; part < 2; ++part) {
            const std::vector<Cand>& v = *parts[part];
            const std::vector<uint32_t> perm = rng.permutation(v.size());  // rand_perm, prediction.rs:216-217
            for (size_t k = 0; k < perm.size() && k < 20; ++k) {
                const Cand c = v[perm[k]];
                const uint32_t x0 = c.x - left_w, y0 = c.y - left_h;
                for (uint32_t yy = 0; yy < sh; ++yy)                        // to_cropped_subimage
                    patches.insert(patches.end(), d + (size_t)(y0 + yy) * w + x0, d + (size_t)(y0 + yy) * w + x0 + sw);
                is_obj.push_back(part ? 1 : 0);
                // img_to_space_coord (types.rs:432-445), f32, products and sums unfused; offset = vec3 - mid (prediction.rs:196-198)
                const float xf = (float)c.x, yf = (float)c.y, z = (float)d[(size_t)c.y * w + c.x];
                float r[3];
                for (int j = 0; j < 3; ++j) {
                    volatile float t = xf * inv[j * 3 + 0];
                    volatile float u = yf * inv[j * 3 + 1];
                    t = t + u;
                    u = 1.0f * inv[j * 3 + 2];
                    t = t + u;
                    r[j] = t;
                }
                const float cc = z / r[2];
                for (int j = 0; j < 3; ++j) {
                    volatile float pj = r[j] * cc;
                    offs.push_back(pj - pos3d[(size_t)f * 3 + j]);
                    rots.push_back((double)rot[(size_t)f * 3 + j]);    // rot[k] as f64, prediction.rs:176
                }
            }
        }
    }
    const uint64_t n = is_obj.size();
    if (!n) throw ModelError(DH_E_ARG, "dh_train_learn: no training samples (every window is background)");
    const std::vector<uint32_t> perm = rng.permutation(n);                // rand_perm(train_ref), prediction.rs:229
    const size_t px = (size_t)sw * sh;
    std::vector<uint16_t> p2(patches.size());
    std::vector<uint8_t> o2(n);
    std::vector<float> f2(n * 3);
    std::vector<double> r2(n * 3);
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t s2 = perm[i];
        std::memcpy(&p2[i * px], &patches[(size_t)s2 * px], px * sizeof(uint16_t));
        o2[i] = is_obj[s2];
        for (int j = 0; j < 3; ++j) { f2[i * 3 + j] = offs[(size_t)s2 * 3 + j]; r2[i * 3 + j] = rots[(size_t)s2 * 3 + j]; }
    }
    dh_train_params t2 = tp;
    t2.seed = tp.seed + 1;
    return train_forest(t2, p2.data(), n, o2.data(), f2.data(), r2.data());
}

void trainset_free(TrainSet* t) { delete t; }

}  // namespace dh
