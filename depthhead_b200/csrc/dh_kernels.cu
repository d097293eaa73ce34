// dh_kernels.cu — hand-written sm_100a kernels for depthhead's Hough-forest prediction path.
//
// Pipeline per chunk of frames (reference: src/hough/prediction.rs:421-753):
//   K1  box_image_kernel         u16 depth -> u32 box-sum image B[y][x] = sum of the rw x rh rectangle at
//                                (x, y), for forests whose feature rectangles all have one size (what the
//                                reference's trainer produces); sat_band_* / sat_rows / sat_cols: the general
//                                summed-area table for forests with mixed rectangle sizes
//   K2  traverse_kernel          TMA-staged tile of B (or of the SAT) in shared memory; one thread per
//                                patch x tree walks root->leaf (houghforest.rs:185-193, types.rs:317-339)
//   K3a patch_gate_kernel        0.7 gate of every patch from the 8-bit probability codes its leaf words carry
//                                (ordered f64 prob sum only where the codes cannot decide), back-projection,
//                                gated-patch list (prediction.rs:551-554,582-584)
//   K3b gate_coarse_kernel       the two coarse seed grids from slices of the gated-patch list
//                                (prediction.rs:590-595,630-636,661-675); <false, .>: gate and grids in one kernel
//   K4a seed_kernel              arg-max seeds (prediction.rs:694-752, 437-460)
//   K4b box_build_kernel         dense local cubes of the SparseArray3D<u32> accumulators
//                                (meanshift.rs:14-68, prediction.rs:635,667)
//   K4c meanshift_kernel         mean-shift in reference accumulation order (meanshift.rs:328-407), one CTA
//                                per accumulator; rebuilds its cube around positions that drift out of it
//   K5  leaf_gate_kernel         estimate_mean_cov traces + valtoadd per leaf, once per model
//                                (meancov_estimation.rs:359-378, prediction.rs:594-600,643)
//   +   mask_kernel (and track_mask_kernel, its writer for scattered frames), hough_image_kernel
//       (prediction.rs:850-905, 760-841), biwi_decode_kernel
//       (db_reader/biwi.rs:81-103); training's split scoring lives in dh_train.cu
//
// Exactness rules (SURVEY Appendix A): float->int is truncation (cvt.rzi, saturating, NaN->0 ==
// Rust `as`); no FMA contraction anywhere a float feeds a truncation or comparison (explicit
// __f*_rn / __d*_rn intrinsics, and the file is compiled with -fmad=false); vote sums are u32
// atomics (order independent, wrap like a release build).
//
// Summed-area table: S[y][x] = sum of pixels with x'<x, y'<y, in u32 with wrap-around.  Any
// rectangle whose true sum is < 2^32 (255*255*65535 < 2^32) is recovered exactly by the four-tap
// difference in modular arithmetic, and (double)sum/(double)count then equals the reference's
// naive loop bit for bit (types.rs:338).
#include "dh_kernels.cuh"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>

namespace dh {

namespace dev {

// ---------------------------------------------------------------- small device helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// IntrinsicMatrix::img_to_space_coord (types.rs:432-445) with Mat3*Vec3 of
// meancov_estimation.rs:201-216: tmp = v0*m[j][0]; tmp = tmp + v1*m[j][1]; tmp = tmp + v2*m[j][2].
__device__ __forceinline__ void img_to_space(const float* Kinv, float x, float y, float z, float out[3]) {
    float r[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        float t = __fmul_rn(x, Kinv[j * 3 + 0]);
        t = __fadd_rn(t, __fmul_rn(y, Kinv[j * 3 + 1]));
        t = __fadd_rn(t, __fmul_rn(1.0f, Kinv[j * 3 + 2]));
        r[j] = t;
    }
    const float c = __fdiv_rn(z, r[2]);
    out[0] = __fmul_rn(r[0], c);
    out[1] = __fmul_rn(r[1], c);
    out[2] = __fmul_rn(r[2], c);
}
// IntrinsicMatrix::space_to_img_coord (types.rs:424-428)
__device__ __forceinline__ void space_to_img(const float* K, const float p[3], float out[2]) {
    float r[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        float t = __fmul_rn(p[0], K[j * 3 + 0]);
        t = __fadd_rn(t, __fmul_rn(p[1], K[j * 3 + 1]));
        t = __fadd_rn(t, __fmul_rn(p[2], K[j * 3 + 2]));
        r[j] = t;
    }
    out[0] = __fdiv_rn(r[0], r[2]);
    out[1] = __fdiv_rn(r[1], r[2]);
}

// ================================================================ K1: summed-area table
// Row pass: exclusive prefix sums of one image row into S[y+1][0..w].  One warp per row,
// 8 pixels per lane per step (one 16-byte load), warp-shuffle scan of the lane totals.
constexpr int kSatRowWarps = 8;
__global__ void __launch_bounds__(kSatRowWarps * 32) sat_rows_kernel(const uint16_t* __restrict__ depth,
                                                                      uint32_t* __restrict__ sat, uint32_t w,
                                                                      uint32_t h, uint32_t pitch) {
    const uint32_t frame = blockIdx.y;
    const uint32_t y = blockIdx.x * kSatRowWarps + (threadIdx.x >> 5);
    if (y >= h) return;
    const uint32_t lane = threadIdx.x & 31;
    const uint16_t* row = depth + ((size_t)frame * h + y) * w;
    uint32_t* out = sat + ((size_t)frame * (h + 1) + (y + 1)) * pitch;
    const bool vec_ok = ((w & 7u) == 0u) && ((reinterpret_cast<uintptr_t>(row) & 15u) == 0u);
    uint32_t carry = 0;
    for (uint32_t seg = 0; seg <= w; seg += 256) {  // positions 0..w inclusive
        const uint32_t x = seg + lane * 8;
        uint32_t v[8];
        if (vec_ok && x + 8 <= w) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + x));
            v[0] = q.x & 0xffffu; v[1] = q.x >> 16; v[2] = q.y & 0xffffu; v[3] = q.y >> 16;
            v[4] = q.z & 0xffffu; v[5] = q.z >> 16; v[6] = q.w & 0xffffu; v[7] = q.w >> 16;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = (x + j < w) ? (uint32_t)__ldg(row + x + j) : 0u;
        }
        uint32_t e[8];
        uint32_t tot = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            e[j] = tot;
            tot += v[j];
        }
        uint32_t incl = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += n;
        }
        const uint32_t base = carry + incl - tot;
        if (x + 7 <= w) {
            uint4 a = make_uint4(base + e[0], base + e[1], base + e[2], base + e[3]);
            uint4 b = make_uint4(base + e[4], base + e[5], base + e[6], base + e[7]);
            *reinterpret_cast<uint4*>(out + x) = a;
            *reinterpret_cast<uint4*>(out + x + 4) = b;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (x + j <= w) out[x + j] = base + e[j];
        }
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// Column pass: in-place inclusive scan down every column (rows 1..h; row 0 stays zero).
// One thread per column, 8 independent loads in flight per thread.
__global__ void __launch_bounds__(128) sat_cols_kernel(uint32_t* __restrict__ sat, uint32_t w, uint32_t h,
                                                        uint32_t pitch) {
    const uint32_t frame = blockIdx.y;
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > w) return;
    uint32_t* col = sat + (size_t)frame * (h + 1) * pitch + pitch + c;  // row 1
    uint32_t acc = 0;
    uint32_t y = 0;
    for (; y + 8 <= h; y += 8) {
        uint32_t v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = col[(size_t)(y + j) * pitch];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            acc += v[j];
            col[(size_t)(y + j) * pitch] = acc;
        }
    }
    for (; y < h; ++y) {
        acc += col[(size_t)y * pitch];
        col[(size_t)y * pitch] = acc;
    }
}

// ---------------------------------------------------------------- banded single-pass variant
// For images up to 1023 pixels wide the table is produced with two reads of the depth and ONE
// write of the table (the two-pass variant above reads and writes the table twice): the frame is cut into bands of kSatBandRows
// rows.  Pass A: per band, the column sums of its rows and their exclusive scan along x, i.e. the
// band's contribution U_b[x] to every table row below it.  Pass B: per band, thread x keeps
// S[y][x] for its column in a register: S[y+1][x] = S[y][x] + (sum of row y left of x), the row
// prefix coming from a block-wide scan of the row, eight rows per barrier.
constexpr int kSatBandRows = 32;
constexpr int kSatBatch = 8;

// exclusive block-wide scan of one value per thread; `tot` (one slot per warp) is scratch
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* tot, uint32_t lane, uint32_t warp, uint32_t n_warps) {
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += n;
    }
    if (lane == 31) tot[warp] = incl;
    __syncthreads();
    uint32_t t = lane < n_warps ? tot[lane] : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, t, d);
        if (lane >= (uint32_t)d) t += n;
    }
    const uint32_t carry = __shfl_sync(0xffffffffu, t, (warp + 31u) & 31u);  // inclusive total of the warps before
    return (warp ? carry : 0u) + incl - v;
}

__global__ void __launch_bounds__(1024) sat_band_sums_kernel(const uint16_t* __restrict__ depth, uint32_t* __restrict__ band_u,
                                                             uint32_t w, uint32_t h, uint32_t n_bands) {
    __shared__ uint32_t s_tot[32];
    const uint32_t frame = blockIdx.y, band = blockIdx.x, x = threadIdx.x;
    const uint32_t y0 = band * kSatBandRows, y1 = min(h, y0 + kSatBandRows);
    const uint16_t* img = depth + (size_t)frame * h * w;
    uint32_t cs = 0;
    if (x < w) {
        uint32_t y = y0;
        for (; y + 8 <= y1; y += 8) {
            uint32_t v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = __ldg(img + (size_t)(y + j) * w + x);
#pragma unroll
            for (int j = 0; j < 8; ++j) cs += v[j];
        }
        for (; y < y1; ++y) cs += __ldg(img + (size_t)y * w + x);
    }
    const uint32_t u = block_excl_scan(cs, s_tot, x & 31u, x >> 5, blockDim.x >> 5);
    if (x <= w) band_u[((size_t)frame * n_bands + band) * (w + 1) + x] = u;
}

// Pass B.  One CTA per band of 32 rows, one warp per row: the row's exclusive prefix sums go to
// shared memory (8 pixels per lane per step, one 16-byte load, warp-shuffle scan of the lane
// totals); then one thread per column walks down the band adding them up and writes the table.
__global__ void __launch_bounds__(kSatBandRows * 32) sat_band_kernel(const uint16_t* __restrict__ depth,
                                                                     const uint32_t* __restrict__ band_u,
                                                                     uint32_t* __restrict__ sat, uint32_t w, uint32_t h,
                                                                     uint32_t pitch, uint32_t n_bands) {
    extern __shared__ __align__(16) uint32_t s_rows[];  // [kSatBandRows][spitch] exclusive row prefixes, positions 0..w
    const uint32_t spitch = (w + 1 + 8) & ~7u;          // every 8-wide store stays inside its row
    const uint32_t frame = blockIdx.y, band = blockIdx.x, tid = threadIdx.x;
    const uint32_t lane = tid & 31u, r = tid >> 5;
    const uint32_t y0 = band * kSatBandRows, y1 = min(h, y0 + kSatBandRows);
    const uint16_t* img = depth + (size_t)frame * h * w;
    if (y0 + r < y1) {
        const uint16_t* row = img + (size_t)(y0 + r) * w;
        uint32_t* srow = s_rows + r * spitch;
        const bool vec_ok = ((w & 7u) == 0u) && ((reinterpret_cast<uintptr_t>(row) & 15u) == 0u);
        uint32_t carry = 0;
        for (uint32_t seg = 0; seg <= w; seg += 256) {  // positions 0..w inclusive
            const uint32_t x = seg + lane * 8;
            uint32_t v[8];
            if (vec_ok && x + 8 <= w) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + x));
                v[0] = q.x & 0xffffu; v[1] = q.x >> 16; v[2] = q.y & 0xffffu; v[3] = q.y >> 16;
                v[4] = q.z & 0xffffu; v[5] = q.z >> 16; v[6] = q.w & 0xffffu; v[7] = q.w >> 16;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = (x + j < w) ? (uint32_t)__ldg(row + x + j) : 0u;
            }
            uint32_t e[8];
            uint32_t tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                e[j] = tot;
                tot += v[j];
            }
            uint32_t incl = tot;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= (uint32_t)d) incl += n;
            }
            const uint32_t base = carry + incl - tot;
            if (x <= w) {  // spitch leaves room for the whole 8-wide store
                *reinterpret_cast<uint4*>(srow + x) = make_uint4(base + e[0], base + e[1], base + e[2], base + e[3]);
                *reinterpret_cast<uint4*>(srow + x + 4) = make_uint4(base + e[4], base + e[5], base + e[6], base + e[7]);
            }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    __syncthreads();
    uint32_t* out = sat + (size_t)frame * (h + 1) * pitch;
    for (uint32_t x = tid; x <= w; x += kSatBandRows * 32) {
        // S[y0][x]: everything above this band and left of x
        uint32_t acc = 0;
        const uint32_t* u = band_u + (size_t)frame * n_bands * (w + 1) + x;
        uint32_t b2 = 0;
        for (; b2 + 4 <= band; b2 += 4) {  // four loads in flight
            const uint32_t u0 = __ldg(u + (size_t)b2 * (w + 1)), u1 = __ldg(u + (size_t)(b2 + 1) * (w + 1)),
                           u2 = __ldg(u + (size_t)(b2 + 2) * (w + 1)), u3 = __ldg(u + (size_t)(b2 + 3) * (w + 1));
            acc += u0 + u1 + u2 + u3;
        }
        for (; b2 < band; ++b2) acc += __ldg(u + (size_t)b2 * (w + 1));
        for (uint32_t y = y0; y < y1; ++y) {
            acc += s_rows[(y - y0) * spitch + x];
            out[(size_t)(y + 1) * pitch + x] = acc;
        }
    }
}

// ---------------------------------------------------------------- K1b: box-sum image
// Forests whose feature rectangles all have one size rw x rh (what the reference's trainer
// produces: houghforest.rs:230-234) never need a general summed-area table: the node test reads
// B[y][x] = sum of the rw x rh rectangle whose top-left pixel is (x, y) (types.rs:317-339 for that
// rectangle), one tap per rectangle.  This kernel writes B straight from the depth image: one
// read of the depth, one write of B, no intermediate table.
//
// The unit of work is a WARP: it owns a strip of at most 256 input columns (8 per lane, one
// 16-byte load per lane per row, fetched eight rows ahead) and sweeps down a band of rows with the
// rh-row window sums of its columns in registers: acc += row r, acc -= row r - rh + 1, the
// departing row coming from a lane-private ring of the last rh rows in shared memory (16 bytes
// per lane per row, no synchronisation).  Per output row the window sums become B either through
// nine shuffles (rectangle width a multiple of the lane's pixel count) or through exclusive
// prefix sums along x staged in a warp-private row of shared memory, B[y][x] = P[x + rw] - P[x];
// 16-byte stores.  No block-level barrier; all arithmetic in u32 (rw*rh*65535 < 2^31 is checked
// at load; prefix sums may wrap, differences are exact).  4 pixels per lane (twice the warps, half
// the ring each) measured slower: 0.47 vs 0.43 ms.
constexpr int kBoxMaxWarps = 8;                 // warps per CTA = strips of one (frame, band), when there are at most 8
constexpr int kBoxAhead = 8;                    // rows fetched ahead
constexpr int kBoxPx = 8;                       // pixels per lane: one 16-byte load, strips of 256 columns

struct BoxRow {
    uint32_t q[kBoxPx / 2];  // kBoxPx u16 pixels
};
__device__ __forceinline__ BoxRow box_fetch(const uint16_t* __restrict__ row, uint32_t w, uint32_t x, bool vec_ok, bool on) {
    BoxRow r;
#pragma unroll
    for (int j = 0; j < kBoxPx / 2; ++j) r.q[j] = 0u;
    if (!on) return r;
    if (vec_ok) {
        const uint4 t = __ldg(reinterpret_cast<const uint4*>(row + x));
        r.q[0] = t.x; r.q[1] = t.y; r.q[2] = t.z; r.q[3] = t.w;
        return r;
    }
#pragma unroll
    for (int j = 0; j < kBoxPx / 2; ++j) {
        const uint32_t lo = (x + 2 * j < w) ? (uint32_t)__ldg(row + x + 2 * j) : 0u;
        const uint32_t hi = (x + 2 * j + 1 < w) ? (uint32_t)__ldg(row + x + 2 * j + 1) : 0u;
        r.q[j] = lo | (hi << 16);
    }
    return r;
}
template <bool kAdd>
__device__ __forceinline__ void box_apply(uint32_t acc[kBoxPx], const BoxRow& r) {
#pragma unroll
    for (int j = 0; j < kBoxPx / 2; ++j) {
        const uint32_t lo = r.q[j] & 0xffffu, hi = r.q[j] >> 16;
        acc[2 * j] = kAdd ? acc[2 * j] + lo : acc[2 * j] - lo;
        acc[2 * j + 1] = kAdd ? acc[2 * j + 1] + hi : acc[2 * j + 1] - hi;
    }
}

// kWhole: rw is a multiple of kBoxPx, i.e. a rectangle row is a suffix of one lane's columns,
// rw/kBoxPx - 1 whole lanes and a prefix of one more lane: B comes straight out of shuffles, without
// the prefix sums over the whole warp and their trip through shared memory.
template <bool kWhole>
__global__ void __launch_bounds__(kBoxMaxWarps * 32) box_image_kernel(const uint16_t* __restrict__ depth, uint32_t* __restrict__ box,
                                                                uint32_t w, uint32_t h, uint32_t rw, uint32_t rh, uint32_t bw,
                                                                uint32_t bh, uint32_t bpitch, uint32_t strip_out, uint32_t n_strips,
                                                                uint32_t band_rows, uint32_t n_bands, uint32_t n_units) {
    constexpr uint32_t kRowPitch = 32 * kBoxPx + 16;      // P[0 .. 32*kBoxPx] + the slack the last active lane may read
    extern __shared__ __align__(16) uint32_t s_box[];  // [warps][2][kRowPitch] prefix rows (general widths only), then [warps][rh][32] pixel rings
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t n_warps = blockDim.x >> 5;  // the strips of one (frame, band) sit in one CTA: their reads and writes
                                               // of a row are adjacent in memory and happen at about the same time
    uint32_t unit = blockIdx.x * n_warps + warp;
    if (unit >= n_units) return;
    const uint32_t strip = unit % n_strips;
    unit /= n_strips;
    const uint32_t band = unit % n_bands, frame = unit / n_bands;
    const uint32_t c0 = strip * strip_out, c1 = min(bw, c0 + strip_out);  // output columns (c0 is a multiple of kBoxPx)
    const uint32_t y0 = band * band_rows, y1 = min(bh, y0 + band_rows);   // output rows
    if (c0 >= c1 || y0 >= y1) return;
    const uint32_t x_end = c1 + rw - 1u;          // one past the last input column (<= w)
    const uint32_t r_end = y1 + rh - 1u;          // one past the last input row (<= h)
    const uint16_t* img = depth + (size_t)frame * h * w;
    const bool vec_ok = ((w & (kBoxPx - 1u)) == 0u) && ((reinterpret_cast<uintptr_t>(img) & (2u * kBoxPx - 1u)) == 0u);
    const uint32_t my_x = c0 + lane * kBoxPx;
    const bool lane_in = my_x < x_end;            // the lane holds input pixels
    const bool lane_out = my_x < c1;              // the lane holds output columns
    const bool q_vec = (rw & 3u) == 0u;
    const uint32_t p_words = kWhole ? 0u : n_warps * 2u * kRowPitch;
    uint32_t* sp0 = s_box + warp * 2u * kRowPitch + lane * kBoxPx;
    BoxRow* ring = reinterpret_cast<BoxRow*>(s_box + p_words) + (size_t)warp * rh * 32u + lane;
    uint32_t* out = box + ((size_t)frame * bh + y0) * bpitch + my_x;
    const uint16_t* row_nxt = img + (size_t)y0 * w;   // next input row to fetch
    uint32_t acc[kBoxPx];
#pragma unroll
    for (int j = 0; j < kBoxPx; ++j) acc[j] = 0u;
    BoxRow q[kBoxAhead];
#pragma unroll
    for (int k = 0; k < kBoxAhead; ++k) {
        q[k] = box_fetch(row_nxt, w, my_x, vec_ok, lane_in && y0 + (uint32_t)k < r_end);
        row_nxt += w;
    }
    uint32_t buf = 0, slot = 0;                   // slot = (r - y0) mod rh
    for (uint32_t r0 = y0; r0 < r_end; r0 += kBoxAhead) {
#pragma unroll
        for (int k = 0; k < kBoxAhead; ++k) {
            const uint32_t r = r0 + (uint32_t)k;
            if (r >= r_end) break;
            const BoxRow cur = q[k];
            q[k] = box_fetch(row_nxt, w, my_x, vec_ok, lane_in && r + kBoxAhead < r_end);
            row_nxt += w;
            ring[slot * 32u] = cur;               // row r takes the place of row r - rh (left the window last round)
            if (++slot == rh) slot = 0;
            box_apply<true>(acc, cur);
            if (r + 1u >= y0 + rh) {              // the window [r - rh + 1, r] is complete
                const BoxRow old = ring[slot * 32u];  // row r - rh + 1 leaves the window
                // exclusive prefix sums of the lane's window sums
                uint32_t e[kBoxPx], tot = 0;
#pragma unroll
                for (int j = 0; j < kBoxPx; ++j) {
                    e[j] = tot;
                    tot += acc[j];
                }
                uint32_t t[kBoxPx];
                if (kWhole) {
                    // B[kBoxPx*l + j] = (T_l - e_l[j]) + T_{l+1} + .. + T_{l+k-1} + e_{l+k}[j],  k = rw / kBoxPx
                    const uint32_t k2 = rw / kBoxPx;
                    uint32_t whole = tot;
                    for (uint32_t i = 1; i < k2; ++i) whole += __shfl_down_sync(0xffffffffu, tot, i);
                    t[0] = whole;
#pragma unroll
                    for (int j = 1; j < kBoxPx; ++j) t[j] = whole - e[j] + __shfl_down_sync(0xffffffffu, e[j], k2);
                } else {
                    // general width: prefix sums over the whole warp, staged in shared memory
                    uint32_t incl = tot;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= (uint32_t)d) incl += n;
                    }
                    const uint32_t base = incl - tot;
#pragma unroll
                    for (int j = 0; j < kBoxPx; ++j) e[j] += base;
                    uint32_t* sp = sp0 + buf * kRowPitch;
#pragma unroll
                    for (int j = 0; j < kBoxPx; j += 4) *reinterpret_cast<uint4*>(sp + j) = make_uint4(e[j], e[j + 1], e[j + 2], e[j + 3]);
                    if (lane == 31u) sp[kBoxPx] = incl;  // P[32 * kBoxPx]
                    __syncwarp();
                    if (lane_out) {
                        if (q_vec) {
#pragma unroll
                            for (int j = 0; j < kBoxPx; j += 4) {
                                const uint4 a = *reinterpret_cast<const uint4*>(sp + rw + j);
                                t[j] = a.x - e[j]; t[j + 1] = a.y - e[j + 1]; t[j + 2] = a.z - e[j + 2]; t[j + 3] = a.w - e[j + 3];
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < kBoxPx; ++j) t[j] = sp[rw + j] - e[j];
                        }
                    }
                    buf ^= 1u;
                }
                if (lane_out) {
                    // columns at or beyond bw are row padding (never read); beyond the pitch nothing is stored
#pragma unroll
                    for (int j = 0; j < kBoxPx; j += 4)
                        if (my_x + (uint32_t)j < bpitch) *reinterpret_cast<uint4*>(out + j) = make_uint4(t[j], t[j + 1], t[j + 2], t[j + 3]);
                }
                out += bpitch;
                box_apply<false>(acc, old);
            }
        }
    }
}

// ================================================================ K2: forest traversal
// Node table prepared for one tile plan: see HotNode (dh_types.hpp).
// prob_codes != nullptr: a leaf child of a UniNode carries the leaf's probability code in bits 23..30
// of the complemented word, ~(leaf | code << 23) with code = min(floor(prob * 256), 255).  The walk
// stores the word as its leaf id, so that the patch gate knows every prob to within 1/256 from the
// leaf words alone (patch_gate_kernel); every reader of leaf ids applies FrameBuffers::leaf_mask.
__global__ void __launch_bounds__(256) plan_nodes_kernel(const NodeRec* __restrict__ nodes, HotNode* __restrict__ hot,
                                                         UniNode* __restrict__ uni, size_t n, uint32_t tw,
                                                         const double* __restrict__ prob_codes) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const NodeRec r = nodes[i];
    HotNode h;
    uint32_t c[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const uint32_t x0 = r.r[k * 4 + 0], y0 = r.r[k * 4 + 1], x1 = r.r[k * 4 + 2], y1 = r.r[k * 4 + 3];
        const uint32_t packed = (y0 * tw + x0) | ((x1 - x0) << 16) | ((y1 - y0) << 24);  // y0*tw + x0 <= 254*256+254
        if (k == 0) h.r1 = packed; else h.r2 = packed;
        c[k] = (x1 - x0) * (y1 - y0);
        if (c[k] == 0u) c[k] = 1u;  // empty rect: sum 0, avg 0.0 (types.rs:335-337)
    }
    h.counts = c[0] | (c[1] << 16);
    h.spare = 0u;
    h.child[0] = r.child[0];
    h.child[1] = r.child[1];
    h.thr_scaled = r.thr_scaled;
    hot[i] = h;
    if (uni) {  // all rectangles have one size: c[0] == c[1] == the common pixel count
        UniNode u;
        u.taps = (h.r1 & 0xffffu) | (h.r2 << 16);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            int32_t c = r.child[k];
            if (c < 0 && prob_codes) {
                const uint32_t leaf = (uint32_t)~c;
                const double pr = prob_codes[leaf];  // in [0, 1], checked on the host
                const uint32_t code = min((uint32_t)__double2uint_rd(__dmul_rn(pr, 256.0)), 255u);
                c = ~(int32_t)(leaf | (code << kProbCodeShift));
            }
            u.child[k] = c;
        }
        // Decision value E for d2 = 2*(s1 - s2), |s1 - s2| < 2^30 (rw*rh <= 16383 is checked at
        // load).  The reference compares fl(fl(s1/c) - fl(s2/c)) > thr; its three roundings move
        // the left side by < 2.2e-11 (|s/c| <= 65535, eps = 2^-53), so whenever the real numbers
        // differ by more than that, (s1 - s2) > thr*c decides.  y = fl(thr*c) is within 1.2e-7 of
        // thr*c for |y| < 2^30.  If y is further than 1e-3 from every integer, no integer s1 - s2
        // comes closer than 9e-4 to thr*c (5.5e-8 after the division by c): the answer is
        // s1 - s2 > floor(y), E = 2*floor(y) + 1 (odd: never equal to d2).  Otherwise only
        // s1 - s2 == m = rint(y) can be a tie: E = 2*m, d2 > E decides the rest and d2 == E goes
        // to the IEEE-division path.  NaN thresholds never pass (E = INT_MAX).
        const double y = __dmul_rn(r.threshold, (double)c[0]);
        int32_t E;
        if (!(y < 1073741824.0)) E = 0x7fffffff;            // y >= 2^30 or NaN: never greater
        else if (y <= -1073741824.0) E = -0x7fffffff;       // always greater
        else {
            const double m = rint(y);
            E = fabs(__dsub_rn(y, m)) <= 1e-3 ? 2 * (int32_t)m : 2 * (int32_t)floor(y) + 1;
        }
        u.e2 = E;
        uni[i] = u;
    }
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_u16(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)v) : "memory");
}

// HoughTreeFunctions::binarize (houghforest.rs:185-193) exactly as written: avg = sum as f64 /
// count as f64 (types.rs:335-338), avg1 - avg2 > threshold.  Only reached at near-ties.
__device__ __noinline__ bool binarize_ieee(const NodeRec* __restrict__ nodes, int32_t node, uint32_t s1, uint32_t s2) {
    const NodeRec r = nodes[node];
    const uint32_t c1 = (uint32_t)(r.r[2] - r.r[0]) * (uint32_t)(r.r[3] - r.r[1]);
    const uint32_t c2 = (uint32_t)(r.r[6] - r.r[4]) * (uint32_t)(r.r[7] - r.r[5]);
    const double avg1 = c1 ? __ddiv_rn(__uint2double_rn(s1), __uint2double_rn(c1)) : 0.0;
    const double avg2 = c2 ? __ddiv_rn(__uint2double_rn(s2), __uint2double_rn(c2)) : 0.0;
    return __dsub_rn(avg1, avg2) > r.threshold;
}

// One CTA per (tile of patches, frame).  The tile's SAT window (tw x th u32) is brought into
// shared memory by ONE TMA bulk-tensor load; all 8 taps of every node test are then shared-memory
// loads (32-bit shared addresses, ld.shared).  Tiles whose whole window is background (window sum
// 0, four taps of the global SAT) do no further work.  Non-background patches of the tile are
// compacted (ballot) so that every lane of the traversal loop owns a live patch x tree pair; lanes
// of a warp are neighbouring patches of the same tree, so the upper levels read the same node
// record (broadcast) and nearby taps.
// kMode 0: general rectangles, nodes through the LSU path; 1: general, nodes through the texture
// path; 2: uniform rectangles (box-sum tile, UniNode through the texture path); 4: as 2, but the
// TMA load brings a window of the box-sum image (box_image_kernel) instead of the summed-area
// table, so the tile needs no conversion and is (sw - rw + 1)-ish wide instead of (sw + 1)-ish.
// Mode 4 fetches the nodes of its first kLdgLevels levels through the LSU path.
constexpr uint32_t kLdgLevels = 7;  // measured: 1.071 -> 1.048 ms (3: 1.057, 5: 1.051, 7-11: 1.048, 13: 1.057)
template <int kThreads, int kMode>
__global__ void __launch_bounds__(kThreads, kThreads == 1024 ? 2 : 3) traverse_kernel(const __grid_constant__ CUtensorMap sat_map,
                                                            cudaTextureObject_t hot_tex,
                                                            const HotNode* __restrict__ hot,
                                                            const UniNode* __restrict__ uni,
                                                            const NodeRec* __restrict__ nodes,
                                                            const int32_t* __restrict__ roots, int32_t* __restrict__ leaf,
                                                            const uint32_t* __restrict__ sat,
                                                            FrameState* __restrict__ fs, Geometry g, TilePlan tp,
                                                            uint32_t uni_rw, uint32_t uni_rh) {
    extern __shared__ uint8_t smem_raw[];
    // 128-byte aligned tile (TMA destination), then the barrier, then the compacted patch list;
    // everything is addressed through 32-bit shared-window addresses
    const uint32_t tile_a = (smem_u32(smem_raw) + 127u) & ~127u;
    const uint32_t tile_bytes = tp.tw * tp.th * 4u;
    const uint32_t bar_a = tile_a + ((tile_bytes + 15u) & ~15u);
    const uint32_t live_a = bar_a + 16u;
    __shared__ uint32_t s_nlive, s_empty;

    const uint32_t frame = blockIdx.y;
    const uint32_t tile_x = blockIdx.x % tp.tiles_x, tile_y = blockIdx.x / tp.tiles_x;
    const uint32_t px0 = tile_x * tp.tpx, py0 = tile_y * tp.tpy;  // first patch of the tile
    const uint32_t tid = threadIdx.x;
    const int T = (int)g.n_trees;
    int32_t* leaf_f = leaf + (size_t)frame * T * g.P;

    // TMA needs the innermost coordinate 16-byte aligned: start the tile at a multiple of 4
    // elements and shift the patch origins by the slack dx (the planner widened tw for it).
    const uint32_t x0 = px0 * g.stride, y0 = py0 * g.stride, ax0 = x0 & ~3u, dx = x0 - ax0;
    if (tid == 0) {
        prefetch_tensormap(&sat_map);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_a), "r"(1u) : "memory");
        fence_mbar_init();
        s_nlive = 0;
        // the load is issued before the tile's background check and lands while warp 0 tests the
        // window (one global round trip less in front of every non-empty tile; measured 1.110 -> 1.052 ms)
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(tile_bytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(tile_a),
            "l"(&sat_map), "r"((int)ax0), "r"((int)y0), "r"((int)frame), "r"(bar_a)
            : "memory");
    }
    if (tid < 32u) {
        // window of the tile's patches: [x0, x1) x [y0, y1); every patch of the tile is background
        // (prediction.rs:567-571) iff no pixel of the window is set
        const uint32_t lastx = min(px0 + tp.tpx, g.npx) - 1u, lasty = min(py0 + tp.tpy, g.npy) - 1u;
        const uint32_t x1 = lastx * g.stride + g.sw, y1 = lasty * g.stride + g.sh;
        bool any;
        if (kMode == 4) {
            // covered by rw x rh rectangles of the box-sum image (the last one of a row / column
            // is pulled back inside the window; sums are non-negative, so overlap is harmless)
            const uint32_t nkx = (x1 - x0 + uni_rw - 1u) / uni_rw, nky = (y1 - y0 + uni_rh - 1u) / uni_rh;
            const uint32_t* B = sat + (size_t)frame * g.box_h * g.box_pitch;
            uint32_t acc = 0;
            for (uint32_t i = tid; i < nkx * nky; i += 32u) {
                const uint32_t kx = i % nkx, ky = i / nkx;
                const uint32_t bx = min(x0 + kx * uni_rw, x1 - uni_rw), by = min(y0 + ky * uni_rh, y1 - uni_rh);
                acc |= __ldg(B + (size_t)by * g.box_pitch + bx);
            }
            any = __any_sync(0xffffffffu, acc != 0u);
        } else {
            // the window's pixel sum is < 2^32 (<= 256*256 pixels), so the modular four-tap
            // difference of the summed-area table is zero iff every pixel is
            const uint32_t* S = sat + (size_t)frame * (g.h + 1) * g.sat_pitch;
            const uint32_t sum = __ldg(S + (size_t)y1 * g.sat_pitch + x1) - __ldg(S + (size_t)y0 * g.sat_pitch + x1) -
                                 __ldg(S + (size_t)y1 * g.sat_pitch + x0) + __ldg(S + (size_t)y0 * g.sat_pitch + x0);
            any = sum != 0u;
        }
        if (tid == 0) s_empty = !any;
    }
    __syncthreads();
    // an empty tile still waits for its load: the CTA must not leave while the async proxy writes its
    // shared memory
    {
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "LAB_WAIT:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
            "@P1 bra DONE;\n"
            "bra LAB_WAIT;\n"
            "DONE:\n"
            "}\n" ::"r"(bar_a),
            "r"(0u)
            : "memory");
    }
    if (s_empty) return;  // prediction.rs:567-571 fails for every patch of the tile: their leaf ids stay -1

    // ---- background test (prediction.rs:567-571: mean over the whole patch > 0  <=>  sum != 0)
    const uint32_t tw4 = tp.tw * 4u;
    const uint32_t org_a = tile_a + dx * 4u;  // patch (0,0) of the tile
    // patches in blocks of 8 x 4, one per warp: the lanes of a warp stay on the same nodes for longer
    // (measured 1.052 -> 1.037 ms against rows of 32 patches)
    const uint32_t nbx = (tp.tpx + 7u) >> 3;
    const uint32_t n_lp = nbx * ((tp.tpy + 3u) >> 2) * 32u;
    for (uint32_t lp = tid; lp < n_lp; lp += kThreads) {
        bool ok = false;
        uint32_t packed = 0;
        const uint32_t blk = lp >> 5;
        const uint32_t lx = (blk % nbx) * 8u + (lp & 7u), ly = (blk / nbx) * 4u + ((lp >> 3) & 3u);
        if (lx < tp.tpx && ly < tp.tpy) {
            const uint32_t gx = px0 + lx, gy = py0 + ly;
            if (gx < g.npx && gy < g.npy) {
                const uint32_t o = org_a + ly * g.stride * tw4 + lx * g.stride * 4u;
                uint32_t sum;
                if (kMode == 4) {  // the patch covered by rw x rh rectangles, the last ones pulled back inside
                    sum = 0;
                    for (uint32_t vy = 0; vy < g.sh; vy += uni_rh) {
                        const uint32_t ra = o + min(vy, g.sh - uni_rh) * tw4;
                        for (uint32_t vx = 0; vx < g.sw; vx += uni_rw) sum |= lds_u32(ra + min(vx, g.sw - uni_rw) * 4u);
                    }
                } else {
                    sum = lds_u32(o + g.sh * tw4 + g.sw * 4u) - lds_u32(o + g.sw * 4u) - lds_u32(o + g.sh * tw4) + lds_u32(o);
                }
                ok = sum != 0u;  // background patches keep the -1 the leaf buffer was filled with
                packed = (ly * g.stride * tp.tw + lx * g.stride) | ((lx | (ly << 8)) << 16);  // origin word offset (< 65536) | patch
            }
        }
        const uint32_t m = __ballot_sync(0xffffffffu, ok);
        uint32_t basei = 0;
        if ((tid & 31u) == 0 && m) basei = atomicAdd(&s_nlive, (uint32_t)__popc(m));
        basei = __shfl_sync(0xffffffffu, basei, 0);
        if (ok) {
            sts_u32(live_a + 4u * (basei + __popc(m & ((1u << (tid & 31u)) - 1u))), packed);
        }
    }
    __syncthreads();
    const uint32_t nlive = s_nlive;
    if (tid == 0 && nlive) atomicAdd(&fs[frame].n_valid, nlive);

    if (kMode == 2 && nlive) {
        // ---- uniform rectangles: turn the SAT tile into box sums in place,
        //      B[y][x] = S[y+rh][x+rw] - S[y][x+rw] - S[y+rh][x] + S[y][x]  (types.rs:317-339 for the
        //      rw x rh rectangle at (x, y)), so that a rectangle is ONE tap.  Rows go in waves of one
        //      per warp: a wave reads, barrier, writes; later waves only touch rows below.
        const uint32_t rw4 = uni_rw * 4u, rh4 = uni_rh * tw4;
        const uint32_t n_rows = tp.th - uni_rh, n_cols = tp.tw - uni_rw;  // B is defined for y < n_rows, x < n_cols
        constexpr int kPerLane = 8;  // tile width <= 256
        for (uint32_t r0 = 0; r0 < n_rows; r0 += kThreads / 32) {
            const uint32_t r = r0 + (tid >> 5);
            const uint32_t row_a = tile_a + r * tw4;
            uint32_t v[kPerLane];
#pragma unroll
            for (int j = 0; j < kPerLane; ++j) {
                const uint32_t x = (uint32_t)j * 32u + (tid & 31u);
                if (r < n_rows && x < n_cols) {
                    const uint32_t a = row_a + x * 4u;
                    v[j] = lds_u32(a + rh4 + rw4) - lds_u32(a + rw4) - lds_u32(a + rh4) + lds_u32(a);
                }
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < kPerLane; ++j) {
                const uint32_t x = (uint32_t)j * 32u + (tid & 31u);
                if (r < n_rows && x < n_cols) sts_u32(row_a + x * 4u, v[j]);
            }
        }
        __syncthreads();
    }

    // ---- root -> leaf walks: item = (tree, live patch); lanes = neighbouring live patches
    uint32_t visits = 0;
    const uint32_t items = nlive * (uint32_t)T;
    const uint4* hot4 = reinterpret_cast<const uint4*>(hot);
    // it / nlive by multiply-high (exact while it * nlive < 2^32)
    const uint32_t nl_magic = (nlive >= 2u && (unsigned long long)items * nlive < (1ull << 32)) ? (uint32_t)((1ull << 32) / nlive) + 1u : 0u;
    if (kMode == 4) {
        // the default walk (uniform rectangles, box-sum tile, nodes through the texture path), in two
        // passes.  The fast pass contains no call: an exact tie (2*(s1 - s2) == E, possible for even E
        // only) abandons the walk and marks the evaluation's leaf slot; the second pass, entered only
        // by threads that saw a tie, redoes the marked evaluations with the IEEE-division path.  The
        // call and everything it keeps alive stay out of the hot loop (no spills around it).
        constexpr int32_t kTieMark = (int32_t)0x80000000;
        bool any_tie = false;
        for (uint32_t it = tid; it < items; it += kThreads) {
            const uint32_t t = nl_magic ? __umulhi(it, nl_magic) : it / nlive;
            const uint32_t lp = lds_u32(live_a + 4u * (it - t * nlive));
            const uint32_t o = org_a + ((lp & 0xffffu) << 2);
            int32_t node = __ldg(roots + t);
            uint32_t nv = 0;
            bool tie = false;
            // the first levels below the root, where the lanes of a warp still sit on a handful of nodes, through
            // the LSU path (a warp-wide load of one address is one wavefront; a texture fetch costs eight or more
            // whatever the addresses)
            for (uint32_t lv = 0; lv < kLdgLevels && node >= 0; ++lv) {
                const uint4 U = __ldg(reinterpret_cast<const uint4*>(uni) + node);
                const uint32_t s1 = lds_u32(o + ((U.x & 0xffffu) << 2)), s2 = lds_u32(o + ((U.x >> 16) << 2));
                const int32_t d2 = (int32_t)(s1 - s2) << 1, E = (int32_t)U.w;
                if (d2 == E) {
                    tie = true;
                    break;
                }
                node = d2 > E ? (int)U.z : (int)U.y;
                ++nv;
            }
            while (node >= 0 && !tie) {
                const uint4 U = tex1Dfetch<uint4>(hot_tex, node);
                const uint32_t s1 = lds_u32(o + ((U.x & 0xffffu) << 2)), s2 = lds_u32(o + ((U.x >> 16) << 2));
                const int32_t d2 = (int32_t)(s1 - s2) << 1, E = (int32_t)U.w;
                if (d2 == E) {
                    tie = true;
                    break;
                }
                node = d2 > E ? (int)U.z : (int)U.y;
                ++nv;
            }
            any_tie |= tie;
            visits += tie ? 0u : nv;
            const uint32_t gp = (py0 + (lp >> 24)) * g.npx + (px0 + ((lp >> 16) & 0xffu));
            leaf_f[(size_t)t * g.P + gp] = tie ? kTieMark : ~node;  // leaf id | probability code << 23 (plan_nodes_kernel)
        }
        if (any_tie) {
            for (uint32_t it = tid; it < items; it += kThreads) {
                const uint32_t t = nl_magic ? __umulhi(it, nl_magic) : it / nlive;
                const uint32_t lp = lds_u32(live_a + 4u * (it - t * nlive));
                const uint32_t gp = (py0 + (lp >> 24)) * g.npx + (px0 + ((lp >> 16) & 0xffu));
                int32_t* slot = leaf_f + (size_t)t * g.P + gp;
                if (*slot != kTieMark) continue;  // written by this very thread in the first pass
                const uint32_t o = org_a + ((lp & 0xffffu) << 2);
                int32_t node = __ldg(roots + t);
                while (node >= 0) {
                    const uint4 U = tex1Dfetch<uint4>(hot_tex, node);
                    const uint32_t s1 = lds_u32(o + ((U.x & 0xffffu) << 2)), s2 = lds_u32(o + ((U.x >> 16) << 2));
                    const int32_t d2 = (int32_t)(s1 - s2) << 1, E = (int32_t)U.w;
                    int32_t next = d2 > E ? (int)U.z : (int)U.y;
                    if (d2 == E) next = binarize_ieee(nodes, node, s1, s2) ? (int)U.z : (int)U.y;
                    node = next;
                    ++visits;
                }
                *slot = ~node;
            }
        }
    } else
    for (uint32_t it = tid; it < items; it += kThreads) {
        const uint32_t t = nl_magic ? __umulhi(it, nl_magic) : it / nlive;
        const uint32_t lp = lds_u32(live_a + 4u * (it - t * nlive));
        const uint32_t lx = (lp >> 16) & 0xffu, ly = lp >> 24;
        const uint32_t o = org_a + ((lp & 0xffffu) << 2);
        int32_t node = __ldg(roots + t);
        if (kMode == 2) {
            while (node >= 0) {
                // taps, child[0], child[1], threshold * count
                const uint4 U = tex1Dfetch<uint4>(hot_tex, node);
                const uint32_t s1 = lds_u32(o + ((U.x & 0xffffu) << 2)), s2 = lds_u32(o + ((U.x >> 16) << 2));
                // binarize (houghforest.rs:185-193) for equal pixel counts c: avg1 - avg2 > thr, decided
                // on integers.  U.w = E (plan_nodes_kernel): the answer is 2*(s1 - s2) > E, and only
                // 2*(s1 - s2) == E (an exact tie up to the reference's own roundings, possible for
                // even E only) takes the IEEE-division path.
                const int32_t d2 = (int32_t)(s1 - s2) << 1, E = (int32_t)U.w;
                int32_t next = d2 > E ? (int)U.z : (int)U.y;
                if (d2 == E) next = binarize_ieee(nodes, node, s1, s2) ? (int)U.z : (int)U.y;
                node = next;
                ++visits;
            }
        } else
        while (node >= 0) {
            uint4 A, B;  // A: rect taps, pixel counts;  B: children, threshold * c1 * c2
            if (kMode == 1) {
                A = tex1Dfetch<uint4>(hot_tex, 2 * node);
                B = tex1Dfetch<uint4>(hot_tex, 2 * node + 1);
            } else {
                A = __ldg(hot4 + 2 * (size_t)node);
                B = __ldg(hot4 + 2 * (size_t)node + 1);
            }
            // SubImage::average_value_in_rect (types.rs:317-339) via four SAT taps per rectangle
            const uint32_t a00 = o + ((A.x & 0xffffu) << 2), aw = __byte_perm(A.x, 0u, 0x4442) << 2, ah = (A.x >> 24) * tw4;
            const uint32_t b00 = o + ((A.y & 0xffffu) << 2), bw = __byte_perm(A.y, 0u, 0x4442) << 2, bh = (A.y >> 24) * tw4;
            const uint32_t s1 = lds_u32(a00 + ah + aw) - lds_u32(a00 + aw) - lds_u32(a00 + ah) + lds_u32(a00);
            const uint32_t s2 = lds_u32(b00 + bh + bw) - lds_u32(b00 + bw) - lds_u32(b00 + bh) + lds_u32(b00);
            // HoughTreeFunctions::binarize (houghforest.rs:185-193): avg1 - avg2 > threshold with
            // avg = sum as f64 / count as f64.  Filtered exact predicate: the real number
            // avg1 - avg2 is N/D with N = s1*c2 - s2*c1, D = c1*c2 (exact in i64); the reference's
            // three roundings move it by < 3e-11, i.e. < 0.13 in units of 1/D, and thr*D carries
            // one more rounding (< 0.13 whenever it can matter), so whenever |N - thr*D| > 2 the
            // sign of N - thr*D IS the reference's answer.  Only near-ties (and NaN thresholds)
            // take the IEEE-division path.
            const uint32_t d1 = A.z & 0xffffu, d2 = A.z >> 16;
            const long long N = (long long)((unsigned long long)s1 * d2) - (long long)((unsigned long long)s2 * d1);
            const double diff = __dsub_rn(__ll2double_rn(N), __hiloint2double((int)B.w, (int)B.z));
            int32_t next = diff > 0.0 ? (int)B.y : (int)B.x;
            if (!(fabs(diff) > 2.0)) next = binarize_ieee(nodes, node, s1, s2) ? (int)B.y : (int)B.x;
            node = next;
            ++visits;
        }
        const uint32_t gp = (py0 + ly) * g.npx + (px0 + lx);
        leaf_f[(size_t)t * g.P + gp] = ~node;
    }

    // ---- per-frame counters (measured mean depth feeds the roofline arithmetic)
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) visits += __shfl_xor_sync(0xffffffffu, visits, d);
    if ((tid & 31u) == 0 && visits) atomicAdd(&fs[frame].node_visits, (unsigned long long)visits);
}

// ================================================================ K3: patch gate + coarse seed grids
// Phase A, one thread per patch: ordered f64 probability sum and the 0.7 gate
// (prediction.rs:582-584) and the back-projected centre (prediction.rs:551-554); gate-passing
// patches are compacted into shared memory and appended to the frame's gated-patch list (one
// reservation per CTA).  Phase B, one thread (or G lanes) per gated patch x tree pair: the leaf's
// votes go into the two coarse seed grids (prediction.rs:630-636, 661-675) held in shared memory;
// non-zero cells are then added to the frame's grids in global memory.  Everything that is
// constant per leaf (valtoadd, spread gates) was precomputed by leaf_gate_kernel.
constexpr int kGateThreads = 512;   // 3 CTAs of 59 KB per SM: 48 warps (256 threads with 48 KB: 32 warps)
constexpr int kTouchedCap = 1024;

// Per-frame intrinsics (dh_predict_frames): the kernels of the pose path take a table [F][18] of
// every frame's K then K^-1 (kFrameK instantiations) instead of Geometry's one matrix.  A CTA
// works on one frame: patch_gate_kernel and seed_kernel load the matrix into registers once per
// thread, gate_coarse_kernel keeps it in shared memory (see there).
constexpr int kFrameKFloats = 18;
__device__ __forceinline__ void load_mat3(const float* __restrict__ src, float m[9]) {
#pragma unroll
    for (int k = 0; k < 9; ++k) m[k] = __ldg(src + k);
}

// 2-D projection of one centre vote onto the 20x20 seed grid (prediction.rs:661-675)
__device__ __forceinline__ uint32_t coarse_pos_cell(const Geometry& g, const float* K, float nx, float ny, float nz) {
    const float np[3] = {nx, ny, nz};
    float p2[2];
    space_to_img(K, np, p2);  // prediction.rs:661
    // max!/min! macros (prediction.rs:19-25): plain comparisons, NaN -> 0.0
    const float mx = (p2[0] > 0.0f) ? p2[0] : 0.0f;
    const float x2d = (mx < (float)(g.w - 1)) ? mx : (float)(g.w - 1);
    const float my = (p2[1] > 0.0f) ? p2[1] : 0.0f;
    const float y2d = (my < (float)(g.h - 1)) ? my : (float)(g.h - 1);
    // (x2d as usize) * 20 / w  (:671-674); the quotient by multiply-high when the host found an
    // exact magic number (numerator * divisor < 2^32), else by division
    const uint32_t nxi = __float2uint_rz(x2d) * kGuessGridParts, nyi = __float2uint_rz(y2d) * kGuessGridParts;
    const uint32_t cx = g.magic_w ? __umulhi(nxi, g.magic_w) : nxi / g.w;
    const uint32_t cy = g.magic_h ? __umulhi(nyi, g.magic_h) : nyi / g.h;
    return cy * kGuessGridParts + cx;
}
// Votes of 32 patch x tree pairs (one per lane) flattened over the lanes of the warp: lane l owns
// votes [start_l, start_l + n_l) of the warp-wide numbering; the owner of vote v is the largest
// lane whose start is <= v (lanes without votes share their successor's start and never win).
__device__ __forceinline__ uint32_t flat_owner(uint32_t start, uint32_t v) {
    uint32_t lo = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const uint32_t cand = lo + (uint32_t)s;
        if (__shfl_sync(0xffffffffu, start, cand) <= v) lo = cand;
    }
    return lo;
}
// Votes of 32 patch x tree pairs (one per lane) spread evenly over the lanes of the warp: in the
// warp-wide numbering, lane l's pair owns votes [start_l, start_l + n_l).  The pairs that have votes
// are compacted, in lane order, into warp-private slots of shared memory (32 bytes: start, first
// vote, weight, patch centre); a window of 32 votes then finds its owners with one warp-wide OR:
// every pair whose first vote falls into the window sets that bit, and vote j belongs to slot
// (pairs that began before the window) + popc(bits <= j) - 1.
struct alignas(16) PairSlot {
    uint4 a;    // start, first vote of the leaf, weight, caller's tag
    float4 h;   // p3 (prediction.rs:554) + patch index
};
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t x, uint32_t lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= (uint32_t)d) x += n;
    }
    return x;
}

// Calls body(vote index, weight, tag, p3, number of the vote within its pair) once per vote of the warp's 32 pairs, 32 votes at a time.
// n: votes of this lane's pair (0 = none), v0: its first vote.  All 32 lanes must call.
template <typename Body>
__device__ __forceinline__ void for_each_vote(uint32_t n, uint32_t v0, uint32_t wgt, uint32_t tag, const float4 h, PairSlot* slots,
                                              uint32_t lane, Body&& body) {
    const uint32_t has = __ballot_sync(0xffffffffu, n > 0u);
    if (!has) return;
    const uint32_t incl = warp_incl_scan(n, lane), start = incl - n;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    __syncwarp();  // the previous call's readers are done with the slots
    if (n > 0u) {
        PairSlot* mine = slots + __popc(has & ((1u << lane) - 1u));
        mine->a = make_uint4(start, v0, wgt, tag);
        mine->h = h;
    }
    __syncwarp();
    uint32_t before = 0;  // pairs whose votes begin before the window
    for (uint32_t vb = 0; vb < total; vb += 32u) {
        const uint32_t rel = start - vb;
        const uint32_t begins = __reduce_or_sync(0xffffffffu, (n > 0u && rel < 32u) ? (1u << rel) : 0u);
        const uint32_t k = before + (uint32_t)__popc(begins & (0xffffffffu >> (31u - lane))) - 1u;
        before += (uint32_t)__popc(begins);
        if (vb + lane < total) {
            const uint4 a = slots[k].a;
            const float4 c = slots[k].h;
            body(a.y + (vb + lane - a.x), a.z, a.w, c, vb + lane - a.x);
        }
    }
}

constexpr int kGateSmemBytes = kGateThreads * 16 + (kGateThreads / 32) * 32 * 32 + (kPosGridCells + kRotGridCells) * 4 + kTouchedCap * 2;

// The patch gate on its own (phase A of gate_coarse_kernel), one thread per patch: the passing patches
// are appended to the frame's gated-patch list, one reservation per warp; gate_coarse_kernel<., true>
// then reads slices of that list.  With probability codes in the leaf words (b.leaf_mask ==
// kLeafIdMask) the gate is decided from the T leaf words of the patch alone, coalesced loads, no
// gather: prob_t lies in [code_t / 256, (code_t + 1) / 256], so the f64 fold of the reference lies
// within [S, S + T] / 256 (up to its own rounding, which g.gate_pass_codes / g.gate_fail_codes leave
// room for); only a sum inside that band (a few percent of the patches) gathers the leaves'
// probabilities and folds them in tree order.  Without codes every patch does (0.19 ms per 1024
// frames of configs[1]: 34 M random 8-byte gathers, bound by the L1 miss path).
constexpr int kPatchGateThreads = 256;
constexpr int kPatchGatePer = 4;  // patches per thread (one: 0.15 ms per 1024 frames of configs[1], four: 0.10 ms).  The kernel
                                  // sits at a third of the HBM rate; loading every leaf word of a patch up front,
                                  // background or not, to save dependent round trips was slower (it reads 40 % more)
template <bool kFrameK>
__global__ void __launch_bounds__(kPatchGateThreads) patch_gate_kernel(FrameBuffers b, Geometry g, ForestDev f,
                                                                       const float* __restrict__ frame_k) {
    const uint32_t frame = blockIdx.y, lane = threadIdx.x & 31u;
    const uint32_t T = g.n_trees;
    const int32_t* leaf_f = b.leaf + (size_t)frame * T * g.P;
    const bool codes = b.leaf_mask == kLeafIdMask;
    uint32_t p[kPatchGatePer], S[kPatchGatePer];
    bool valid[kPatchGatePer], gate[kPatchGatePer];
#pragma unroll
    for (int k = 0; k < kPatchGatePer; ++k) {
        p[k] = (blockIdx.x * kPatchGatePer + k) * kPatchGateThreads + threadIdx.x;
        const int32_t w0 = p[k] < g.P ? leaf_f[p[k]] : -1;
        valid[k] = w0 >= 0;  // background patches carry -1 in the slice of tree 0
        S[k] = (uint32_t)w0 >> kProbCodeShift;
        gate[k] = false;
    }
    if (codes) {
        for (uint32_t t = 1; t < T; ++t) {
#pragma unroll
            for (int k = 0; k < kPatchGatePer; ++k)
                if (valid[k]) S[k] += (uint32_t)leaf_f[(size_t)t * g.P + p[k]] >> kProbCodeShift;
        }
    }
#pragma unroll
    for (int k = 0; k < kPatchGatePer; ++k) {
        if (!valid[k]) continue;
        bool exact = !codes;
        if (codes) {
            gate[k] = S[k] >= g.gate_pass_codes;
            exact = !gate[k] && S[k] + T > g.gate_fail_codes;
        }
        if (exact) {
            // prob = sum(leaf.prob) / len: f64 fold from 0.0 in tree order (prediction.rs:582);
            // four independent gathers in flight, the additions stay in tree order
            double s = 0.0;
            for (uint32_t t0 = 0; t0 < T; t0 += 4) {
                int32_t L[4];
                double pr[4];
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (t0 + u < T) L[u] = (int32_t)((uint32_t)leaf_f[(size_t)(t0 + u) * g.P + p[k]] & b.leaf_mask);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (t0 + u < T) pr[u] = __ldg(f.leaf_prob + L[u]);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (t0 + u < T) s = __dadd_rn(s, pr[u]);
            }
            gate[k] = s >= g.gate_min_sum;  // sum / T > 0.7 (prediction.rs:584), see Geometry::gate_min_sum
        }
    }
    // the depth under the centre of every passing patch (prediction.rs:551), in flight with the list reservation
    uint16_t z[kPatchGatePer];
    uint32_t m[kPatchGatePer], total = 0;
#pragma unroll
    for (int k = 0; k < kPatchGatePer; ++k) {
        z[k] = 0;
        if (gate[k]) {
            const uint32_t gx = p[k] % g.npx, gy = p[k] / g.npx;
            z[k] = b.depth[((size_t)frame * g.h + g.left_h + gy * g.stride) * g.w + g.left_w + gx * g.stride];
        }
        if (b.gate && p[k] < g.P) b.gate[(size_t)frame * g.P + p[k]] = gate[k] ? 1 : 0;
        m[k] = __ballot_sync(0xffffffffu, gate[k]);
        total += (uint32_t)__popc(m[k]);
    }
    if (!total) return;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&b.fs[frame].n_gate, total);  // one reservation per warp
    base = __shfl_sync(0xffffffffu, base, 0);
    float kinv[9];
    if (kFrameK) load_mat3(frame_k + (size_t)frame * kFrameKFloats + 9, kinv);
#pragma unroll
    for (int k = 0; k < kPatchGatePer; ++k) {
        if (gate[k]) {
            const uint32_t gx = p[k] % g.npx, gy = p[k] / g.npx;
            const uint32_t x = g.left_w + gx * g.stride, y = g.left_h + gy * g.stride;
            float p3[3];
            img_to_space(kFrameK ? kinv : g.Kinv, (float)x, (float)y, (float)z[k], p3);  // prediction.rs:554
            b.gated[(size_t)frame * g.P + base + __popc(m[k] & ((1u << lane) - 1u))] = make_float4(p3[0], p3[1], p3[2], __uint_as_float(p[k]));
            if (b.p3) {
                float* o = b.p3 + ((size_t)frame * g.P + p[k]) * 3;
                o[0] = p3[0]; o[1] = p3[1]; o[2] = p3[2];
            }
        }
        base += (uint32_t)__popc(m[k]);
    }
}

// One pass over the votes of every pair feeds both grids (a vote is an offset and a rotation; the
// pair's tag says which of the two spread gates is open).
// kFromList: the patch gate has already been applied by patch_gate_kernel: the CTA
// takes slices of kGateThreads entries of the frame's gated-patch list (blockIdx.x, + gridDim.x, ...)
// instead of gating the kGateThreads patches of its own index range, so that every CTA that runs
// has a full slice behind the fixed costs of its seed grids (clearing and flushing 8400 cells);
// CTAs beyond the end of the list leave at once.
// kFrameK: the frame's K (and, in phase A, K^-1) come from frame_k instead of g, copied once per CTA
// into 72 bytes of shared memory behind the other arrays: this kernel runs at the 40-register cap of
// 3 CTAs of 512 threads per SM, and 9 more live registers spilled.
template <bool kFromList, bool kFrameK>
__global__ void __launch_bounds__(kGateThreads, 3) gate_coarse_kernel(FrameBuffers b, Geometry g, ForestDev f,
                                                                      const float* __restrict__ frame_k) {
    extern __shared__ __align__(16) uint8_t gate_smem[];
    float4* s_gated = reinterpret_cast<float4*>(gate_smem);                                   // [kGateThreads] p3 + patch index of the CTA's gated patches
    PairSlot(*s_slots)[32] = reinterpret_cast<PairSlot(*)[32]>(gate_smem + kGateThreads * 16);  // [warps][32] vote spreading, one set per warp
    uint32_t* s_grid = reinterpret_cast<uint32_t*>(gate_smem + kGateThreads * 16 + (kGateThreads / 32) * 32 * 32);  // [0,400) centre, [400,8400) rotation
    uint16_t* s_touched = reinterpret_cast<uint16_t*>(s_grid + kPosGridCells + kRotGridCells);  // rotation cells this CTA made non-zero
    float* s_k = reinterpret_cast<float*>(gate_smem + kGateSmemBytes);  // kFrameK: the frame's K then K^-1
    __shared__ uint32_t s_ngate, s_base, s_ntouched, s_next;
    const uint32_t frame = blockIdx.y, tid = threadIdx.x, lane = tid & 31u;
    const uint32_t p = blockIdx.x * kGateThreads + tid;
    const uint32_t T = g.n_trees;
    const int32_t* leaf_f = b.leaf + (size_t)frame * T * g.P;
    FrameState* fs = b.fs + frame;
    uint32_t slice0 = blockIdx.x * kGateThreads, n_list = 0;
    if (kFromList) {
        n_list = fs->n_gate;  // complete: written by patch_gate_kernel
        if (slice0 >= n_list) return;
    }
    if (tid == 0) {
        s_ngate = 0;
        s_ntouched = 0;
        s_next = 0;
    }
    if (kFrameK && tid < (uint32_t)kFrameKFloats) s_k[tid] = __ldg(frame_k + (size_t)frame * kFrameKFloats + tid);
    if (kFromList)
        for (int i = tid; i < kPosGridCells + kRotGridCells; i += kGateThreads) s_grid[i] = 0;
    __syncthreads();

    uint32_t ngate;
    if (!kFromList) {
        // ---- phase A
        bool gate = false;
        float p3[3] = {0.f, 0.f, 0.f};
        if (p < g.P) {
            if (leaf_f[p] >= 0) {
                // prob = sum(leaf.prob) / len: f64 fold from 0.0 in tree order (prediction.rs:582);
                // four independent gathers in flight, the additions stay in tree order
                double s = 0.0;
                for (uint32_t t0 = 0; t0 < T; t0 += 4) {
                    int32_t L[4];
                    double pr[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (t0 + u < T) L[u] = (int32_t)((uint32_t)leaf_f[(size_t)(t0 + u) * g.P + p] & b.leaf_mask);
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (t0 + u < T) pr[u] = __ldg(f.leaf_prob + L[u]);
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (t0 + u < T) s = __dadd_rn(s, pr[u]);
                }
                gate = s >= g.gate_min_sum;  // sum / T > 0.7 (prediction.rs:584), see Geometry::gate_min_sum
            }
            if (gate) {
                const uint32_t gx = p % g.npx, gy = p / g.npx;
                const uint32_t x = g.left_w + gx * g.stride, y = g.left_h + gy * g.stride;
                const uint16_t z = b.depth[((size_t)frame * g.h + y) * g.w + x];  // prediction.rs:551
                img_to_space(kFrameK ? s_k + 9 : g.Kinv, (float)x, (float)y, (float)z, p3);  // prediction.rs:554
                if (b.p3) {
                    float* o = b.p3 + ((size_t)frame * g.P + p) * 3;
                    o[0] = p3[0]; o[1] = p3[1]; o[2] = p3[2];
                }
            }
            if (b.gate) b.gate[(size_t)frame * g.P + p] = gate ? 1 : 0;
        }
        {
            const uint32_t m = __ballot_sync(0xffffffffu, gate);
            uint32_t base = 0;
            if (lane == 0 && m) base = atomicAdd(&s_ngate, (uint32_t)__popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (gate) s_gated[base + __popc(m & ((1u << lane) - 1u))] = make_float4(p3[0], p3[1], p3[2], __uint_as_float(p));
        }
        __syncthreads();
        ngate = s_ngate;
        if (ngate == 0u) return;
        if (tid == 0) s_base = atomicAdd(&fs->n_gate, ngate);
        for (int i = tid; i < kPosGridCells + kRotGridCells; i += kGateThreads) s_grid[i] = 0;
        __syncthreads();
        if (tid < ngate) b.gated[(size_t)frame * g.P + s_base + tid] = s_gated[tid];
    }

    uint32_t cnt_c = 0, cnt_r = 0;
    unsigned long long nmid = 0, nrot = 0;
    for (;;) {  // kFromList: one round per slice of the list; else one round
        if (kFromList) {
            ngate = min((uint32_t)kGateThreads, n_list - slice0);
            if (tid < ngate) s_gated[tid] = __ldcg(b.gated + (size_t)frame * g.P + slice0 + tid);
            __syncthreads();
        }
        // ---- phase B: pair = (tree, gated patch), neighbouring lanes = neighbouring gated patches.
        // A warp takes 32 pairs at a time and spreads their votes evenly over its lanes (for_each_vote),
        // so leaves with few, many or no votes cost the same per vote.
        const uint32_t npairs = ngate * T;
        // batches of 32 pairs are handed out through a shared counter: their vote counts differ a lot
        for (;;) {
            uint32_t blk = 0;
            if (lane == 0) blk = atomicAdd(&s_next, 32u);
            blk = __shfl_sync(0xffffffffu, blk, 0);
            if (blk >= npairs) break;
            const uint32_t i = blk + lane;
            uint32_t n_c = 0, n_r = 0, v0 = 0, wgt = 0;
            float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < npairs) {
                const uint32_t t = i / ngate;
                h = s_gated[i - t * ngate];
                const int32_t L = (int32_t)((uint32_t)leaf_f[(size_t)t * g.P + __float_as_uint(h.w)] & b.leaf_mask);
                const LeafInfo li = f.leaf_info[L];
                if (li.flags & kLeafVotes) {  // prob > 0 (prediction.rs:590), weight != 0, a spread gate open
                    v0 = li.vote_start;
                    wgt = li.valtoadd;
                    if (li.flags & kLeafOffOk) { n_c = li.n_votes; ++cnt_c; nmid += li.n_votes; }
                    // rotation votes: the leaf's distinct seed-grid cells with their multiplicities (leaf_gate_kernel)
                    if (li.flags & kLeafRotOk) { n_r = li.flags >> kLeafRotCellsShift; ++cnt_r; nrot += li.n_votes; }
                }
            }
            // centre votes -> 20x20 grid: np = p3 - offset (prediction.rs:647); np.z < 0 is skipped (:650)
            auto centre_vote = [&](uint32_t vote, uint32_t ow, const float4& c) {
                const float4 o = __ldg(f.offsets + vote);
                const float nx = __fsub_rn(c.x, o.x), ny = __fsub_rn(c.y, o.y), nz = __fsub_rn(c.z, o.z);
                if (!(nz < 0.0f)) atomicAdd(&s_grid[coarse_pos_cell(g, kFrameK ? s_k : g.K, nx, ny, nz)], ow);
            };
            // rotation votes -> 20^3 grid; rough = r * 20 / 120 per axis (prediction.rs:630-636), static per vote
            auto rot_vote = [&](uint32_t entry, uint32_t ow) {
                const uint32_t e = __ldg(f.rot_cells + entry), cell = e & ((1u << kRotCellBits) - 1u);
                if (atomicAdd(&s_grid[kPosGridCells + cell], ow * (e >> kRotCellBits)) == 0u) {
                    const uint32_t slot = atomicAdd(&s_ntouched, 1u);
                    if (slot < (uint32_t)kTouchedCap) s_touched[slot] = (uint16_t)cell;
                }
            };
            {
                // item j of a pair is its centre vote j (j < n_c) and its rotation cell j (j < n_r <= n_votes)
                const uint32_t tag = (n_c ? 1u : 0u) | (n_r << 1);
                for_each_vote(max(n_c, n_r), v0, wgt, tag, h, s_slots[tid >> 5], lane,
                              [&](uint32_t vote, uint32_t ow, uint32_t tg, const float4& c, uint32_t j) {
                                  if (tg & 1u) centre_vote(vote, ow, c);
                                  if (j < (tg >> 1)) rot_vote(vote, ow);
                              });
            }
        }
        if (!kFromList) break;
        slice0 += gridDim.x * kGateThreads;
        if (slice0 >= n_list) break;
        __syncthreads();  // every warp is done with this slice's patches and has left the batch loop
        if (tid == 0) s_next = 0;
    }
    // per-frame counters, one atomic per warp
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        nmid += __shfl_xor_sync(0xffffffffu, nmid, d);
        nrot += __shfl_xor_sync(0xffffffffu, nrot, d);
        cnt_c += __shfl_xor_sync(0xffffffffu, cnt_c, d);
        cnt_r += __shfl_xor_sync(0xffffffffu, cnt_r, d);
    }
    if (lane == 0) {
        if (cnt_c) atomicAdd(&fs->n_chits, cnt_c);
        if (cnt_r) atomicAdd(&fs->n_rhits, cnt_r);
        if (nmid) atomicAdd(&fs->n_mid_votes, nmid);
        if (nrot) atomicAdd(&fs->n_rot_votes, nrot);
    }
    __syncthreads();
    uint32_t* gout = b.grids + (size_t)frame * (kPosGridCells + kRotGridCells);
    for (int i = tid; i < kPosGridCells; i += kGateThreads) {
        const uint32_t v = s_grid[i];
        if (v) atomicAdd(gout + i, v);
    }
    const uint32_t ntouched = s_ntouched;
    if (ntouched <= (uint32_t)kTouchedCap) {
        // a cell whose sum wrapped to 0 may be listed twice: the exchange makes the second visit add 0
        for (uint32_t i = tid; i < ntouched; i += kGateThreads) {
            const uint32_t c = kPosGridCells + s_touched[i];
            const uint32_t v = atomicExch(&s_grid[c], 0u);
            if (v) atomicAdd(gout + c, v);
        }
    } else {
        for (int i = kPosGridCells + tid; i < kPosGridCells + kRotGridCells; i += kGateThreads) {
            const uint32_t v = s_grid[i];
            if (v) atomicAdd(gout + i, v);
        }
    }
}

// ================================================================ K4a: seeds
// One CTA per frame: arg-max of the two coarse grids -> mean-shift seeds (prediction.rs:694-752,
// 437-460) and the origin of the frame's two accumulator cubes.
constexpr int kBox = 32;                      // cells per axis of the dense accumulator cube: the 20-cell window plus 6 cells of margin
constexpr int kBoxCells = kBox * kBox * kBox; // 32 768 cells = 128 KB (40^3: 414 k frames/s, 32^3: 434 k, 28^3: 439 k, 24^3: 398 k with 1269 rebuilds per 1024 frames)
constexpr int kSeedThreads = 512;
constexpr int kMsHistory = 64;

struct Best {
    uint32_t val, idx;
};
__device__ __forceinline__ Best better(Best a, Best b) {
    // first maximum in scan order == strict `>` fold (prediction.rs:694-702, 733-742)
    return (b.val > a.val || (b.val == a.val && b.idx < a.idx)) ? b : a;
}
__device__ Best block_argmax(const uint32_t* cells, int n, Best* s_red) {
    Best best{0u, 0u};
    for (int i = threadIdx.x; i < n; i += blockDim.x) best = better(best, Best{cells[i], (uint32_t)i});
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        Best o{__shfl_xor_sync(0xffffffffu, best.val, d), __shfl_xor_sync(0xffffffffu, best.idx, d)};
        best = better(best, o);
    }
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        Best r = s_red[0];
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) r = better(r, s_red[i]);
        s_red[0] = r;
    }
    __syncthreads();
    Best r = s_red[0];
    __syncthreads();
    return r;
}

// Centre seed of coarse cell `cell` (prediction.rs:706-729, 750): z = mean of the non-zero depth in
// the cell's pixels, the cell centre back-projected with kinv, truncated.  Whole CTA of kSeedThreads.
__device__ __forceinline__ void cell_seed(const Geometry& g, const uint16_t* img, uint32_t cell, const float* kinv,
                                          unsigned long long* s_sum, uint32_t* s_cnt, int32_t sm[3]) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t gpw = g.w / kGuessGridParts, gph = g.h / kGuessGridParts;
    const uint32_t cgx = cell % kGuessGridParts, cgy = cell / kGuessGridParts;
    unsigned long long zs = 0;
    uint32_t zc = 0;
    for (uint32_t i = tid; i < gpw * gph; i += kSeedThreads) {
        const uint32_t v = img[(size_t)(gph * cgy + i / gpw) * g.w + gpw * cgx + i % gpw];
        if (v > 0) {
            zs += v;
            zc += 1;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        zs += __shfl_xor_sync(0xffffffffu, zs, d);
        zc += __shfl_xor_sync(0xffffffffu, zc, d);
    }
    if (lane == 0) {
        s_sum[warp] = zs;
        s_cnt[warp] = zc;
    }
    __syncthreads();
    zs = 0;
    zc = 0;
    for (int i = 0; i < kSeedThreads / 32; ++i) {
        zs += s_sum[i];
        zc += s_cnt[i];
    }
    const float meanz = zc > 0 ? (float)__ddiv_rn((double)zs, (double)zc) : 0.0f;
    const float mxf = __fmul_rn(__fadd_rn((float)cgx, 0.5f), (float)gpw);  // :727-729
    const float myf = __fmul_rn(__fadd_rn((float)cgy, 0.5f), (float)gph);
    float m3[3];
    img_to_space(kinv, mxf, myf, meanz, m3);
    for (int k = 0; k < 3; ++k) sm[k] = __float2int_rz(m3[k]);  // :750
}

template <bool kFrameK>
__global__ void __launch_bounds__(kSeedThreads) seed_kernel(FrameBuffers b, Geometry g, uint32_t iterations,
                                                            const float* __restrict__ frame_k) {
    __shared__ Best s_red[kSeedThreads / 32];
    __shared__ unsigned long long s_sum[kSeedThreads / 32];
    __shared__ uint32_t s_cnt[kSeedThreads / 32];
    const uint32_t frame = blockIdx.x, tid = threadIdx.x;
    FrameState* fs = b.fs + frame;
    const uint32_t* grid = b.grids + (size_t)frame * (kPosGridCells + kRotGridCells);
    const uint32_t guessed = fs->has_guess;

    // ---- centre seed (prediction.rs:694-729, 750)
    int32_t sm[3];
    {
        const Best bp = block_argmax(grid, kPosGridCells, s_red);
        float kinv[9];
        if (kFrameK) load_mat3(frame_k + (size_t)frame * kFrameKFloats + 9, kinv);
        cell_seed(g, b.depth + (size_t)frame * g.h * g.w, bp.idx, kFrameK ? kinv : g.Kinv, s_sum, s_cnt, sm);
        if (guessed & 1u)  // prediction.rs:437-441
            for (int k = 0; k < 3; ++k) sm[k] = __float2int_rz(fs->midp_guess[k]);
    }
    // ---- rotation seed (prediction.rs:733-747, 448-460)
    int32_t sr[3];
    {
        const Best br = block_argmax(grid + kPosGridCells, kRotGridCells, s_red);  // :733-742
        const uint32_t rc[3] = {br.idx % 20u, (br.idx % 400u) / 20u, br.idx / 400u};
        for (int k = 0; k < 3; ++k) {
            // :745-747, or the caller's guess :448-450; then :458-460
            double deg = __ddiv_rn(__dadd_rn(__dmul_rn((double)rc[k], 360.0), 180.0), (double)kGuessGridParts);
            if (guessed & 2u) deg = __dadd_rn(__ddiv_rn(__dmul_rn(fs->rot_guess[k], 180.0), 3.14159), 180.0);
            sr[k] = __double2int_rz(__ddiv_rn(__dmul_rn(deg, (double)kRotGridParts), 360.0));
        }
    }
    if (tid == 0) {
        for (int k = 0; k < 3; ++k) {
            fs->seed_mid[k] = sm[k];
            fs->seed_rot[k] = sr[k];
            // cube centred on the seed: kBox/2 - 10 cells of margin around the seed's 20^3 window; a window that leaves it
            // makes the mean-shift CTA rebuild the cube around its position
            fs->box_org[0][k] = (int32_t)((uint32_t)sm[k] - (uint32_t)(kBox / 2));
            fs->box_org[1][k] = (int32_t)((uint32_t)sr[k] - (uint32_t)(kBox / 2));
        }
        fs->box_valid[0] = fs->box_valid[1] = iterations > 0 ? 1u : 0u;
    }
}

// ================================================================ K4b: accumulator cubes
// SparseArray3D<u32> (meanshift.rs:14-68) restricted to a dense kBox^3 cube of cells per
// (frame, accumulator), z fastest: plain u32 atomicAdd per in-cube vote, no hashing; votes outside
// the cube never touch memory.  One thread (or G lanes) per gated patch x tree pair.
// 32-bit and exact for every int32 cell and origin: for x >= org the difference fits u32.
__device__ __forceinline__ bool in_box(int x, int y, int z, const int32_t* org, uint32_t* idx) {
    const uint32_t rx = (uint32_t)x - (uint32_t)org[0], ry = (uint32_t)y - (uint32_t)org[1], rz = (uint32_t)z - (uint32_t)org[2];
    if (x < org[0] || y < org[1] || z < org[2] || rx >= (uint32_t)kBox || ry >= (uint32_t)kBox || rz >= (uint32_t)kBox) return false;
    *idx = (rx * kBox + ry) * kBox + rz;
    return true;
}
// lo..hi (cells an axis of a leaf's votes can reach) misses [org, org + kBox)
__device__ __forceinline__ bool misses_box(int lo, int hi, int org) {
    return hi < org || (lo >= org && (uint32_t)lo - (uint32_t)org >= (uint32_t)kBox);
}

// Adds the votes of one frame that fall into the cube(s).  Warp `first_warp` of `n_warps` takes
// pairs 32 at a time (one per lane) and spreads their votes over its lanes (flat_owner).
// which_mask: bit0 centre cube, bit1 rotation cube.  All 32 lanes of a warp must call.
__device__ __forceinline__ void accumulate_pairs(const float4* __restrict__ gated, uint32_t ngate, uint32_t T,
                                                 const int32_t* __restrict__ leaf_f, uint32_t leaf_mask, uint32_t P, uint32_t first_warp,
                                                 uint32_t n_warps, const ForestDev& f, uint32_t which_mask,
                                                 const int32_t* org_c, uint32_t* cube_c, const int32_t* org_r,
                                                 uint32_t* cube_r) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t npairs = ngate * T;
    for (uint32_t blk = first_warp * 32u; blk < npairs; blk += n_warps * 32u) {
        const uint32_t i = blk + lane;
        uint32_t n_c = 0, n_r = 0, v0 = 0, wgt = 0;
        float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < npairs) {
            const uint32_t t = i / ngate;
            h = __ldg(gated + (i - t * ngate));
            const int32_t L = (int32_t)((uint32_t)leaf_f[(size_t)t * P + __float_as_uint(h.w)] & leaf_mask);
            // the leaf's record: vote range, weight, spread gates and vote bounding boxes in one sector
            const uint4 r0 = __ldg(reinterpret_cast<const uint4*>(f.leaf_box + L));
            const uint4 r1 = __ldg(reinterpret_cast<const uint4*>(f.leaf_box + L) + 1);
            const uint32_t flags = r0.y >> 24;
            if (flags & kLeafVotes) {
                // Skip the leaf when the bounding box of its votes misses the cube.  Conservative,
                // hence exact: p3 - o and the truncation are monotone, so every vote cell lies in
                // [trunc(p3 - omax), trunc(p3 - omin)] per axis (the record's bounds are rounded
                // outwards); rotation bins lie in [rmin, rmax].
                bool do_c = (which_mask & 1u) && (flags & kLeafOffOk), do_r = (which_mask & 2u) && (flags & kLeafRotOk);
                if (do_c) {
                    const float omin[3] = {__uint_as_float(r1.x & 0xffff0000u), __uint_as_float(r1.y << 16), __uint_as_float(r1.y & 0xffff0000u)};
                    const float omax[3] = {__uint_as_float(r1.z << 16), __uint_as_float(r1.z & 0xffff0000u), __uint_as_float(r1.w << 16)};
                    const float pc[3] = {h.x, h.y, h.z};
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        if (misses_box(__float2int_rz(__fsub_rn(pc[k], omax[k])), __float2int_rz(__fsub_rn(pc[k], omin[k])), org_c[k])) do_c = false;
                }
                if (do_r) {
                    const int rmin[3] = {(int)(r0.w & 0xffu), (int)((r0.w >> 8) & 0xffu), (int)((r0.w >> 16) & 0xffu)};
                    const int rmax[3] = {(int)(r0.w >> 24), (int)(r1.x & 0xffu), (int)((r1.x >> 8) & 0xffu)};
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        if (misses_box(rmin[k], rmax[k], org_r[k])) do_r = false;
                }
                v0 = r0.x;
                wgt = r0.z;
                if (do_c) n_c = r0.y & 0xffffffu;
                if (do_r) n_r = r0.y & 0xffffffu;
            }
        }
        if (which_mask & 1u) {
            const uint32_t incl = warp_incl_scan(n_c, lane), start = incl - n_c;
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
            for (uint32_t vb = 0; vb < total; vb += 32u) {
                const uint32_t v = min(vb + lane, total - 1u);
                const uint32_t own = flat_owner(start, v);
                const uint32_t k = v - __shfl_sync(0xffffffffu, start, own);
                const uint32_t ov0 = __shfl_sync(0xffffffffu, v0, own), ow = __shfl_sync(0xffffffffu, wgt, own);
                const float px = __shfl_sync(0xffffffffu, h.x, own), py = __shfl_sync(0xffffffffu, h.y, own),
                            pz = __shfl_sync(0xffffffffu, h.z, own);
                if (vb + lane < total) {
                    const float4 o = __ldg(f.offsets + ov0 + k);
                    const float nx = __fsub_rn(px, o.x), ny = __fsub_rn(py, o.y), nz = __fsub_rn(pz, o.z);
                    uint32_t idx;  // mid[(x as i32, y as i32, z as i32)] += valtoadd  (prediction.rs:650,667)
                    if (!(nz < 0.0f) && in_box(__float2int_rz(nx), __float2int_rz(ny), __float2int_rz(nz), org_c, &idx))
                        atomicAdd(cube_c + idx, ow);
                }
            }
        }
        if (which_mask & 2u) {
            const uint32_t incl = warp_incl_scan(n_r, lane), start = incl - n_r;
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
            for (uint32_t vb = 0; vb < total; vb += 32u) {
                const uint32_t v = min(vb + lane, total - 1u);
                const uint32_t own = flat_owner(start, v);
                const uint32_t k = v - __shfl_sync(0xffffffffu, start, own);
                const uint32_t ov0 = __shfl_sync(0xffffffffu, v0, own), ow = __shfl_sync(0xffffffffu, wgt, own);
                if (vb + lane < total) {
                    const uint32_t bins = __ldg(f.rot_bins + ov0 + k);
                    uint32_t idx;  // rot[(r1, r2, r3)] += valtoadd  (prediction.rs:635)
                    if (in_box((int)(bins & 0xffu), (int)((bins >> 8) & 0xffu), (int)((bins >> 16) & 0xffu), org_r, &idx))
                        atomicAdd(cube_r + idx, ow);
                }
            }
        }
    }
}

constexpr int kBuildThreads = 256;
// kWhich: bit0 centre cube, bit1 rotation cube (3: the pose pass; 1 or 2: the tries of extra heads)
template <uint32_t kWhich>
__global__ void __launch_bounds__(kBuildThreads) box_build_kernel(FrameBuffers b, Geometry g, ForestDev f) {
    const uint32_t frame = blockIdx.y;
    const FrameState* fs = b.fs + frame;
    if (!fs->box_valid[kWhich == 2u ? 1 : 0]) return;  // meanshift_iterations == 0: the accumulators are never read
    const int32_t org_c[3] = {fs->box_org[0][0], fs->box_org[0][1], fs->box_org[0][2]};
    const int32_t org_r[3] = {fs->box_org[1][0], fs->box_org[1][1], fs->box_org[1][2]};
    uint32_t* cube_c = b.cubes + (size_t)(2u * frame) * kBoxCells;
    accumulate_pairs(b.gated + (size_t)frame * g.P, fs->n_gate, g.n_trees, b.leaf + (size_t)frame * g.n_trees * g.P, b.leaf_mask, g.P,
                     blockIdx.x * (kBuildThreads / 32) + (threadIdx.x >> 5), gridDim.x * (kBuildThreads / 32), f, kWhich, org_c,
                     cube_c, org_r, cube_c + kBoxCells);
}

// ================================================================ K4c: mean-shift
// MeanShift::meanshift (meanshift.rs:328-407) on the dense cube, one CTA per accumulator.  Per
// round the sixteen warps read the 20^3 window (16 loads in flight per lane), rank its non-zero
// cells in reference order (ballots + one cross-warp prefix) (x outermost, z innermost, offsets -10..+9: meanshift.rs:340-346),
// stage the summands in shared memory at that rank and four lanes fold them into the f32
// accumulators one after the other in exactly that order.  A round moves the position by at most
// 10 cells and the cube leaves 6 cells of margin around the seed's window (most runs move a cell or
// two per round; a larger cube costs more in clears and cache misses than rebuilds do); if the window
// would leave the cube, the cube is rebuilt around the current position from the frame's gated patches
// (counted in FrameState::rebuilds), so the results stay exactly those of the unbounded map.
constexpr int kMsThreads = 512;
constexpr int kMsWarps = kMsThreads / 32;
constexpr int kMsSegment = 1024;  // non-zero window cells summed per pass
constexpr uint32_t kMsChunks = kKernelCells / 32;  // 250 steps of 32 cells
constexpr int kMsLoads = (kKernelCells + kMsThreads - 1) / kMsThreads;  // 16 window cells per thread
constexpr int kMsSmemBytes = kMsSegment * 8 + 4 * kMsSegment * 4 + (kMsLoads / 2) * kMsThreads * 4;  // list of non-zero cells + summands + cell offsets
constexpr uint32_t kMsNoCell = 0xffffu;  // packed cell offset of a thread's load slot beyond the window

__device__ __forceinline__ void store_result(dh_result* r, uint32_t which, const int32_t* pos) {
    if (which == 0) {  // prediction.rs:486-488
        r->mid_point[0] = (float)pos[0];
        r->mid_point[1] = (float)pos[1];
        r->mid_point[2] = (float)pos[2];
        r->_pad = 0;
        r->bounding_box[0] = r->bounding_box[1] = r->bounding_box[2] = r->bounding_box[3] = 0;  // :491
    } else {           // prediction.rs:477-482
        for (int k = 0; k < 3; ++k)
            r->rotation[k] = __dmul_rn(__ddiv_rn(__dsub_rn((double)pos[k], (double)kRotGridParts / 2.0),
                                                 (double)(kRotGridParts / 2)),
                                       3.14159);
    }
}

// Clears one cube and re-accumulates the frame's votes around a new origin (whole CTA).
__device__ __noinline__ void rebuild_cube(const float4* __restrict__ gated, uint32_t ngate, uint32_t T,
                                          const int32_t* __restrict__ leaf_f, uint32_t leaf_mask, uint32_t P, const LeafInfo* leaf_info,
                                          const LeafBox* leaf_box, const float4* offsets, const uint32_t* rot_bins,
                                          uint32_t which, int32_t ox, int32_t oy, int32_t oz, uint32_t* box) {
    const int32_t org[3] = {ox, oy, oz};
    ForestDev f{};
    f.leaf_info = leaf_info;
    f.leaf_box = leaf_box;
    f.offsets = offsets;
    f.rot_bins = rot_bins;
    uint4* bz = reinterpret_cast<uint4*>(box);
    for (int i = threadIdx.x; i < kBoxCells / 4; i += kMsThreads) __stcg(bz + i, make_uint4(0u, 0u, 0u, 0u));
    __threadfence();
    __syncthreads();
    accumulate_pairs(gated, ngate, T, leaf_f, leaf_mask, P, threadIdx.x >> 5, kMsThreads / 32, f, 1u << which, org, box, org, box);
    __threadfence();
    __syncthreads();
}

// The window never goes to shared memory.  A thread keeps its 16 cells in registers from the gather to
// the ranking, the non-zero ones are written as (cell, value) at their rank, and the summands are then
// computed densely, one thread per non-zero cell (walking all 250 chunks of 32 cells with only the
// non-zero lanes working took 53 % of the kernel's instructions, measured).
// which_only: 2 = both accumulators of every frame (item = 2 * frame + which); 0 or 1 = that accumulator of
// every frame (item = frame), and only of frames whose FrameState::active has its bit (tries of extra heads).
__global__ void __launch_bounds__(kMsThreads, 3) meanshift_kernel(FrameBuffers b, Geometry g, ForestDev f, uint32_t iterations,
                                                                  uint32_t n_items, uint32_t which_only) {
    extern __shared__ __align__(16) uint8_t ms_smem[];
    uint2* s_list = reinterpret_cast<uint2*>(ms_smem);       // [kMsSegment] (ord, value) of the non-zero cells by rank
    float(*s_terms)[kMsSegment] = reinterpret_cast<float(*)[kMsSegment]>(ms_smem + kMsSegment * 8);  // [4][kMsSegment]
                                                       // summands (num x,y,z, den) in reference order
    uint32_t* s_offp = reinterpret_cast<uint32_t*>(ms_smem + kMsSegment * 8 + 4 * kMsSegment * 4);  // [kMsLoads / 2][kMsThreads]
    __shared__ uint32_t s_mask[kMsChunks];             // non-zero window cells, bit j of word c = ord c*32+j
    __shared__ uint32_t s_off[kMsChunks + 1];          // rank of the first non-zero cell of every chunk
    __shared__ int32_t s_hist[kMsHistory + 1][3];      // positions P_0 (seed), P_1, ... for cycle detection
    __shared__ int32_t s_pos[3], s_org[3];
    __shared__ uint32_t s_flags, s_done;
    __shared__ uint32_t s_item;
    __shared__ unsigned long long s_sup[kMsWarps];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    // cube offsets of this thread's window cells ord = j * kMsThreads + tid, two per word, computed
    // once and parked in shared memory (eight registers less across the rounds)
#pragma unroll
    for (int j = 0; j < kMsLoads; j += 2) {
        uint32_t pk = 0;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const uint32_t ord = (uint32_t)(j + u) * kMsThreads + tid;
            const uint32_t xo = ord / 400u, yo = (ord / 20u) % 20u, zo = ord % 20u;
            pk |= (ord < (uint32_t)kKernelCells ? (xo * kBox + yo) * kBox + zo : kMsNoCell) << (16 * u);
        }
        s_offp[(j >> 1) * kMsThreads + tid] = pk;
    }
    // The CTAs of the launch (as many as fit the GPU at once) take accumulators from a counter: the first
    // one by their index, the following ones as they become free (a launch of one CTA per accumulator ran
    // 2.3 rounds of CTAs and paid for three).
    for (uint32_t item = blockIdx.x; item < n_items;) {
    const uint32_t frame = which_only < 2u ? item : item >> 1, which = which_only < 2u ? which_only : item & 1u;
    FrameState* fs = b.fs + frame;
    uint32_t* box = b.cubes + (size_t)(2u * frame + which) * kBoxCells;
    if (which_only < 2u && !((fs->active >> which) & 1u)) {  // this frame's search has stopped, or its try was dropped
        if (tid == 0) s_item = gridDim.x + atomicAdd(&b.fs[0].work_next, 1u);
        __syncthreads();
        item = s_item;
        __syncthreads();
        continue;
    }
    const bool built = fs->box_valid[which] != 0u;  // box_build_kernel filled the cube around box_org
    if (tid == 0) {
        s_flags = 0;
        s_done = 0;
        const int32_t* seed = which == 0 ? fs->seed_mid : fs->seed_rot;
        for (int k = 0; k < 3; ++k) {
            s_pos[k] = s_hist[0][k] = seed[k];
            s_org[k] = fs->box_org[which][k];
        }
    }
    uint32_t rebuilds = 0;
    uint32_t it = 0;
    for (; it < iterations; ++it) {
        __syncthreads();
        const int32_t pos[3] = {s_pos[0], s_pos[1], s_pos[2]};
        int32_t org[3] = {s_org[0], s_org[1], s_org[2]};
        bool inside = true;
        for (int k = 0; k < 3; ++k) {
            const long long lo = (long long)pos[k] - 10 - org[k], hi = (long long)pos[k] + 9 - org[k];
            if (lo < 0 || hi >= kBox) inside = false;
        }
        if (!inside) {
            // rebuild the cube around the current position
            ++rebuilds;
            __syncthreads();
            for (int k = 0; k < 3; ++k) org[k] = (int32_t)((uint32_t)pos[k] - (uint32_t)(kBox / 2));
            if (tid == 0)
                for (int k = 0; k < 3; ++k) s_org[k] = org[k];
            rebuild_cube(b.gated + (size_t)frame * g.P, fs->n_gate, g.n_trees, b.leaf + (size_t)frame * g.n_trees * g.P, b.leaf_mask, g.P,
                         f.leaf_info, f.leaf_box, f.offsets, f.rot_bins, which, org[0], org[1], org[2], box);
        }
        const uint32_t base = ((uint32_t)((long long)pos[0] - 10 - org[0]) * kBox + (uint32_t)((long long)pos[1] - 10 - org[1])) * kBox +
                              (uint32_t)((long long)pos[2] - 10 - org[2]);
        // gather the 20^3 window, all loads of a thread in flight at once.  ord enumerates the cells in
        // the reference loop order (x outermost, z innermost); a warp's load j is chunk j * kMsWarps + warp.
        uint32_t v[kMsLoads];
#pragma unroll
        for (int j = 0; j < kMsLoads; j += 2) {
            const uint32_t pk = s_offp[(j >> 1) * kMsThreads + tid];
            const uint32_t o0 = pk & 0xffffu, o1 = pk >> 16;
            v[j] = o0 != kMsNoCell ? __ldcg(box + base + o0) : 0u;
            v[j + 1] = o1 != kMsNoCell ? __ldcg(box + base + o1) : 0u;
        }
        // non-zero mask of every 32-cell chunk straight from the registers
#pragma unroll
        for (int j = 0; j < kMsLoads; ++j) {
            const uint32_t m = __ballot_sync(0xffffffffu, v[j] != 0u);
            const uint32_t c = (uint32_t)j * kMsWarps + warp;
            if (lane == 0 && c < kMsChunks) s_mask[c] = m;
        }
        __syncthreads();
        // (warp 0) the exclusive prefix of the chunks' populations = rank of their first non-zero cell
        if (warp == 0) {
            uint32_t run = 0;
            for (uint32_t c0 = 0; c0 < kMsChunks; c0 += 32) {
                const uint32_t c = c0 + lane;
                const uint32_t n = c < kMsChunks ? (uint32_t)__popc(s_mask[c]) : 0u;
                uint32_t incl = n;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= (uint32_t)d) incl += o;
                }
                if (c < kMsChunks) s_off[c] = run + incl - n;
                run += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) s_off[kMsChunks] = run;
        }
        __syncthreads();
        const uint32_t nnz = s_off[kMsChunks];
        float acc = 0.0f;
        for (uint32_t seg = 0; seg < nnz; seg += kMsSegment) {
            // every non-zero cell goes to the list at its rank in reference order ...
#pragma unroll
            for (int j = 0; j < kMsLoads; ++j) {
                if (v[j] != 0u) {
                    const uint32_t c = (uint32_t)j * kMsWarps + warp;
                    const uint32_t r = s_off[c] + (uint32_t)__popc(s_mask[c] & ((1u << lane) - 1u)) - seg;
                    if (r < (uint32_t)kMsSegment) s_list[r] = make_uint2((uint32_t)j * kMsThreads + tid, v[j]);
                }
            }
            __syncthreads();
            // ... and its four summands are computed by the thread of that rank
            const uint32_t cnt = min((uint32_t)kMsSegment, nnz - seg);
            for (uint32_t r = tid; r < cnt; r += kMsThreads) {
                const uint2 e = s_list[r];
                const uint32_t xo = e.x / 400u, yo = (e.x / 20u) % 20u, zo = e.x % 20u;
                // influence * factor with kernel[(x+10, y+10, z+10)], dense index z*400 + y*20 + x
                // (meanshift.rs:370-377, 78-88); then abs_pos * that
                const float wgt = __fmul_rn(__ldg(f.ms_kernel + zo * 400u + yo * 20u + xo), (float)e.y);
                s_terms[0][r] = __fmul_rn((float)(int)((uint32_t)pos[0] + xo - 10u), wgt);
                s_terms[1][r] = __fmul_rn((float)(int)((uint32_t)pos[1] + yo - 10u), wgt);
                s_terms[2][r] = __fmul_rn((float)(int)((uint32_t)pos[2] + zo - 10u), wgt);
                s_terms[3][r] = wgt;
            }
            __syncthreads();
            if (warp == 0 && lane < 4) {  // sequential f32 accumulation in reference order (meanshift.rs:337-380)
                const uint32_t cnt = min((uint32_t)kMsSegment, nnz - seg);
                const float4* t4 = reinterpret_cast<const float4*>(s_terms[lane]);
                uint32_t i = 0;
                if (cnt >= 8) {  // software-pipelined: the next eight summands load while these are added
                    float4 a0 = t4[0], a1 = t4[1];
                    for (; i + 16 <= cnt; i += 8) {
                        const float4 n0 = t4[(i >> 2) + 2], n1 = t4[(i >> 2) + 3];
                        acc = __fadd_rn(acc, a0.x); acc = __fadd_rn(acc, a0.y); acc = __fadd_rn(acc, a0.z); acc = __fadd_rn(acc, a0.w);
                        acc = __fadd_rn(acc, a1.x); acc = __fadd_rn(acc, a1.y); acc = __fadd_rn(acc, a1.z); acc = __fadd_rn(acc, a1.w);
                        a0 = n0;
                        a1 = n1;
                    }
                    acc = __fadd_rn(acc, a0.x); acc = __fadd_rn(acc, a0.y); acc = __fadd_rn(acc, a0.z); acc = __fadd_rn(acc, a0.w);
                    acc = __fadd_rn(acc, a1.x); acc = __fadd_rn(acc, a1.y); acc = __fadd_rn(acc, a1.z); acc = __fadd_rn(acc, a1.w);
                    i += 8;
                }
                const float* t = s_terms[lane];
                for (; i < cnt; ++i) acc = __fadd_rn(acc, t[i]);
            }
            __syncthreads();
        }
        if (warp == 0) {
            const float den = __shfl_sync(0xffffffffu, acc, 3);
            if (den == 0.0f) {  // "Breaking meanshift - zero sum" (meanshift.rs:385-388)
                if (lane == 0) {
                    s_flags |= 1u;
                    s_done = 1;
                }
            } else {
                const int np = __float2int_rz(__fdiv_rn(acc, den));  // meanshift.rs:391-394
                const int nx = __shfl_sync(0xffffffffu, np, 0), ny = __shfl_sync(0xffffffffu, np, 1),
                          nz = __shfl_sync(0xffffffffu, np, 2);
                // Cycle detection (result-neutral): the update is a deterministic function of
                // the position, so once P_{k+1} equals an earlier P_j the sequence is periodic
                // with period k+1-j and P_iterations is read off the history (a fixed point is
                // the period-1 case).
                const uint32_t k1 = it + 1;
                int found = -1;
                if (k1 <= (uint32_t)kMsHistory) {
                    for (uint32_t j = lane; j < k1; j += 32)
                        if (s_hist[j][0] == nx && s_hist[j][1] == ny && s_hist[j][2] == nz) found = (int)j;
                    found = __reduce_max_sync(0xffffffffu, found);
                }
                if (lane == 0) {
                    if (b.ms_trace && it < b.ms_trace_cap) {
                        int32_t* tr = b.ms_trace + (((size_t)frame * 2 + which) * b.ms_trace_cap + it) * 3;
                        tr[0] = nx; tr[1] = ny; tr[2] = nz;
                    }
                    if (found >= 0) {
                        const uint32_t j = (uint32_t)found, period = k1 - j;
                        const uint32_t fin = j + (iterations - j) % period;  // index of P_iterations (< k1)
                        s_pos[0] = s_hist[fin][0]; s_pos[1] = s_hist[fin][1]; s_pos[2] = s_hist[fin][2];
                        s_done = 2;
                    } else {
                        s_pos[0] = nx; s_pos[1] = ny; s_pos[2] = nz;
                        if (k1 <= (uint32_t)kMsHistory) {
                            s_hist[k1][0] = nx; s_hist[k1][1] = ny; s_hist[k1][2] = nz;
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (s_done) {
            if (s_done == 2) ++it;  // this round was executed
            break;
        }
    }
    __syncthreads();
    if (b.support && which == 0u) {
        // the u32 cells of the final window: the cube holds them unless the last update (or the cycle stop) left it
        const int32_t pos[3] = {s_pos[0], s_pos[1], s_pos[2]};
        int32_t org[3] = {s_org[0], s_org[1], s_org[2]};
        bool inside = built;
        for (int k = 0; k < 3; ++k) {
            const long long lo = (long long)pos[k] - 10 - org[k], hi = (long long)pos[k] + 9 - org[k];
            if (lo < 0 || hi >= kBox) inside = false;
        }
        if (!inside) {
            ++rebuilds;
            __syncthreads();
            for (int k = 0; k < 3; ++k) org[k] = (int32_t)((uint32_t)pos[k] - (uint32_t)(kBox / 2));
            if (tid == 0)
                for (int k = 0; k < 3; ++k) s_org[k] = org[k];
            rebuild_cube(b.gated + (size_t)frame * g.P, fs->n_gate, g.n_trees, b.leaf + (size_t)frame * g.n_trees * g.P, b.leaf_mask, g.P,
                         f.leaf_info, f.leaf_box, f.offsets, f.rot_bins, which, org[0], org[1], org[2], box);
        }
        const uint32_t base = ((uint32_t)((long long)pos[0] - 10 - org[0]) * kBox + (uint32_t)((long long)pos[1] - 10 - org[1])) * kBox +
                              (uint32_t)((long long)pos[2] - 10 - org[2]);
        unsigned long long sum = 0;
#pragma unroll
        for (int j = 0; j < kMsLoads; j += 2) {
            const uint32_t pk = s_offp[(j >> 1) * kMsThreads + tid];
            const uint32_t o0 = pk & 0xffffu, o1 = pk >> 16;
            if (o0 != kMsNoCell) sum += __ldcg(box + base + o0);
            if (o1 != kMsNoCell) sum += __ldcg(box + base + o1);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
        if (lane == 0) s_sup[warp] = sum;
        __syncthreads();
        if (tid == 0) {
            unsigned long long t = 0;
            for (int i = 0; i < kMsWarps; ++i) t += s_sup[i];
            fs->support = t;
        }
        __syncthreads();
    }
    if (b.clear_cubes) {
        // leave the cube empty for the next pass over this scratch: 128 KB of stores that overlap the
        // other CTAs' rounds instead of one memset of every cube in front of the vote stage
        uint4* bz = reinterpret_cast<uint4*>(box);
        for (int i = tid; i < kBoxCells / 4; i += kMsThreads) __stcg(bz + i, make_uint4(0u, 0u, 0u, 0u));
    }
    if (tid == 0) {
        fs->ms_iters[which] = it;
        fs->ms_flags[which] = s_flags;
        fs->rebuilds[which] = rebuilds;
        for (int k = 0; k < 3; ++k) fs->box_org[which][k] = s_org[k];
        const int32_t fin[3] = {s_pos[0], s_pos[1], s_pos[2]};
        store_result(b.results + frame, which, fin);
        s_item = gridDim.x + atomicAdd(&b.fs[0].work_next, 1u);
    }
    __syncthreads();  // the next accumulator; nobody still reads this one's shared state
    item = s_item;
    __syncthreads();
    }
}

// ================================================================ K4d: extra heads (dh_predict_frames_heads)
// Rules: DESIGN.md §7 "Several heads per frame"; oracle: orc_predict_heads.  One CTA per frame for the
// seed and patch kernels; the cubes and mean-shift of a try are box_build_kernel and meanshift_kernel on the
// try's buffers (HeadsBuffers), one accumulator of each frame per launch.
constexpr int kHeadsThreads = kSeedThreads;

// the try's centre as integers: the mean-shift position that store_result wrote as floats (exact below 2^24)
__device__ __forceinline__ void centre_of(const dh_result& r, int32_t c[3]) {
    for (int k = 0; k < 3; ++k) c[k] = (int32_t)r.mid_point[k];
}

// Try `round` >= 1: suppress the previous try in the working grid, then seed this one from its first maximum.
__global__ void __launch_bounds__(kHeadsThreads) heads_seed_kernel(FrameBuffers b, HeadsBuffers hb, Geometry g, uint32_t round,
                                                                  uint32_t iterations, const float* __restrict__ frame_k) {
    __shared__ uint32_t s_grid[kPosGridCells];
    __shared__ Best s_red[kHeadsThreads / 32];
    __shared__ unsigned long long s_sum[kHeadsThreads / 32];
    __shared__ uint32_t s_cnt[kHeadsThreads / 32];
    __shared__ float s_uvr[3];
    const uint32_t frame = blockIdx.x, tid = threadIdx.x;
    HeadsState* st = hb.st + frame;
    FrameState* fs = hb.fs + frame;
    if (frame == 0 && tid == 0) hb.fs[0].work_next = 0;  // the centre mean-shift launch hands out its items afresh
    if (!st->searching) {
        if (tid == 0) {
            fs->active = 0;
            fs->box_valid[0] = fs->box_valid[1] = 0;
        }
        return;
    }
    const uint32_t* src = round == 1 ? b.grids + (size_t)frame * (kPosGridCells + kRotGridCells) : hb.grid + (size_t)frame * kPosGridCells;
    for (int i = tid; i < kPosGridCells; i += kHeadsThreads) s_grid[i] = src[i];
    const float* Kf = frame_k + (size_t)frame * kFrameKFloats;
    if (tid == 0) {
        // the previous try's centre in the image: space_to_img clamped like coarse_pos_cell, and R in pixels at its depth
        const dh_result& prev = round == 1 ? b.results[frame] : hb.res[frame];
        float K[9], p2[2];
        load_mat3(Kf, K);
        const float p3[3] = {prev.mid_point[0], prev.mid_point[1], prev.mid_point[2]};
        space_to_img(K, p3, p2);
        const float mx = (p2[0] > 0.0f) ? p2[0] : 0.0f, my = (p2[1] > 0.0f) ? p2[1] : 0.0f;
        s_uvr[0] = (mx < (float)(g.w - 1)) ? mx : (float)(g.w - 1);
        s_uvr[1] = (my < (float)(g.h - 1)) ? my : (float)(g.h - 1);
        const float z = p3[2];
        s_uvr[2] = z > 0.0f ? __fdiv_rn(__fmul_rn(hb.radius, K[0]), z) : 0.0f;
    }
    __syncthreads();
    {
        const float u = s_uvr[0], v = s_uvr[1], r = s_uvr[2], rr = __fmul_rn(r, r);
        const uint32_t gpw = g.w / kGuessGridParts, gph = g.h / kGuessGridParts;
        for (int i = tid; i < kPosGridCells; i += kHeadsThreads) {
            const uint32_t gx = (uint32_t)i % kGuessGridParts, gy = (uint32_t)i / kGuessGridParts;
            // nearest point of the closed cell rectangle, squared distance without fused operations
            const float nx = fminf(fmaxf(u, (float)(gx * gpw)), (float)((gx + 1) * gpw));
            const float ny = fminf(fmaxf(v, (float)(gy * gph)), (float)((gy + 1) * gph));
            const float dx = __fsub_rn(u, nx), dy = __fsub_rn(v, ny);
            if (__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) <= rr) s_grid[i] = 0;
        }
    }
    __syncthreads();
    if (tid == 0 && st->seed_cell < (uint32_t)kPosGridCells) s_grid[st->seed_cell] = 0;
    __syncthreads();
    const Best best = block_argmax(s_grid, kPosGridCells, s_red);  // first maximum, as the reference's arg-max
    if (best.val < hb.min_cell_votes) {
        if (tid == 0) {
            st->searching = 0;
            fs->active = 0;
            fs->box_valid[0] = fs->box_valid[1] = 0;
        }
        return;
    }
    int32_t sm[3];
    float kinv[9];
    load_mat3(Kf + 9, kinv);
    cell_seed(g, b.depth + (size_t)frame * g.h * g.w, best.idx, kinv, s_sum, s_cnt, sm);
    for (int i = tid; i < kPosGridCells; i += kHeadsThreads) hb.grid[(size_t)frame * kPosGridCells + i] = s_grid[i];
    if (tid == 0) {
        st->seed_cell = best.idx;
        for (int k = 0; k < 3; ++k) {
            fs->seed_mid[k] = sm[k];
            fs->box_org[0][k] = (int32_t)((uint32_t)sm[k] - (uint32_t)(kBox / 2));
        }
        fs->box_valid[0] = iterations > 0 ? 1u : 0u;
        fs->box_valid[1] = 0;
        fs->active = 1u;
        fs->n_gate = b.fs[frame].n_gate;  // the centre cube (and its rebuilds) take every gated patch
    }
}

// After the centre of try `round` (round 0: head 0, the pass's own result): the duplicate test, the gated
// patches within R of the centre, and (round >= 1) their coarse rotation grid and the rotation seed.
constexpr int kHeadsPatchSmem = kRotGridCells * 4;
__global__ void __launch_bounds__(kHeadsThreads) heads_patch_kernel(FrameBuffers b, HeadsBuffers hb, Geometry g, ForestDev f,
                                                                   uint32_t round, uint32_t iterations) {
    extern __shared__ __align__(16) uint32_t s_rot[];  // [8000] coarse rotation grid of the kept patches
    __shared__ Best s_red[kHeadsThreads / 32];
    __shared__ uint32_t s_kept;
    const uint32_t frame = blockIdx.x, tid = threadIdx.x, lane = tid & 31u;
    HeadsState* st = hb.st + frame;
    FrameState* fs = hb.fs + frame;
    if (frame == 0 && tid == 0) hb.fs[0].work_next = 0;  // the rotation mean-shift launch hands out its items afresh
    if (round > 0 && !(fs->active & 1u)) return;
    const dh_result& r = round == 0 ? b.results[frame] : hb.res[frame];
    int32_t c[3];
    centre_of(r, c);
    if (round > 0) {
        // a centre within R of an accepted head is a duplicate: integer squared distance against floor(R)^2
        const long long fr = (long long)floorf(hb.radius), lim = fr * fr;
        bool dup = false;
        for (uint32_t a = 0; a < st->n_acc; ++a) {
            const long long dx = (long long)c[0] - st->centre[a][0], dy = (long long)c[1] - st->centre[a][1],
                            dz = (long long)c[2] - st->centre[a][2];
            if (dx * dx + dy * dy + dz * dz <= lim) dup = true;
        }
        if (dup) {
            if (tid == 0) {
                fs->active = 0;
                fs->box_valid[1] = 0;
            }
            return;
        }
    }
    if (tid == 0) s_kept = 0;
    if (round > 0)
        for (int i = tid; i < kRotGridCells; i += kHeadsThreads) s_rot[i] = 0;
    __syncthreads();
    // gated patches within R of the centre: f32 differences, ((dx^2 + dy^2) + dz^2) <= R^2 without fused operations
    const float cx = r.mid_point[0], cy = r.mid_point[1], cz = r.mid_point[2], rr = __fmul_rn(hb.radius, hb.radius);
    const uint32_t ngate = b.fs[frame].n_gate;
    const float4* gated = b.gated + (size_t)frame * g.P;
    float4* kept = hb.gated + (size_t)frame * g.P;
    for (uint32_t i0 = 0; i0 < ngate; i0 += kHeadsThreads) {
        const uint32_t i = i0 + tid;
        bool in = false;
        float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < ngate) {
            p = gated[i];
            const float dx = __fsub_rn(p.x, cx), dy = __fsub_rn(p.y, cy), dz = __fsub_rn(p.z, cz);
            in = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)) <= rr;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, in);
        uint32_t base = 0;
        if (lane == 0 && m) base = atomicAdd(&s_kept, (uint32_t)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (in && round > 0) kept[base + __popc(m & ((1u << lane) - 1u))] = p;
    }
    __syncthreads();
    const uint32_t nkept = s_kept;
    if (round == 0) {
        // head 0: the pass's result, its support and seed cell; the search starts from it
        uint32_t cell = 0xffffffffu;
        if (!(b.fs[frame].has_guess & 1u)) cell = block_argmax(b.grids + (size_t)frame * (kPosGridCells + kRotGridCells), kPosGridCells, s_red).idx;
        if (tid == 0) {
            dh_head h;
            h.pose = r;
            h.support = b.fs[frame].support;
            h.n_patches = nkept;
            h.seed_cell = cell;
            hb.out[(size_t)frame * hb.max_heads] = h;
            hb.n_heads[frame] = 1;
            for (int k = 0; k < 3; ++k) st->centre[0][k] = c[k];
            st->n_acc = 1;
            st->searching = hb.max_heads > 1u ? 1u : 0u;
            st->seed_cell = cell;
            st->n_patches = nkept;
        }
        return;
    }
    // the kept patches' rotation votes into the coarse grid: the leaves' static cell lists (leaf_gate_kernel)
    const uint32_t T = g.n_trees;
    const int32_t* leaf_f = b.leaf + (size_t)frame * T * g.P;
    for (uint32_t i = tid; i < nkept * T; i += kHeadsThreads) {
        const uint32_t t = i / nkept;
        const float4 p = kept[i - t * nkept];
        const int32_t L = (int32_t)((uint32_t)leaf_f[(size_t)t * g.P + __float_as_uint(p.w)] & b.leaf_mask);
        const LeafInfo li = f.leaf_info[L];
        if ((li.flags & kLeafVotes) && (li.flags & kLeafRotOk)) {
            const uint32_t n = li.flags >> kLeafRotCellsShift;
            for (uint32_t j = 0; j < n; ++j) {
                const uint32_t e = __ldg(f.rot_cells + li.vote_start + j);
                atomicAdd(&s_rot[e & ((1u << kRotCellBits) - 1u)], li.valtoadd * (e >> kRotCellBits));
            }
        }
    }
    __syncthreads();
    const Best br = block_argmax(s_rot, kRotGridCells, s_red);  // prediction.rs:733-742 on these patches
    if (tid == 0) {
        const uint32_t rc[3] = {br.idx % 20u, (br.idx % 400u) / 20u, br.idx / 400u};
        for (int k = 0; k < 3; ++k) {
            const double deg = __ddiv_rn(__dadd_rn(__dmul_rn((double)rc[k], 360.0), 180.0), (double)kGuessGridParts);
            fs->seed_rot[k] = __double2int_rz(__ddiv_rn(__dmul_rn(deg, (double)kRotGridParts), 360.0));
            fs->box_org[1][k] = (int32_t)((uint32_t)fs->seed_rot[k] - (uint32_t)(kBox / 2));
        }
        fs->box_valid[1] = iterations > 0 ? 1u : 0u;
        fs->active = 2u;
        fs->n_gate = nkept;  // the rotation cube (and its rebuilds) take the kept patches, in hb.gated
        for (int k = 0; k < 3; ++k) st->centre[st->n_acc][k] = c[k];
        st->n_patches = nkept;
    }
}

// The accepted try of this round becomes the frame's next head.
__global__ void __launch_bounds__(128) heads_commit_kernel(HeadsBuffers hb, uint32_t n) {
    const uint32_t frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= n) return;
    HeadsState* st = hb.st + frame;
    const FrameState* fs = hb.fs + frame;
    if (!(fs->active & 2u)) return;
    dh_head h;
    h.pose = hb.res[frame];
    h.support = fs->support;
    h.n_patches = st->n_patches;
    h.seed_cell = st->seed_cell;
    hb.out[(size_t)frame * hb.max_heads + st->n_acc] = h;
    st->n_acc += 1;
    hb.n_heads[frame] = st->n_acc;
    if (st->n_acc >= hb.max_heads) st->searching = 0;
}

// float -> bfloat16 bit pattern, rounded towards -inf / +inf (exact for values a bfloat16 holds; inf stays inf)
__device__ __forceinline__ uint16_t bf16_down(float x) {
    const uint32_t b = __float_as_uint(x);
    return (uint16_t)(((b >> 31) && (b & 0xffffu) && (b & 0x7f800000u) != 0x7f800000u ? b + 0x10000u : b) >> 16);
}
__device__ __forceinline__ uint16_t bf16_up(float x) {
    const uint32_t b = __float_as_uint(x);
    return (uint16_t)((!(b >> 31) && (b & 0xffffu) && (b & 0x7f800000u) != 0x7f800000u ? b + 0x10000u : b) >> 16);
}

// ================================================================ K5: per-leaf static gates
// estimate_mean_cov (meancov_estimation.rs:359-378) in reference order, one thread per leaf.
// Only the diagonal of the covariance is needed for the trace (entries are independent).
__global__ void __launch_bounds__(128) leaf_gate_kernel(const double* __restrict__ leaf_prob,
                                                        const uint32_t* __restrict__ vote_start,
                                                        const uint32_t* __restrict__ n_votes,
                                                        const float* __restrict__ offsets,
                                                        const double* __restrict__ rotations,
                                                        const uint32_t* __restrict__ rot_bins,
                                                        LeafInfo* __restrict__ out, LeafBox* __restrict__ box_out,
                                                        uint32_t* __restrict__ rot_cells, uint32_t n_leaves) {
    const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_leaves) return;
    const uint32_t v0 = vote_start[l], n = n_votes[l];
    LeafInfo li{v0, n, 0u, 0u};
    if (n > 0) {
        // valtoadd = ((1000.0 * prob) as usize / offsets.len()) as u32   (prediction.rs:594-595)
        const unsigned long long q = __double2ull_rz(__dmul_rn(1000.0, leaf_prob[l]));
        li.valtoadd = (uint32_t)(q / (unsigned long long)n);
        // rotations, f64
        {
            const double* s = rotations + (size_t)v0 * 3;
            double mean[3] = {s[0], s[1], s[2]};
            for (uint32_t i = 1; i < n; ++i)
                for (int k = 0; k < 3; ++k) mean[k] = __dadd_rn(mean[k], s[(size_t)i * 3 + k]);
            const double dn = (double)n;
            for (int k = 0; k < 3; ++k) mean[k] = __ddiv_rn(mean[k], dn);
            double cov[3];
            for (int k = 0; k < 3; ++k) {
                const double d = __dsub_rn(s[k], mean[k]);
                cov[k] = __dmul_rn(d, d);
            }
            for (uint32_t i = 1; i < n; ++i)
                for (int k = 0; k < 3; ++k) {
                    const double d = __dsub_rn(s[(size_t)i * 3 + k], mean[k]);
                    cov[k] = __dadd_rn(cov[k], __dmul_rn(d, d));
                }
            const double dn1 = (double)(n - 1);
            double tr = 0.0;  // trace(): fold from 0.0 (meancov_estimation.rs:260-265)
            for (int k = 0; k < 3; ++k) tr = __dadd_rn(tr, __ddiv_rn(cov[k], dn1));
            if (tr <= kMaxVarianceRot) li.flags |= kLeafRotOk;  // NaN (n == 1) -> false
        }
        // offsets, f32 with the divisors cast f64 -> f32 (meancov_estimation.rs:290-304)
        {
            const float* s = offsets + (size_t)v0 * 3;
            float mean[3] = {s[0], s[1], s[2]};
            for (uint32_t i = 1; i < n; ++i)
                for (int k = 0; k < 3; ++k) mean[k] = __fadd_rn(mean[k], s[(size_t)i * 3 + k]);
            const float dn = (float)(double)n;
            for (int k = 0; k < 3; ++k) mean[k] = __fdiv_rn(mean[k], dn);
            float cov[3];
            for (int k = 0; k < 3; ++k) {
                const float d = __fsub_rn(s[k], mean[k]);
                cov[k] = __fmul_rn(d, d);
            }
            for (uint32_t i = 1; i < n; ++i)
                for (int k = 0; k < 3; ++k) {
                    const float d = __fsub_rn(s[(size_t)i * 3 + k], mean[k]);
                    cov[k] = __fadd_rn(cov[k], __fmul_rn(d, d));
                }
            const float dn1 = (float)(double)(n - 1);
            float tr = 0.0f;
            for (int k = 0; k < 3; ++k) tr = __fadd_rn(tr, __fdiv_rn(cov[k], dn1));
            if (tr <= kMaxVarianceOffset) li.flags |= kLeafOffOk;
        }
        // the leaf casts votes at all: prob > 0 (prediction.rs:590), a non-zero weight, a spread gate open
        if (leaf_prob[l] > 0.0 && li.valtoadd != 0u && (li.flags & (kLeafRotOk | kLeafOffOk))) li.flags |= kLeafVotes;
    }
    out[l] = li;
    // bounding boxes of the leaf's votes (box_build skips leaves that cannot reach a cube) and
    // the coarse rotation cell of every vote: rough = r * 20 / 120 per axis, dense index
    // z*400 + y*20 + x (prediction.rs:630-636)
    float omin[3] = {0.0f, 0.0f, 0.0f}, omax[3] = {0.0f, 0.0f, 0.0f};
    uint8_t rmin[3] = {0, 0, 0}, rmax[3] = {0, 0, 0};
    uint32_t n_cells = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t bins = rot_bins[v0 + i];
        uint32_t q[3];
        for (int k = 0; k < 3; ++k) {
            const float o = offsets[(size_t)(v0 + i) * 3 + k];
            const uint8_t r = (uint8_t)((bins >> (8 * k)) & 0xffu);
            if (i == 0 || o < omin[k]) omin[k] = o;
            if (i == 0 || o > omax[k]) omax[k] = o;
            if (!isfinite(o) || !isfinite(omin[k])) {  // stays open once a non-finite offset was seen
                omin[k] = -INFINITY;
                omax[k] = INFINITY;
            }
            if (i == 0 || r < rmin[k]) rmin[k] = r;
            if (i == 0 || r > rmax[k]) rmax[k] = r;
            q[k] = (uint32_t)r * kGuessGridParts / kRotGridParts;
        }
        // compact list of the leaf's cells: (cell | votes in it << 13) in the first n_cells slots of its
        // range.  Short lists are searched linearly; a leaf with very many votes keeps one entry per vote.
        const uint32_t cell = q[2] * 400u + q[1] * 20u + q[0];
        uint32_t j = n_cells;
        if (n <= 1024u)
            for (j = 0; j < n_cells; ++j)
                if ((rot_cells[v0 + j] & ((1u << kRotCellBits) - 1u)) == cell && (rot_cells[v0 + j] >> kRotCellBits) < kRotCellMaxCount) break;
        if (j < n_cells) rot_cells[v0 + j] += 1u << kRotCellBits;
        else rot_cells[v0 + n_cells++] = cell | (1u << kRotCellBits);
    }
    LeafBox bx;
    bx.vote_start = v0;
    bx.n_votes_flags = n | ((li.flags & 7u) << 24);
    bx.valtoadd = li.valtoadd;
    bx.rmin[0] = rmin[0]; bx.rmin[1] = rmin[1]; bx.rmin[2] = rmin[2];
    bx.rmax0 = rmax[0]; bx.rmax1 = rmax[1]; bx.rmax2 = rmax[2];
    bx.omin0 = bf16_down(omin[0]); bx.omin1 = bf16_down(omin[1]); bx.omin2 = bf16_down(omin[2]);
    bx.omax[0] = bf16_up(omax[0]); bx.omax[1] = bf16_up(omax[1]); bx.omax[2] = bf16_up(omax[2]);
    bx.spare = 0;
    box_out[l] = bx;
    out[l].flags = li.flags | (n_cells << kLeafRotCellsShift);
}

// ================================================================ next-row back-ends on the same front-end
// The 2-D back ends work on a chunk of F frames per launch: the frame index comes from the grid and
// every per-frame buffer is [F][h][w] (leaf ids [F][T][P], as the traversal writes them).
//
// predict_mask (prediction.rs:850-905): per non-background patch, mean prob -> u8, splat to a
// stepwidth^2 block.  Patches are visited in raster order by the reference and later patches
// overwrite earlier ones; blocks of distinct patches never overlap (block origin = centre - s/2,
// size s, centres s apart), so the order is irrelevant.  One thread per (frame, patch).
__global__ void __launch_bounds__(256) mask_kernel(FrameBuffers b, Geometry g, const double* __restrict__ leaf_prob,
                                                   uint8_t* __restrict__ mask) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x, frame = blockIdx.y;
    if (p >= g.P) return;
    const int T = (int)g.n_trees;
    const int32_t* leaf = b.leaf + (size_t)frame * g.n_trees * g.P;
    mask += (size_t)frame * g.w * g.h;
    if (leaf[p] < 0) return;
    double s = 0.0;
    for (int t = 0; t < T; ++t) s = __dadd_rn(s, __ldg(leaf_prob + ((uint32_t)leaf[(size_t)t * g.P + p] & b.leaf_mask)));
    const double prob = __ddiv_rn(s, (double)T);
    const double scaled = __dmul_rn(prob, 255.0);
    // `as u8`: saturating, NaN -> 0
    const uint8_t pv = !(scaled > 0.0) ? 0 : (scaled >= 255.0 ? 255 : (uint8_t)__double2uint_rz(scaled));
    const uint32_t gx = p % g.npx, gy = p / g.npx;
    const uint32_t x = g.left_w + gx * g.stride, y = g.left_h + gy * g.stride;
    const uint32_t sw = g.stride, half = sw / 2;
    for (uint32_t j = 0; j < sw; ++j)
        for (uint32_t i = 0; i < sw; ++i) {
            if (x + i < half || y + j < half) continue;
            if (x + i - half >= g.w || y + j - half >= g.h) continue;
            mask[(size_t)(y + j - half) * g.w + (x + i - half)] = pv;
        }
}

// predict_mask for the passes of dh_predict_tracks_mask, whose frames are scattered over the output:
// slot j of a pass is output frame slots[j].frame (slots != nullptr) or frame0 + j * frame_step.  A
// memset of the chunk cannot clear scattered frames, so this writer stores EVERY pixel: a CTA owns a
// tile of kTrackMaskTileW x kTrackMaskTileH pixels of one frame, settles the u8 of every patch whose
// block meets the tile in shared memory (the arithmetic of mask_kernel; 0 for background), then
// gives each pixel the value of the block that holds it, or 0 outside every block.  Pixel X lies in
// the block of patch column gx = (X + s/2 - left_w) / s iff X + s/2 >= left_w and gx < npx (blocks
// are s wide, s apart, and start at the patch centre - s/2), the same for rows.
constexpr uint32_t kTrackMaskTileW = 128, kTrackMaskTileH = 8;
__global__ void __launch_bounds__(256) track_mask_kernel(FrameBuffers b, Geometry g, const double* __restrict__ leaf_prob,
                                                         const TrackSlot* __restrict__ slots, uint32_t frame0, uint32_t frame_step,
                                                         uint8_t* __restrict__ mask) {
    // at most (tile - 1) / s + 2 block columns / rows meet a tile
    __shared__ uint8_t pv_s[(kTrackMaskTileW + 1) * (kTrackMaskTileH + 1)];
    const uint32_t j = blockIdx.z, x0 = blockIdx.x * kTrackMaskTileW, y0 = blockIdx.y * kTrackMaskTileH;
    const uint32_t s = g.stride, half = s / 2;
    const uint32_t x1 = min(x0 + kTrackMaskTileW, g.w) - 1u, y1 = min(y0 + kTrackMaskTileH, g.h) - 1u;  // last pixel of the tile
    // block columns [cx0, cx1) and rows [cy0, cy1) that meet the tile
    const uint32_t cx0 = x0 + half >= g.left_w ? (x0 + half - g.left_w) / s : 0u;
    const uint32_t cx1 = x1 + half >= g.left_w ? min((x1 + half - g.left_w) / s + 1u, g.npx) : 0u;
    const uint32_t cy0 = y0 + half >= g.left_h ? (y0 + half - g.left_h) / s : 0u;
    const uint32_t cy1 = y1 + half >= g.left_h ? min((y1 + half - g.left_h) / s + 1u, g.npy) : 0u;
    const uint32_t ncx = cx1 > cx0 ? cx1 - cx0 : 0u, ncy = cy1 > cy0 ? cy1 - cy0 : 0u;
    const int T = (int)g.n_trees;
    const int32_t* leaf = b.leaf + (size_t)j * g.n_trees * g.P;
    for (uint32_t k = threadIdx.x; k < ncx * ncy; k += blockDim.x) {
        const uint32_t p = (cy0 + k / ncx) * g.npx + cx0 + k % ncx;
        uint8_t pv = 0;
        if (leaf[p] >= 0) {
            double sum = 0.0;
            for (int t = 0; t < T; ++t) sum = __dadd_rn(sum, __ldg(leaf_prob + ((uint32_t)leaf[(size_t)t * g.P + p] & b.leaf_mask)));
            const double scaled = __dmul_rn(__ddiv_rn(sum, (double)T), 255.0);
            pv = !(scaled > 0.0) ? 0 : (scaled >= 255.0 ? 255 : (uint8_t)__double2uint_rz(scaled));
        }
        pv_s[k] = pv;
    }
    __syncthreads();
    const uint32_t frame = slots ? (uint32_t)slots[j].frame : frame0 + j * frame_step;
    uint8_t* out = mask + (size_t)frame * g.w * g.h;
    const uint32_t lane = threadIdx.x & 31u, row = threadIdx.x >> 5;  // a warp stores 32 adjacent bytes of one row
    const uint32_t y = y0 + row;
    if (y > y1) return;
    const uint32_t gy = (y + half - g.left_h) / s;
    const bool in_y = y + half >= g.left_h && gy < g.npy;
    for (uint32_t x = x0 + lane; x <= x1; x += 32u) {
        const uint32_t gx = (x + half - g.left_w) / s;
        uint8_t v = 0;
        if (in_y && x + half >= g.left_w && gx < g.npx) v = pv_s[(gy - cy0) * ncx + (gx - cx0)];
        out[(size_t)y * g.w + x] = v;
    }
}

// build_hough_image before the blur (prediction.rs:760-841).  u16 wrap-around adds are done as
// u32 atomics into the frame's accumulator and truncated by the reader (sum mod 2^16 is the same
// either way).  One thread per (frame, tree, patch).  kFrameK: the frame's K and K^-1 come from
// frame_k, loaded into registers by the threads that pass the leaf tests (most return before).
template <bool kFrameK>
__global__ void __launch_bounds__(256) hough_image_kernel(FrameBuffers b, Geometry g, ForestDev f, uint32_t* __restrict__ acc,
                                                         const float* __restrict__ frame_k) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x, frame = blockIdx.y;
    const uint32_t T = g.n_trees;
    if (idx >= g.P * T) return;
    const uint32_t p = idx % g.P, t = idx / g.P;
    const int32_t* leaf = b.leaf + (size_t)frame * T * g.P;
    if (leaf[p] < 0) return;  // background patch: decided on the slice of tree 0 (the only one prefilled with -1)
    const int32_t L = (int32_t)((uint32_t)leaf[(size_t)t * g.P + p] & b.leaf_mask);
    const double lp = f.leaf_prob[L];
    if (!(lp >= 0.95)) return;                                             // :805
    const uint32_t v0 = f.leaf_info[L].vote_start, n = f.leaf_info[L].n_votes;
    if (n == 0) return;
    const uint32_t valtoadd = (uint32_t)(uint16_t)(__double2ull_rz(__dmul_rn(255.0, lp)) / n);  // :807-808
    const uint32_t gx = p % g.npx, gy = p / g.npx;
    const uint32_t x = g.left_w + gx * g.stride, y = g.left_h + gy * g.stride;
    const size_t frame_px = (size_t)g.w * g.h;
    acc += (size_t)frame * frame_px;
    float p3[3], fk[9], fkinv[9];
    if (kFrameK) {
        load_mat3(frame_k + (size_t)frame * kFrameKFloats, fk);
        load_mat3(frame_k + (size_t)frame * kFrameKFloats + 9, fkinv);
    }
    img_to_space(kFrameK ? fkinv : g.Kinv, (float)x, (float)y, (float)b.depth[(size_t)frame * frame_px + (size_t)y * g.w + x], p3);
    for (uint32_t k = 0; k < n; ++k) {
        float np[3], p2[2];
        const float4 o = f.offsets[v0 + k];
        np[0] = __fsub_rn(p3[0], o.x);
        np[1] = __fsub_rn(p3[1], o.y);
        np[2] = __fsub_rn(p3[2], o.z);
        space_to_img(kFrameK ? fk : g.K, np, p2);
        const int nx = __float2int_rz(p2[0]), ny = __float2int_rz(p2[1]);  // :816
        if (nx < 0 || (uint32_t)nx >= g.w || ny < 0 || (uint32_t)ny >= g.h) continue;
        atomicAdd(&acc[(size_t)ny * g.w + nx], valtoadd);
    }
}
// the raw vote image: the low 16 bits of the u32 sums
__global__ void narrow_u16_kernel(const uint32_t* __restrict__ in, uint16_t* __restrict__ out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint16_t)(in[i] & 0xffffu);
}

// ---- the blur of build_hough_image (prediction.rs:844 gaussian_blur_f32, imageproc 0.12: restated, unpinned)
// Separable: a horizontal pass over the u16 vote image, then a vertical pass over its u16 result.
// Per output pixel acc = 0; for the taps in order acc = acc + (float)pixel * k[i] (no FMA); the
// coordinate is clamped to the image; the result is stored as u16 by truncation with saturation
// (Clamp<f32> for u16).  One thread per output pixel; the pixels a block's outputs need are staged
// in shared memory (a row segment of 128 + 2r pixels, or a column segment of 32 + 2r rows x 32 columns).
// The frame is blockIdx.z.  The horizontal pass reads the u32 vote sums and narrows them to u16 on
// the load, so the blurred path has no separate narrowing pass.
__device__ __forceinline__ uint16_t clamp_f32_u16(float x) {
    if (x < 65535.0f) return x > 0.0f ? (uint16_t)__float2uint_rz(x) : (uint16_t)0;
    return 65535;
}
constexpr int kBlurHx = 128, kBlurHy = 4;   // horizontal pass: outputs per block
constexpr int kBlurVx = 32, kBlurVy = 32;   // vertical pass
__global__ void __launch_bounds__(kBlurHx * kBlurHy) blur_h_kernel(const uint32_t* __restrict__ in, uint16_t* __restrict__ out, uint32_t w,
                                                                    uint32_t h, const float* __restrict__ k, int radius) {
    extern __shared__ uint16_t s_px[];  // [kBlurHy][kBlurHx + 2 radius]
    const int span = kBlurHx + 2 * radius;
    const int x0 = (int)blockIdx.x * kBlurHx, y = (int)(blockIdx.y * kBlurHy + threadIdx.y);
    const size_t frame_px = (size_t)w * h;
    in += blockIdx.z * frame_px;
    out += blockIdx.z * frame_px;
    uint16_t* row = s_px + threadIdx.y * span;
    if (y < (int)h)
        for (int i = threadIdx.x; i < span; i += kBlurHx) {
            const int xs = min(max(x0 + i - radius, 0), (int)w - 1);
            row[i] = (uint16_t)(in[(size_t)y * w + xs] & 0xffffu);
        }
    __syncthreads();
    const int x = x0 + (int)threadIdx.x;
    if (y >= (int)h || x >= (int)w) return;
    float acc = 0.0f;
    for (int i = 0; i <= 2 * radius; ++i) acc = __fadd_rn(acc, __fmul_rn((float)row[threadIdx.x + i], __ldg(k + i)));
    out[(size_t)y * w + x] = clamp_f32_u16(acc);
}
// out: the blurred image (nullptr: not written).  keys != nullptr: the arg-max of
// predict_parameter_from2dhough (prediction.rs:343-367) rides along: Iterator::max_by_key over the
// pixels in index order returns the LAST of equal maxima, which is the largest
// (value << 32) | pixel index; every block folds its pixels to one such key and the frame's key is
// the 64-bit atomicMax over the blocks (keys[frame] starts at 0, below every pixel's key).
__global__ void __launch_bounds__(kBlurVx * kBlurVy) blur_v_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint32_t w,
                                                                    uint32_t h, const float* __restrict__ k, int radius,
                                                                    unsigned long long* __restrict__ keys) {
    extern __shared__ uint16_t s_px[];  // [kBlurVy + 2 radius][kBlurVx]
    __shared__ unsigned long long s_key[kBlurVx * kBlurVy / 32];
    const int span = kBlurVy + 2 * radius;
    const int x = (int)(blockIdx.x * kBlurVx + threadIdx.x), y0 = (int)blockIdx.y * kBlurVy;
    const size_t frame_px = (size_t)w * h;
    in += blockIdx.z * frame_px;
    if (x < (int)w)
        for (int i = threadIdx.y; i < span; i += kBlurVy) {
            const int ys = min(max(y0 + i - radius, 0), (int)h - 1);
            s_px[i * kBlurVx + threadIdx.x] = in[(size_t)ys * w + x];
        }
    __syncthreads();
    const int y = y0 + (int)threadIdx.y;
    const bool inside = y < (int)h && x < (int)w;
    unsigned long long key = 0;
    if (inside) {
        float acc = 0.0f;
        for (int i = 0; i <= 2 * radius; ++i) acc = __fadd_rn(acc, __fmul_rn((float)s_px[(threadIdx.y + i) * kBlurVx + threadIdx.x], __ldg(k + i)));
        const uint16_t v = clamp_f32_u16(acc);
        const uint32_t idx = (uint32_t)y * w + (uint32_t)x;
        if (out) out[blockIdx.z * frame_px + idx] = v;
        key = ((unsigned long long)v << 32) | idx;
    }
    if (!keys) return;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, key, d);
        key = o > key ? o : key;
    }
    const uint32_t tid = threadIdx.y * kBlurVx + threadIdx.x;
    if ((tid & 31u) == 0) s_key[tid >> 5] = key;
    __syncthreads();
    if (tid < 32) {
        key = s_key[tid];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, key, d);
            key = o > key ? o : key;
        }
        if (tid == 0) atomicMax(keys + blockIdx.z, key);
    }
}
// predict_parameter_from2dhough (prediction.rs:343-367) from the frames' arg-max keys: z = the
// depth at that pixel and the back-projection of (x, y, z); rotation 0, bounding box 0.  One thread per frame.
// kFrameK: the back-projection uses the frame's K^-1 from frame_k.
template <bool kFrameK>
__global__ void hough2d_pose_kernel(const unsigned long long* __restrict__ keys, const uint16_t* __restrict__ depth, Geometry g,
                                    uint32_t n_frames, dh_result* __restrict__ out, const float* __restrict__ frame_k) {
    const uint32_t frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= n_frames) return;
    const uint32_t w = g.w, bi = (uint32_t)(keys[frame] & 0xffffffffull);
    const uint32_t x = bi % w, y = bi / w;
    float p[3], kinv[9];
    if (kFrameK) load_mat3(frame_k + (size_t)frame * kFrameKFloats + 9, kinv);
    img_to_space(kFrameK ? kinv : g.Kinv, (float)x, (float)y, (float)depth[(size_t)frame * w * g.h + (size_t)y * w + x], p);
    dh_result& r = out[frame];
    r.mid_point[0] = p[0]; r.mid_point[1] = p[1]; r.mid_point[2] = p[2];
    r._pad = 0;
    r.rotation[0] = r.rotation[1] = r.rotation[2] = 0.0;
    r.bounding_box[0] = r.bounding_box[1] = r.bounding_box[2] = r.bounding_box[3] = 0;
}

// ================================================================ Biwi run-length decode
// read_depth (biwi.rs:81-103): [u32 w][u32 h] then, until w*h pixels are covered,
// [u32 n_empty][u32 n_full][n_full x u16].  The position of a run header depends on every header
// before it, so ONE thread has to follow the chain; everything else is parallel.  One CTA per
// frame, the file staged through shared memory in 16 KB pieces (coalesced 4-byte loads); per piece
//   1. thread 0 follows the chain inside shared memory and only notes the header positions
//      (load n_full, store the position, advance);
//   2. all threads: a block-wide prefix sum of n_empty + n_full (saturating at w*h + 1) gives
//      every run its first pixel; the reference's failure conditions are checked per run, the
//      first failing run deciding; runs longer than 2048 pixels are set aside;
//   3. the warps copy the runs' pixels (from the staged bytes where they lie inside the piece),
//      the long runs with the whole CTA.
// The frame was zeroed beforehand, so empty runs cost nothing.  Damaged files set the frame's
// status: 1 truncated (the reference's UnexpectedEof), 2 a run past the last pixel (its `unwrap`
// panic; also reported when the same run is truncated as well), 3 header is not w x h.
constexpr int kRleThreads = 256;
constexpr int kRlePieceWords = 4096;    // 16 KB of file per round
constexpr int kRleRuns = 2048;          // a piece holds at most 2048 headers
constexpr int kRlePerThread = kRleRuns / kRleThreads;
constexpr uint32_t kRleLongRun = 2048;  // pixels: longer runs are copied by the whole CTA
constexpr uint32_t kRleLongCap = 16;    // a 16 KB piece cannot start more than 4 of them

__device__ __forceinline__ uint32_t rle_u32(const uint16_t* p16, uint32_t i) { return (uint32_t)p16[i] | ((uint32_t)p16[i + 1] << 16); }

__global__ void __launch_bounds__(kRleThreads) biwi_decode_kernel(const uint8_t* __restrict__ blob,
                                                                  const unsigned long long* __restrict__ offsets,
                                                                  const unsigned long long* __restrict__ ends,
                                                                  unsigned long long blob_base, uint32_t w, uint32_t h,
                                                                  uint16_t* __restrict__ out, uint32_t* __restrict__ status) {
    __shared__ __align__(16) uint32_t s_piece[kRlePieceWords + 2];
    __shared__ uint32_t s_run_pos[kRleRuns];   // byte position of the run's header inside the file
    __shared__ uint32_t s_run_p[kRleRuns];     // pixels covered before the run (saturating at npx + 1)
    __shared__ uint32_t s_warp_tot[kRleThreads / 32];
    __shared__ uint32_t s_long[kRleLongCap];
    __shared__ uint32_t s_nrun, s_pos, s_p, s_nlong, s_err, s_done, s_end_run, s_bad_run;
    const uint32_t frame = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (offsets[frame] == ~0ull) return;  // no file for this frame: its pixels arrived another way
    // frame i occupies [offsets[i], offsets[i+1]), or [offsets[i], ends[i]) when the files do not follow one another
    const unsigned long long o0 = offsets[frame] - blob_base, o1 = (ends ? ends[frame] : offsets[frame + 1]) - blob_base;
    const uint8_t* file = blob + o0;                  // 4-byte aligned (checked on the host)
    const uint32_t len = (uint32_t)(o1 - o0);
    const uint32_t npx = w * h, cap = npx + 1u;       // npx <= 2^30 (checked on the host): sums of two capped values fit u32
    uint16_t* dst = out + (size_t)frame * npx;
    const uint16_t* piece16 = reinterpret_cast<const uint16_t*>(s_piece);
    if (tid == 0) {
        s_err = 0;
        s_done = npx == 0u ? 1u : 0u;
        s_pos = 8;         // byte position of the next run header
        s_p = 0;           // pixels covered so far
        if (len < 8u) s_err = 1;
        else if (reinterpret_cast<const uint32_t*>(file)[0] != w || reinterpret_cast<const uint32_t*>(file)[1] != h) s_err = 3;
    }
    for (;;) {
        __syncthreads();
        if (s_err || s_done) break;
        const uint32_t pos0 = s_pos, p0 = s_p;
        if (pos0 > len || len - pos0 < 8u) {          // read_u32 of the next header hits the end of the file (biwi.rs:90,94)
            if (tid == 0) s_err = 1;
            continue;
        }
        // ---- stage the piece that starts at the next header
        const uint32_t base = pos0 & ~3u;
        const uint32_t avail = min((uint32_t)kRlePieceWords + 2u, (len - base + 3u) / 4u);  // padding up to 4 bytes is readable
        for (uint32_t i = tid; i < avail; i += kRleThreads) s_piece[i] = __ldg(reinterpret_cast<const uint32_t*>(file + base) + i);
        if (tid == 0) {
            s_nlong = 0;
            s_end_run = 0xffffffffu;
            s_bad_run = 0xffffffffu;
        }
        __syncthreads();
        // ---- 1. thread 0 follows the chain (headers are only 2-byte aligned: n_full is read as two halves)
        if (tid == 0) {
            uint32_t pos = pos0, n = 0;
            const uint32_t lim = min(base + (uint32_t)kRlePieceWords * 4u, len);  // a header must end inside the piece and the file
            while (pos + 8u <= lim && n < (uint32_t)kRleRuns) {
                const uint32_t nf = rle_u32(piece16, (pos - base + 4u) >> 1);
                s_run_pos[n++] = pos;
                if (nf > ((len - pos - 8u) >> 1)) {   // its pixels run past the end of the file: the chain ends here
                    pos = 0xffffffffu;
                    break;
                }
                pos += 8u + 2u * nf;
            }
            s_nrun = n;
            s_pos = pos;
        }
        __syncthreads();
        const uint32_t nrun = s_nrun;
        // ---- 2. first pixel of every run: block-wide exclusive scan of n_empty + n_full
        uint32_t loc[kRlePerThread], tot = 0;
#pragma unroll
        for (int j = 0; j < kRlePerThread; ++j) {
            const uint32_t r = tid * kRlePerThread + (uint32_t)j;
            uint32_t c = 0;
            if (r < nrun) {
                const uint32_t hp = (s_run_pos[r] - base) >> 1;
                c = min(min(rle_u32(piece16, hp), cap) + min(rle_u32(piece16, hp + 2u), cap), cap);
            }
            loc[j] = tot;
            tot = min(tot + c, cap);
        }
        uint32_t incl = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl = min(incl + nb, cap);
        }
        if (lane == 31u) s_warp_tot[warp] = incl;
        __syncthreads();
        uint32_t before = p0;
        for (uint32_t k = 0; k < warp; ++k) before = min(before + s_warp_tot[k], cap);
        // exclusive prefix of this lane inside the warp: redo it from the neighbour's inclusive value (saturation forbids a subtraction)
        const uint32_t left = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane) before = min(before + left, cap);
#pragma unroll
        for (int j = 0; j < kRlePerThread; ++j) {
            const uint32_t r = tid * kRlePerThread + (uint32_t)j;
            if (r < nrun) s_run_p[r] = min(before + loc[j], cap);
        }
        __syncthreads();
        // ---- the reference's events per run, in its order; the first run at or past the last pixel ends the frame
        for (uint32_t r = tid; r < nrun; r += kRleThreads) {
            const uint32_t p = s_run_p[r];
            if (p >= npx) {                           // biwi.rs:89: the loop ended before this header would be read
                atomicMin(&s_end_run, r);
                continue;
            }
            const uint32_t pos = s_run_pos[r], hp = (pos - base) >> 1;
            const uint32_t ne = rle_u32(piece16, hp), nf = rle_u32(piece16, hp + 2u);
            const uint32_t room = npx - p;
            uint32_t e = 0;
            if (ne > room || nf > room - ne) e = 2;                    // `it.next().unwrap()` past the last pixel (biwi.rs:92,97)
            else if (nf > ((len - pos - 8u) >> 1)) e = 1;              // read_u16 hits the end of the file (biwi.rs:96)
            if (e) atomicMin(&s_bad_run, (r << 2) | e);
            else if (nf > kRleLongRun) {
                const uint32_t k = atomicAdd(&s_nlong, 1u);
                if (k < kRleLongCap) s_long[k] = r;
            }
        }
        __syncthreads();
        const uint32_t end_run = min(nrun, s_end_run);
        const bool failed = s_bad_run != 0xffffffffu && (s_bad_run >> 2) < end_run;
        // ---- 3. copy: one warp per run; pixels are 2-byte aligned in the file
        if (!failed) {
            for (uint32_t r = warp; r < end_run; r += kRleThreads / 32) {
                const uint32_t pos = s_run_pos[r], hp = (pos - base) >> 1;
                const uint32_t ne = rle_u32(piece16, hp), nf = rle_u32(piece16, hp + 2u);
                if (nf > kRleLongRun) continue;
                const uint32_t src = pos + 8u, d0 = s_run_p[r] + ne;
                const bool staged = src + 2u * nf <= base + avail * 4u;  // whole run inside the staged piece
                const uint16_t* px = reinterpret_cast<const uint16_t*>(file + src);
                const uint32_t so = (src - base) >> 1;
                for (uint32_t i = lane; i < nf; i += 32u) dst[d0 + i] = staged ? piece16[so + i] : __ldg(px + i);
            }
            const uint32_t nlong = min(s_nlong, kRleLongCap);
            for (uint32_t k = 0; k < nlong; ++k) {
                const uint32_t r = s_long[k];
                if (r >= end_run) continue;
                const uint32_t pos = s_run_pos[r], hp = (pos - base) >> 1;
                const uint32_t ne = rle_u32(piece16, hp), nf = rle_u32(piece16, hp + 2u);
                const uint16_t* px = reinterpret_cast<const uint16_t*>(file + pos + 8u);
                const uint32_t d0 = s_run_p[r] + ne;
                for (uint32_t i = tid; i < nf; i += kRleThreads) dst[d0 + i] = __ldg(px + i);
            }
        }
        __syncthreads();
        if (tid == 0) {
            if (failed) s_err = s_bad_run & 3u;
            else if (s_end_run != 0xffffffffu) s_done = 1;
            else {
                // pixels covered after this round's runs
                uint32_t p = p0;
                for (uint32_t k = 0; k < kRleThreads / 32; ++k) p = min(p + s_warp_tot[k], cap);
                s_p = p;
                if (p >= npx) s_done = 1;
            }
        }
    }
    if (tid == 0) status[frame] = s_err;
}

// ================================================================ debug: dump one accumulator cube
__global__ void box_dump_kernel(FrameBuffers b, uint32_t frame, int which, int32_t* keys_out, uint32_t* vals_out,
                                unsigned long long* count) {
    const FrameState* fs = b.fs + frame;
    if (!fs->box_valid[which]) return;
    const uint32_t* box = b.cubes + ((size_t)frame * 2 + (uint32_t)which) * kBoxCells;
    const int32_t* org = fs->box_org[which];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < (uint32_t)kBoxCells; i += gridDim.x * blockDim.x) {
        const uint32_t v = box[i];
        if (!v) continue;
        const unsigned long long o = atomicAdd(count, 1ull);
        if (keys_out) {
            keys_out[o * 3 + 0] = org[0] + (int32_t)(i / (kBox * kBox));  // z fastest
            keys_out[o * 3 + 1] = org[1] + (int32_t)((i / kBox) % kBox);
            keys_out[o * 3 + 2] = org[2] + (int32_t)(i % kBox);
            vals_out[o] = v;
        }
    }
}

// ================================================================ seeded sequences
// examples/live_prediction.rs:75-88: frame t of a sequence is predicted with the pose of frame
// t - 1 as its seeds — the centre only if its z exceeds a threshold (500 mm there; latest_midp starts
// at 0, so the first frame has no centre seed), the rotation whenever there was a previous frame.
// One thread per sequence copies the previous pass's result into the frame state the seed kernel reads.
__global__ void __launch_bounds__(128) seq_guess_kernel(FrameState* __restrict__ fs, const dh_result* __restrict__ prev, uint32_t n,
                                                        float min_seed_z) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const dh_result r = prev[i];
    uint32_t g = 2u;
    if (r.mid_point[2] > min_seed_z) {
        g |= 1u;
        fs[i].midp_guess[0] = r.mid_point[0];
        fs[i].midp_guess[1] = r.mid_point[1];
        fs[i].midp_guess[2] = r.mid_point[2];
    }
    fs[i].rot_guess[0] = r.rotation[0];
    fs[i].rot_guess[1] = r.rotation[1];
    fs[i].rot_guess[2] = r.rotation[2];
    fs[i].has_guess = g;
}

// ================================================================ tracks (dh_predict_tracks)
// One thread per slot of a pass: the slot's frame state (zero but for the seeds, as dh_predict's) and
// its row of the K / K^-1 table.  A track's first frame takes the caller's seeds; every later frame
// the previous pass's result at the planned position, by the rule of seq_guess_kernel.  Biwi passes
// also fold the decode status of the slot into the lowest bad global frame index (index << 2 | code).
__global__ void __launch_bounds__(128) track_guess_kernel(FrameState* __restrict__ fs, float* __restrict__ frame_k,
                                                          const TrackSlot* __restrict__ slots, const TrackArgs* __restrict__ tracks,
                                                          const dh_result* __restrict__ prev, uint32_t n, float min_seed_z,
                                                          const uint32_t* __restrict__ status, unsigned long long* __restrict__ bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const TrackSlot s = slots[i];
    const TrackArgs& a = tracks[s.track];
    FrameState st = {};
    if (s.prev < 0) {
        st.has_guess = a.has_guess;
        if (a.has_guess & 1u)
            for (int k = 0; k < 3; ++k) st.midp_guess[k] = a.midp_guess[k];
        if (a.has_guess & 2u)
            for (int k = 0; k < 3; ++k) st.rot_guess[k] = a.rot_guess[k];
    } else {
        const dh_result r = prev[s.prev];
        st.has_guess = 2u;
        if (r.mid_point[2] > min_seed_z) {
            st.has_guess |= 1u;
            for (int k = 0; k < 3; ++k) st.midp_guess[k] = r.mid_point[k];
        }
        for (int k = 0; k < 3; ++k) st.rot_guess[k] = r.rotation[k];
    }
    fs[i] = st;
    for (int k = 0; k < 18; ++k) frame_k[(size_t)i * 18 + k] = a.K[k];
    if (status && status[i]) atomicMin(bad, ((unsigned long long)(uint32_t)s.frame << 2) | (status[i] & 3u));
}

// Device-resident frames of a pass: frame slots[f].frame of src into slot f of dst, 16 bytes per load
// when every frame starts 16-byte aligned (else 2).  blockIdx.y = slot.
__global__ void __launch_bounds__(256) track_gather_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ dst,
                                                           const TrackSlot* __restrict__ slots, size_t frame_px, uint32_t vec) {
    const uint32_t f = blockIdx.y;
    const uint16_t* s = src + (size_t)(uint32_t)slots[f].frame * frame_px;
    uint16_t* d = dst + (size_t)f * frame_px;
    const size_t step = (size_t)gridDim.x * blockDim.x, i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec) {
        const uint4* s4 = reinterpret_cast<const uint4*>(s);
        uint4* d4 = reinterpret_cast<uint4*>(d);
        for (size_t i = i0; i < frame_px / 8; i += step) d4[i] = __ldg(s4 + i);
    } else {
        for (size_t i = i0; i < frame_px; i += step) d[i] = __ldg(s + i);
    }
}

// ================================================================ work counters of a pass
__global__ void __launch_bounds__(256) counters_kernel(const FrameState* __restrict__ fs, uint32_t n_frames,
                                                       unsigned long long* __restrict__ out, uint32_t P, uint32_t T) {
    unsigned long long v[DH_N_COUNTERS];
    for (int k = 0; k < DH_N_COUNTERS; ++k) v[k] = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_frames; i += gridDim.x * blockDim.x) {
        const FrameState& f = fs[i];
        v[0] += 1;
        v[1] += P;
        v[2] += f.n_valid;
        v[3] += (unsigned long long)f.n_valid * T;
        v[4] += f.node_visits;
        v[5] += f.n_gate;
        v[6] += f.n_chits + f.n_rhits;
        v[7] += f.n_mid_votes;
        v[8] += f.n_rot_votes;
        v[10] += f.ms_iters[0] + f.ms_iters[1];
        v[11] += f.rebuilds[0] + f.rebuilds[1];
    }
    for (int k = 0; k < DH_N_COUNTERS; ++k) {
        unsigned long long x = v[k];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(&out[k], x);
    }
}

constexpr int kTraverseThreads = 512;

}  // namespace dev

using namespace dev;

// ================================================================ launch wrappers
// cudaFuncSetAttribute is per device: remember, per device, the largest dynamic shared-memory
// size each kernel family was configured for (several contexts on several GPUs may live in one
// process; a context is single-threaded, but two contexts may race here, hence the atomics).
namespace {
constexpr int kMaxDevices = 64;
struct SmemConfig {
    std::atomic<uint32_t> bytes[kMaxDevices];
    SmemConfig() { for (auto& b : bytes) b.store(0); }
    // true if `want` exceeds what the current device was configured for (and records it)
    bool raise(uint32_t want) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= kMaxDevices) return true;
        uint32_t cur = bytes[dev].load();
        while (want > cur)
            if (bytes[dev].compare_exchange_weak(cur, want)) return true;
        return false;
    }
};
}  // namespace

int launch_sat(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, cudaStream_t s) {
    if (b.band_u && g.w + 1 <= 1024) {
        int launches = 0;
        // banded pass: per-band column-sum scans, then the table
        const uint32_t n_bands = (g.h + kSatBandRows - 1) / kSatBandRows;
        const uint32_t threads = (g.w + 1 + 31) & ~31u;
        const uint32_t smem = kSatBandRows * ((g.w + 1 + 8) & ~7u) * 4u;
        static SmemConfig configured;
        if (configured.raise(smem)) cudaFuncSetAttribute(sat_band_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        dim3 gr(n_bands, n_frames);
        sat_band_sums_kernel<<<gr, threads, 0, s>>>(b.depth, b.band_u, g.w, g.h, n_bands);
        sat_band_kernel<<<gr, kSatBandRows * 32, smem, s>>>(b.depth, b.band_u, b.sat, g.w, g.h, g.sat_pitch, n_bands);
        launches += 2;
        return launches;
    }
    dim3 gr((g.h + kSatRowWarps - 1) / kSatRowWarps, n_frames);
    sat_rows_kernel<<<gr, kSatRowWarps * 32, 0, s>>>(b.depth, b.sat, g.w, g.h, g.sat_pitch);
    dim3 gc((g.w + 1 + 127) / 128, n_frames);
    sat_cols_kernel<<<gc, 128, 0, s>>>(b.sat, g.w, g.h, g.sat_pitch);
    return 2;
}

// Box-sum image mode needs: rectangles no larger than 128 per side (strips of 256 input columns
// per warp; prefix sums of 256 window sums stay well-defined) and a patch that a handful of rectangles cover
// (the background test of a patch ORs ceil(sw/rw) * ceil(sh/rh) taps).
bool box_image_supported(uint32_t w, uint32_t h, uint32_t sw, uint32_t sh, uint32_t rw, uint32_t rh) {
    if (!rw || !rh || rw > 128u || rh > 128u || rw > sw || rh > sh || w < rw || h < rh) return false;
    return ((sw + rw - 1u) / rw) * ((sh + rh - 1u) / rh) <= 64u;
}

int launch_box_image(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, int n_sms, bool allow_whole, uint32_t bands,
                     cudaStream_t s) {
    const bool whole = allow_whole && (g.rw & 7u) == 0u;
    // strips: a multiple of kBoxPx output columns each, at most 32*kBoxPx + 1 - rw (column c reads P[c + rw] <= P[32*kBoxPx])
    const uint32_t max_out = (32u * kBoxPx + 1u - g.rw) & ~(uint32_t)(kBoxPx - 1);
    const uint32_t n_strips = (g.box_w + max_out - 1u) / max_out;
    const uint32_t strip_out = (((g.box_w + n_strips - 1u) / n_strips) + kBoxPx - 1u) & ~(uint32_t)(kBoxPx - 1);
    const uint32_t per_warp = (whole ? 0u : 2u * (32u * kBoxPx + 16u) * 4u) + g.rh * 64u * kBoxPx;
    uint32_t wpc = n_strips <= (uint32_t)kBoxMaxWarps ? n_strips : 2u;  // warps per CTA
    while (wpc > 1u && wpc * per_warp > 100u * 1024u) --wpc;           // tall rectangles: long pixel rings
    const uint32_t smem = wpc * per_warp;
    static SmemConfig configured;
    if (configured.raise(smem)) {
        cudaFuncSetAttribute(box_image_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(box_image_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    // bands: a band re-reads the rh - 1 rows above it, so few of them, but enough that the launch has
    // about two rounds of CTAs (the CTAs of a single round do not divide evenly over the SMs and the
    // fullest SM sets the time: 512 frames x 1 band = 3.46 CTAs per SM ran 0.428 ms, 4 bands 0.376 ms);
    // never shorter than rh rows.  bands > 0 forces the count.
    const uint32_t ctas_per_sm = std::max<uint32_t>(1u, std::min<uint32_t>(16u, (227u * 1024u) / (smem + 1024u)));
    const uint32_t slots = (uint32_t)n_sms * ctas_per_sm * wpc;
    const uint32_t units = n_strips * n_frames;
    uint32_t n_bands = std::max<uint32_t>(1u, std::min<uint32_t>((2u * slots + units - 1u) / units, std::max<uint32_t>(1u, g.box_h / g.rh)));
    if (bands) n_bands = std::max<uint32_t>(1u, std::min<uint32_t>(bands, std::max<uint32_t>(1u, g.box_h / g.rh)));
    const uint32_t band_rows = (g.box_h + n_bands - 1u) / n_bands;
    n_bands = (g.box_h + band_rows - 1u) / band_rows;
    const uint32_t n_units = n_strips * n_bands * n_frames;
    const uint32_t blocks = (n_units + wpc - 1u) / wpc;
    if (whole)
        box_image_kernel<true><<<blocks, wpc * 32u, smem, s>>>(b.depth, b.box, g.w, g.h, g.rw, g.rh, g.box_w, g.box_h, g.box_pitch,
                                                              strip_out, n_strips, band_rows, n_bands, n_units);
    else
        box_image_kernel<false><<<blocks, wpc * 32u, smem, s>>>(b.depth, b.box, g.w, g.h, g.rw, g.rh, g.box_w, g.box_h, g.box_pitch,
                                                               strip_out, n_strips, band_rows, n_bands, n_units);
    return 1;
}

uint32_t traverse_smem_bytes(uint32_t tw, uint32_t th, uint32_t patches_per_tile) {
    const uint32_t tile_bytes = (tw * th * 4u + 15u) & ~15u;
    return 128u + tile_bytes + 16u + ((patches_per_tile + 31u) & ~31u) * 4u + 64u;
}

int traverse_kernel_attrs(int* regs, int* max_smem) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, traverse_kernel<kTraverseThreads, 0>);
    if (e != cudaSuccess) return (int)e;
    if (regs) *regs = a.numRegs;
    if (max_smem) *max_smem = a.maxDynamicSharedSizeBytes;
    return 0;
}

template <int kThreads>
static void launch_traverse_t(const CUtensorMap& sat_map, const FrameBuffers& b, const Geometry& g, const TilePlan& tp,
                              const ForestDev& f, uint32_t n_frames, cudaStream_t s) {
    static SmemConfig configured;
    if (configured.raise(tp.smem_bytes)) {
        cudaFuncSetAttribute(traverse_kernel<kThreads, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_bytes);
        cudaFuncSetAttribute(traverse_kernel<kThreads, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_bytes);
        cudaFuncSetAttribute(traverse_kernel<kThreads, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_bytes);
        cudaFuncSetAttribute(traverse_kernel<kThreads, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_bytes);
    }
    dim3 gr(tp.tiles_x * tp.tiles_y, n_frames);
    if (f.uni && g.rw)
        traverse_kernel<kThreads, 4><<<gr, kThreads, tp.smem_bytes, s>>>(sat_map, f.hot_tex, f.hot, f.uni, f.nodes, f.roots, b.leaf, b.box,
                                                                       b.fs, g, tp, f.uni_rw, f.uni_rh);
    else if (f.uni)
        traverse_kernel<kThreads, 2><<<gr, kThreads, tp.smem_bytes, s>>>(sat_map, f.hot_tex, f.hot, f.uni, f.nodes, f.roots, b.leaf, b.sat,
                                                                       b.fs, g, tp, f.uni_rw, f.uni_rh);
    else if (f.hot_tex)
        traverse_kernel<kThreads, 1><<<gr, kThreads, tp.smem_bytes, s>>>(sat_map, f.hot_tex, f.hot, f.uni, f.nodes, f.roots, b.leaf, b.sat,
                                                                       b.fs, g, tp, 0u, 0u);
    else
        traverse_kernel<kThreads, 0><<<gr, kThreads, tp.smem_bytes, s>>>(sat_map, 0, f.hot, f.uni, f.nodes, f.roots, b.leaf, b.sat, b.fs, g,
                                                                       tp, 0u, 0u);
}

void launch_traverse(const CUtensorMap& sat_map, const FrameBuffers& b, const Geometry& g, const TilePlan& tp,
                     const ForestDev& f, uint32_t n_frames, cudaStream_t s) {
    if (tp.threads >= 1024) launch_traverse_t<1024>(sat_map, b, g, tp, f, n_frames, s);
    else launch_traverse_t<512>(sat_map, b, g, tp, f, n_frames, s);
}

void launch_plan_nodes(const NodeRec* nodes, HotNode* hot, UniNode* uni, size_t n_nodes, uint32_t tile_width,
                       const double* prob_codes, cudaStream_t s) {
    if (n_nodes == 0) return;
    plan_nodes_kernel<<<(unsigned)((n_nodes + 255) / 256), 256, 0, s>>>(nodes, hot, uni, n_nodes, tile_width, prob_codes);
}

uint32_t sat_band_rows() { return (uint32_t)kSatBandRows; }
uint32_t vote_box_cells() { return (uint32_t)kBoxCells; }
uint32_t vote_box_dim() { return (uint32_t)kBox; }

// The back end after the traversal, in launch order.  The coarse grids, the accumulator cubes
// and the queue header must be zero when these run.  Each returns the kernels it launched.
template <bool kFrameK>
static int launch_gate_coarse_t(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, bool from_list,
                                int n_sms, uint32_t want_ctas, const float* frame_k, cudaStream_t s) {
    constexpr int kSmem = kGateSmemBytes + (kFrameK ? kFrameKFloats * 4 : 0);
    static SmemConfig configured;
    if (configured.raise((uint32_t)kSmem)) {
        cudaFuncSetAttribute(gate_coarse_kernel<false, kFrameK>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        cudaFuncSetAttribute(gate_coarse_kernel<true, kFrameK>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    }
    const uint32_t per_frame = (g.P + kGateThreads - 1) / kGateThreads;
    if (from_list) {
        // the patch gate writes the frames' gated-patch lists, the seed-grid CTAs take slices of them.  Few CTAs per
        // frame when there are many frames (a slice is a full CTA of work), every possible slice its own
        // CTA when there are few frames (a single frame must still spread over the GPU).
        const uint32_t fill = (6u * (uint32_t)n_sms + n_frames - 1u) / n_frames;
        const uint32_t ctas = std::max<uint32_t>(1u, std::min<uint32_t>(per_frame, want_ctas ? want_ctas : std::max<uint32_t>(4u, fill)));
        patch_gate_kernel<kFrameK><<<dim3((g.P + kPatchGateThreads * kPatchGatePer - 1) / (kPatchGateThreads * kPatchGatePer), n_frames),
                                     kPatchGateThreads, 0, s>>>(b, g, f, frame_k);
        gate_coarse_kernel<true, kFrameK><<<dim3(ctas, n_frames), kGateThreads, kSmem, s>>>(b, g, f, frame_k);
        return 2;
    }
    gate_coarse_kernel<false, kFrameK><<<dim3(per_frame, n_frames), kGateThreads, kSmem, s>>>(b, g, f, frame_k);
    return 1;
}

int launch_gate_coarse(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, bool from_list, int n_sms,
                       uint32_t want_ctas, cudaStream_t s, const float* frame_k) {
    if (!g.P) return 0;
    return frame_k ? launch_gate_coarse_t<true>(b, g, f, n_frames, from_list, n_sms, want_ctas, frame_k, s)
                   : launch_gate_coarse_t<false>(b, g, f, n_frames, from_list, n_sms, want_ctas, nullptr, s);
}

int launch_seed_and_cubes(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames,
                          uint32_t iterations, cudaStream_t s, const float* frame_k) {
    if (frame_k) seed_kernel<true><<<n_frames, kSeedThreads, 0, s>>>(b, g, iterations, frame_k);
    else seed_kernel<false><<<n_frames, kSeedThreads, 0, s>>>(b, g, iterations, nullptr);
    if (!g.P || !iterations) return 1;
    // enough blocks per frame that a thread sees a handful of hits
    const uint32_t per_frame =
        std::max<uint32_t>(1u, std::min<uint32_t>(64u, (g.P * g.n_trees / 8u + kBuildThreads - 1) / kBuildThreads));
    dim3 gr(per_frame, n_frames);
    box_build_kernel<3u><<<gr, kBuildThreads, 0, s>>>(b, g, f);
    return 2;
}

int launch_meanshift(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint32_t iterations,
                     int n_sms, cudaStream_t s) {
    static SmemConfig configured;
    if (configured.raise((uint32_t)kMsSmemBytes))
        cudaFuncSetAttribute(meanshift_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMsSmemBytes);
    // persistent CTAs: three per SM (registers; measured 0.247 -> 0.239 ms against one CTA per accumulator)
    const uint32_t n_items = 2u * n_frames;
    const uint32_t grid = std::min<uint32_t>(n_items, 3u * (uint32_t)std::max(n_sms, 1));
    meanshift_kernel<<<grid, kMsThreads, kMsSmemBytes, s>>>(b, g, f, iterations, n_items, 2u);
    return 1;
}

int launch_heads_round(const FrameBuffers& b, const HeadsBuffers& hb, const Geometry& g, const ForestDev& f, uint32_t n_frames,
                       uint32_t round, uint32_t iterations, int n_sms, const float* frame_k, cudaStream_t s) {
    static SmemConfig configured;
    if (configured.raise((uint32_t)kHeadsPatchSmem))
        cudaFuncSetAttribute(heads_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHeadsPatchSmem);
    if (round == 0) {
        heads_patch_kernel<<<n_frames, kHeadsThreads, kHeadsPatchSmem, s>>>(b, hb, g, f, 0u, iterations);
        return 1;
    }
    // the try's view of the pass: its own frame states, cubes and results; the gated patches of the centre
    // cube are the pass's, those of the rotation cube the ones within R
    FrameBuffers t = b;
    t.fs = hb.fs;
    t.cubes = hb.cubes;
    t.results = hb.res;
    t.ms_trace = nullptr;
    t.clear_cubes = 1;
    t.support = 1;
    const uint32_t per_frame =
        std::max<uint32_t>(1u, std::min<uint32_t>(64u, (g.P * g.n_trees / 8u + kBuildThreads - 1) / kBuildThreads));
    const uint32_t grid = std::min<uint32_t>(n_frames, 3u * (uint32_t)std::max(n_sms, 1));
    static SmemConfig ms_configured;
    if (ms_configured.raise((uint32_t)kMsSmemBytes))
        cudaFuncSetAttribute(meanshift_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMsSmemBytes);
    int launches = 0;
    heads_seed_kernel<<<n_frames, kHeadsThreads, 0, s>>>(b, hb, g, round, iterations, frame_k);
    ++launches;
    if (g.P && iterations) {
        box_build_kernel<1u><<<dim3(per_frame, n_frames), kBuildThreads, 0, s>>>(t, g, f);
        ++launches;
    }
    meanshift_kernel<<<grid, kMsThreads, kMsSmemBytes, s>>>(t, g, f, iterations, n_frames, 0u);
    heads_patch_kernel<<<n_frames, kHeadsThreads, kHeadsPatchSmem, s>>>(b, hb, g, f, round, iterations);
    launches += 2;
    t.gated = hb.gated;
    if (g.P && iterations) {
        box_build_kernel<2u><<<dim3(per_frame, n_frames), kBuildThreads, 0, s>>>(t, g, f);
        ++launches;
    }
    meanshift_kernel<<<grid, kMsThreads, kMsSmemBytes, s>>>(t, g, f, iterations, n_frames, 1u);
    heads_commit_kernel<<<(n_frames + 127) / 128, 128, 0, s>>>(hb, n_frames);
    return launches + 2;
}

void launch_leaf_gates(const double* leaf_prob, const uint32_t* vote_start, const uint32_t* n_votes,
                       const float* offsets, const double* rotations, const uint32_t* rot_bins, LeafInfo* out,
                       LeafBox* box_out, uint32_t* rot_cells, uint32_t n_leaves, cudaStream_t s) {
    leaf_gate_kernel<<<(n_leaves + 127) / 128, 128, 0, s>>>(leaf_prob, vote_start, n_votes, offsets, rotations, rot_bins, out,
                                                           box_out, rot_cells, n_leaves);
}

void launch_mask(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint8_t* mask, cudaStream_t s) {
    mask_kernel<<<dim3((g.P + 255) / 256, n_frames), 256, 0, s>>>(b, g, f.leaf_prob, mask);
}

void launch_track_mask(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, const TrackSlot* slots,
                       uint32_t frame0, uint32_t frame_step, uint8_t* mask, cudaStream_t s) {
    if (!n_frames) return;
    const dim3 grid((g.w + kTrackMaskTileW - 1) / kTrackMaskTileW, (g.h + kTrackMaskTileH - 1) / kTrackMaskTileH, n_frames);
    track_mask_kernel<<<grid, kTrackMaskTileW * kTrackMaskTileH / 4, 0, s>>>(b, g, f.leaf_prob, slots, frame0, frame_step, mask);
}

void launch_hough_votes(const FrameBuffers& b, const Geometry& g, const ForestDev& f, uint32_t n_frames, uint32_t* acc32, cudaStream_t s,
                        const float* frame_k) {
    const uint32_t n = g.P * g.n_trees;
    const dim3 grid((n + 255) / 256, n_frames);
    if (frame_k) hough_image_kernel<true><<<grid, 256, 0, s>>>(b, g, f, acc32, frame_k);
    else hough_image_kernel<false><<<grid, 256, 0, s>>>(b, g, f, acc32, nullptr);
}

void launch_narrow_u16(const uint32_t* acc32, uint16_t* out16, size_t n, cudaStream_t s) {
    narrow_u16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(acc32, out16, n);
}

int launch_gaussian_blur(const uint32_t* in, uint16_t* tmp, uint16_t* out, unsigned long long* keys, uint32_t w, uint32_t h,
                         uint32_t n_frames, const float* k, int radius, cudaStream_t s) {
    const uint32_t smem_h = (uint32_t)(kBlurHy * (kBlurHx + 2 * radius)) * 2u, smem_v = (uint32_t)((kBlurVy + 2 * radius) * kBlurVx) * 2u;
    static SmemConfig ch, cv;
    if (ch.raise(smem_h)) cudaFuncSetAttribute(blur_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h);
    if (cv.raise(smem_v)) cudaFuncSetAttribute(blur_v_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_v);
    blur_h_kernel<<<dim3((w + kBlurHx - 1) / kBlurHx, (h + kBlurHy - 1) / kBlurHy, n_frames), dim3(kBlurHx, kBlurHy), smem_h, s>>>(
        in, tmp, w, h, k, radius);
    blur_v_kernel<<<dim3((w + kBlurVx - 1) / kBlurVx, (h + kBlurVy - 1) / kBlurVy, n_frames), dim3(kBlurVx, kBlurVy), smem_v, s>>>(
        tmp, out, w, h, k, radius, keys);
    return 2;
}
void launch_hough2d_pose(const unsigned long long* keys, const uint16_t* depth, const Geometry& g, uint32_t n_frames, dh_result* out,
                         cudaStream_t s, const float* frame_k) {
    if (frame_k) hough2d_pose_kernel<true><<<(n_frames + 127) / 128, 128, 0, s>>>(keys, depth, g, n_frames, out, frame_k);
    else hough2d_pose_kernel<false><<<(n_frames + 127) / 128, 128, 0, s>>>(keys, depth, g, n_frames, out, nullptr);
}

void launch_seq_guess(FrameState* fs, const dh_result* prev, uint32_t n, float min_seed_z, cudaStream_t s) {
    if (n) seq_guess_kernel<<<(n + 127) / 128, 128, 0, s>>>(fs, prev, n, min_seed_z);
}

void launch_track_guess(FrameState* fs, float* frame_k, const TrackSlot* slots, const TrackArgs* tracks, const dh_result* prev,
                        uint32_t n, float min_seed_z, const uint32_t* status, unsigned long long* bad, cudaStream_t s) {
    if (n) track_guess_kernel<<<(n + 127) / 128, 128, 0, s>>>(fs, frame_k, slots, tracks, prev, n, min_seed_z, status, bad);
}

void launch_track_gather(const uint16_t* src, uint16_t* dst, const TrackSlot* slots, uint32_t n, size_t frame_px, cudaStream_t s) {
    if (!n) return;
    const uint32_t vec = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0 && frame_px % 8 == 0) ? 1u : 0u;
    const size_t words = vec ? frame_px / 8 : frame_px;
    const uint32_t blocks = (uint32_t)std::min<size_t>(64, std::max<size_t>(1, (words + 1023) / 1024));
    track_gather_kernel<<<dim3(blocks, n), 256, 0, s>>>(src, dst, slots, frame_px, vec);
}

void launch_counters(const FrameBuffers& b, const Geometry& g, uint32_t n_frames, unsigned long long* out,
                     cudaStream_t s) {
    const uint32_t blocks = (n_frames + 255) / 256;
    counters_kernel<<<blocks, 256, 0, s>>>(b.fs, n_frames, out, g.P, g.n_trees);
}

void launch_biwi_decode(const uint8_t* blob, const unsigned long long* offsets, const unsigned long long* ends,
                        unsigned long long blob_base, uint32_t n, uint32_t w, uint32_t h, uint16_t* out, uint32_t* status, cudaStream_t s) {
    if (n) biwi_decode_kernel<<<n, kRleThreads, 0, s>>>(blob, offsets, ends, blob_base, w, h, out, status);
}

void launch_box_dump(const FrameBuffers& b, uint32_t frame, int which, int32_t* keys, uint32_t* vals,
                     unsigned long long* count, cudaStream_t s) {
    box_dump_kernel<<<128, 256, 0, s>>>(b, frame, which, keys, vals, count);
}

}  // namespace dh
