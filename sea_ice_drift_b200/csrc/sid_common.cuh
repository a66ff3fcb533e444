// sid_common.cuh -- device helpers shared by all kernels of the MCC hot path.
//
// Arithmetic contract (what makes results reproducible bit for bit on any IEEE-754 machine):
//   * correlation numerators, window sums and template sums are exact integers;
//   * everything OpenCV's common_matchTemplate does in double is done here in double
//     with explicit round-to-nearest intrinsics, so the compiler can never contract
//     a multiply-add into an FMA (an FMA rounds once and would change the last bit);
//   * template coordinates follow scipy.ndimage.affine_transform's evaluation order
//     (off + i*m0 + j*m1, left to right) in double, again without FMA;
//   * np.gradient / np.hypot / np.median / np.std run in float32 as NumPy does.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include <math.h>

namespace sid {

// ---------------------------------------------------------------- float <-> sortable key
__device__ __forceinline__ uint32_t f32_key(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(u);
}

// ---------------------------------------------------------------- block reductions
// All take a small shared scratch area and are called by every thread of the CTA.
struct BlockScratch {
    double red[32];
    uint32_t hist[256];
    uint32_t sel[4];            // bin, rank inside the bin, population of the bin, candidate counter
    uint32_t wtot[32];
    uint32_t cand[64];
};

__device__ __forceinline__ double block_sum(double v, BlockScratch &bs) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) bs.red[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += bs.red[w];
    return t;
}

// k-th smallest (0-based) of n floats: 4-pass MSD radix select on sortable keys.
__device__ float block_select(const float *__restrict__ d, int n, int k, BlockScratch &bs) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    uint32_t prefix = 0, mask = 0;
    uint32_t kk = (uint32_t)k;
    const int iters = (n + nt - 1) / nt;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += nt) bs.hist[i] = 0;
        __syncthreads();
        for (int it = 0; it < iters; ++it) {
            const int i = it * nt + tid;
            uint32_t bin = 0xffffffffu;
            if (i < n) {
                const uint32_t key = f32_key(d[i]);
                if ((key & mask) == prefix) bin = (key >> shift) & 255u;
            }
            // warp-aggregated histogram update: one atomic per distinct bin per warp
            const uint32_t peers = __match_any_sync(0xffffffffu, bin);
            if (bin != 0xffffffffu && lane == (__ffs(peers) - 1)) atomicAdd(&bs.hist[bin], __popc(peers));
        }
        __syncthreads();
        if (warp == 0) {
            uint32_t h[8], s = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { h[j] = bs.hist[lane * 8 + j]; s += h[j]; }
            uint32_t incl = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const uint32_t excl = incl - s;
            if (kk >= excl && kk < incl) {
                uint32_t c = excl;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (kk < c + h[j]) { bs.sel[0] = lane * 8 + j; bs.sel[1] = kk - c; break; }
                    c += h[j];
                }
            }
        }
        __syncthreads();
        prefix |= bs.sel[0] << shift;
        mask |= 0xffu << shift;
        kk = bs.sel[1];
        __syncthreads();
    }
    return key_f32(prefix);
}

// Same selection with 11/11/10-bit digits (3 passes) on a caller-provided 2048-bin histogram
// (shared memory that is free at that point of the kernel).
__device__ float block_select_wide(const float *__restrict__ d, int n, int k, uint32_t *__restrict__ hist, BlockScratch &bs) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    uint32_t prefix = 0, mask = 0;
    uint32_t kk = (uint32_t)k;
    const int iters = (n + nt - 1) / nt;
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
        const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
        const int bits = pass == 2 ? 10 : 11;
        const int nbins = 1 << bits;
        for (int i = tid; i < nbins; i += nt) hist[i] = 0;
        __syncthreads();
        for (int it = 0; it < iters; ++it) {
            const int i = it * nt + tid;
            uint32_t bin = 0xffffffffu;
            if (i < n) {
                const uint32_t key = f32_key(d[i]);
                if ((key & mask) == prefix) bin = (key >> shift) & (uint32_t)(nbins - 1);
            }
            const uint32_t peers = __match_any_sync(0xffffffffu, bin);
            if (bin != 0xffffffffu && lane == (__ffs(peers) - 1)) atomicAdd(&hist[bin], __popc(peers));
        }
        __syncthreads();
        {   // rank search over the histogram with the whole CTA: per-thread chunk sums, block-wide exclusive
            // scan, then the single owning thread walks its chunk
            const int per = (nbins + nt - 1) / nt;
            const int b0 = tid * per;
            uint32_t s = 0;
            for (int j = 0; j < per; ++j) if (b0 + j < nbins) s += hist[b0 + j];
            uint32_t incl = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) bs.wtot[warp] = incl;
            __syncthreads();
            uint32_t woff = 0;
            for (int w = 0; w < warp; ++w) woff += bs.wtot[w];
            const uint32_t excl = woff + incl - s;
            if (kk >= excl && kk < excl + s) {
                uint32_t c = excl;
                for (int j = 0; j < per; ++j) {
                    const uint32_t h = hist[b0 + j];
                    if (kk < c + h) { bs.sel[0] = b0 + j; bs.sel[1] = kk - c; bs.sel[2] = h; bs.sel[3] = 0; break; }
                    c += h;
                }
            }
        }
        __syncthreads();
        prefix |= bs.sel[0] << shift;
        mask |= (uint32_t)(nbins - 1) << shift;
        kk = bs.sel[1];
        const uint32_t pop = bs.sel[2];
        if (pass < 2 && pop <= 64u) {
            // few elements share the prefix: collect them and rank directly instead of further passes
            for (int it = 0; it < iters; ++it) {
                const int i = it * nt + tid;
                if (i < n) {
                    const uint32_t key = f32_key(d[i]);
                    if ((key & mask) == prefix) bs.cand[atomicAdd(&bs.sel[3], 1u)] = key;
                }
            }
            __syncthreads();
            if (tid < (int)pop) {
                const uint32_t mine = bs.cand[tid];
                uint32_t rank = 0;
                for (uint32_t j = 0; j < pop; ++j) {
                    const uint32_t o = bs.cand[j];
                    rank += (o < mine) || (o == mine && j < (uint32_t)tid);
                }
                if (rank == kk) bs.sel[0] = mine;
            }
            __syncthreads();
            const uint32_t key = bs.sel[0];
            __syncthreads();
            return key_f32(key);
        }
        __syncthreads();
    }
    return key_f32(prefix);
}

// np.median of n float32 values (no NaN handling needed: NCC maps are finite).
// `wide_hist`: optional 2048-word shared-memory scratch enabling the 3-pass variant.
__device__ float block_median(const float *__restrict__ d, int n, BlockScratch &bs, uint32_t *wide_hist = nullptr) {
    if (wide_hist) {
        if (n & 1) return block_select_wide(d, n, n / 2, wide_hist, bs);
        const float a = block_select_wide(d, n, n / 2 - 1, wide_hist, bs);
        const float b = block_select_wide(d, n, n / 2, wide_hist, bs);
        return __fmul_rn(__fadd_rn(a, b), 0.5f);
    }
    if (n & 1) return block_select(d, n, n / 2, bs);
    const float a = block_select(d, n, n / 2 - 1, bs);
    const float b = block_select(d, n, n / 2, bs);
    return __fmul_rn(__fadd_rn(a, b), 0.5f);
}

// np.std (float32 input, ddof=0): float32 mean / deviations / squares, sums in double.
__device__ float block_std(const float *__restrict__ d, int n, BlockScratch &bs) {
    const int tid = threadIdx.x, nt = blockDim.x;
    double s = 0.0;
    for (int i = tid; i < n; i += nt) s += (double)d[i];
    s = block_sum(s, bs);
    const float mean = __double2float_rn(s / (double)n);
    double q = 0.0;
    for (int i = tid; i < n; i += nt) {
        const float dv = __fsub_rn(d[i], mean);
        q += (double)__fmul_rn(dv, dv);
    }
    q = block_sum(q, bs);
    const float var = __double2float_rn(q / (double)n);
    return __fsqrt_rn(var);
}

// ---------------------------------------------------------------- NCC normalisation
// cv::meanStdDev + the template part of common_matchTemplate.
struct TemplStats {
    double mean;   // templMean
    double norm;   // templNorm = sqrt(sdv^2) / sqrt(invArea)
    int flat;      // sdv^2 < DBL_EPSILON -> whole map = 1
};

__device__ __forceinline__ TemplStats templ_stats(uint32_t tsum, uint32_t tsq, double inv_area, double sqrt_inv_area) {
    TemplStats st;
    st.mean = __dmul_rn((double)tsum, inv_area);
    double var = __dsub_rn(__dmul_rn((double)tsq, inv_area), __dmul_rn(st.mean, st.mean));
    if (var < 0.0) var = 0.0;
    const double sdv = __dsqrt_rn(var);
    const double tn = __dmul_rn(sdv, sdv);
    st.flat = tn < DBL_EPSILON;
    st.norm = __ddiv_rn(__dsqrt_rn(tn), sqrt_inv_area);
    return st;
}

// sqrt(max(winSqSum - winSum^2/N, 0)), or 0 under OpenCV's "avoid rounding errors" rule
__device__ __forceinline__ double window_den(uint32_t wsum, uint32_t wsq, double inv_area) {
    const double t = (double)wsum;
    const double mean2 = __dmul_rn(__dmul_rn(t, t), inv_area);
    const double sum2 = (double)wsq;
    double diff2 = __dsub_rn(sum2, mean2);
    if (diff2 < 0.0) diff2 = 0.0;
    double thr = __dmul_rn(10.0 * (double)FLT_EPSILON, sum2);
    if (thr > 0.5) thr = 0.5;
    return diff2 <= thr ? 0.0 : __dsqrt_rn(diff2);
}

// out-of-line copy for call sites that would otherwise inline dozens of instances (instruction-cache footprint)
__device__ __noinline__ float ncc_value_call(int corr, uint32_t wsum, double wden, double mean, double norm) {
    double num = __dsub_rn((double)corr, __dmul_rn((double)wsum, mean));
    const double t = __dmul_rn(wden, norm);
    const double an = fabs(num);
    if (an < t) num = __ddiv_rn(num, t);
    else if (an < __dmul_rn(t, 1.125)) num = num > 0.0 ? 1.0 : -1.0;
    else num = 0.0;
    return __double2float_rn(num);
}

// three angles of one output position per call: three independent FP64 chains (ILP), one call overhead
struct Ncc3 { float v0, v1, v2; };
__device__ __forceinline__ double ncc_finish(double num, double t) {
    const double an = fabs(num);
    if (an < t) return __ddiv_rn(num, t);
    if (an < __dmul_rn(t, 1.125)) return num > 0.0 ? 1.0 : -1.0;
    return 0.0;
}
// Four NCC values at once, branch-free on the common path so that the four FP64 division chains interleave (the IEEE
// software division has a branch to its slow path after every quotient, which serialises consecutive divisions).
// Quotient: Newton-refined reciprocal -> within ~1 ulp(double) of num/t; its float32 rounding equals the float32 rounding
// of the correctly rounded double unless a float32 rounding boundary (mantissa bits below float32 = 1000...0) lies
// within a few double ulps; those (~1 in 2^24), tiny divisors and tiny quotients are redone with the IEEE division.
// Result bit for bit == (float)ncc_finish(num, t).
__device__ __forceinline__ void ncc_finish4(const double (&num)[4], const double (&t)[4], float (&v)[4]) {
    double r[4], q[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r[c]) : "d"(t[c]));
#pragma unroll
    for (int c = 0; c < 4; ++c) { const double e = fma(-t[c], r[c], 1.0); r[c] = fma(r[c], e, r[c]); }
#pragma unroll
    for (int c = 0; c < 4; ++c) { const double e = fma(-t[c], r[c], 1.0); r[c] = fma(r[c], e, r[c]); }
#pragma unroll
    for (int c = 0; c < 4; ++c) q[c] = num[c] * r[c];
#pragma unroll
    for (int c = 0; c < 4; ++c) q[c] = fma(r[c], fma(-t[c], q[c], num[c]), q[c]);
    bool redo = false;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const unsigned long long low = (unsigned long long)__double_as_longlong(q[c]) & 0x1fffffffull;
        const unsigned long long d = low > 0x10000000ull ? low - 0x10000000ull : 0x10000000ull - low;
        // anything but the plain quotient (|num| >= t: OpenCV's +-1 / 0 cases) goes through the exact path below
        const bool fast_ok = fabs(num[c]) < t[c] && d > 16ull && t[c] > 1e-280 && fabs(q[c]) > 1e-30;
        redo = redo || !fast_ok;
        v[c] = __double2float_rn(q[c]);
    }
    if (redo) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = __double2float_rn(ncc_finish(num[c], t[c]));
    }
}
// four positions of one angle from their exact integers: numerator, window sum, window sum of squares (non-flat template)
__device__ __forceinline__ void ncc_ints4(const int32_t (&corr)[4], const uint32_t (&wsum)[4], const uint32_t (&wsq)[4],
                                          const TemplStats &st, double inv_area, float (&v)[4]) {
    double num[4], tt[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        num[c] = __dsub_rn((double)corr[c], __dmul_rn((double)wsum[c], st.mean));
        tt[c] = __dmul_rn(window_den(wsum[c], wsq[c], inv_area), st.norm);
    }
    ncc_finish4(num, tt, v);
}
__device__ __forceinline__ float4 ncc_vec4(int4 c, uint4 ws, uint4 wq, const TemplStats &st, double inv_area) {
    const int32_t cc[4] = {c.x, c.y, c.z, c.w};
    const uint32_t s4[4] = {ws.x, ws.y, ws.z, ws.w}, q4[4] = {wq.x, wq.y, wq.z, wq.w};
    float v[4];
    ncc_ints4(cc, s4, q4, st, inv_area, v);
    return make_float4(v[0], v[1], v[2], v[3]);
}

__device__ __noinline__ Ncc3 ncc_value_call3(int c0, int c1, int c2, uint32_t wsum, double wden,
                                             double m0, double n0, double m1, double n1, double m2, double n2) {
    const double ws = (double)wsum;
    const double num0 = __dsub_rn((double)c0, __dmul_rn(ws, m0));
    const double num1 = __dsub_rn((double)c1, __dmul_rn(ws, m1));
    const double num2 = __dsub_rn((double)c2, __dmul_rn(ws, m2));
    const double t0 = __dmul_rn(wden, n0), t1 = __dmul_rn(wden, n1), t2 = __dmul_rn(wden, n2);
    Ncc3 r;
    r.v0 = __double2float_rn(ncc_finish(num0, t0));
    r.v1 = __double2float_rn(ncc_finish(num1, t1));
    r.v2 = __double2float_rn(ncc_finish(num2, t2));
    return r;
}

__device__ __forceinline__ float ncc_value(int64_t corr, uint32_t wsum, double wden, const TemplStats &st) {
    if (st.flat) return 1.0f;
    double num = __dsub_rn((double)corr, __dmul_rn((double)wsum, st.mean));
    const double t = __dmul_rn(wden, st.norm);
    const double an = fabs(num);
    if (an < t) num = __ddiv_rn(num, t);
    else if (an < __dmul_rn(t, 1.125)) num = num > 0.0 ? 1.0 : -1.0;
    else num = 0.0;
    return __double2float_rn(num);
}

// ---------------------------------------------------------------- rotated template sample
// get_template (reference pmlib.py:89-115): output pixel (i, j) samples image 1 at
//   row = (off0 + i*cos) + j*sin,   col = (off1 + i*(-sin)) + j*cos      (FP64, no FMA)
__device__ __forceinline__ void template_coord(double off0, double off1, double cs, double sn, int i, int j,
                                               double &row, double &col) {
    const double di = (double)i, dj = (double)j;
    row = __dadd_rn(__dadd_rn(off0, __dmul_rn(di, cs)), __dmul_rn(dj, sn));
    col = __dadd_rn(__dadd_rn(off1, __dmul_rn(di, -sn)), __dmul_rn(dj, cs));
}
// Sample at (row, col).  CHECKED: apply scipy's mode='constant' rule (outside [0, dim-1] -> 0) and
// clamp the bilinear neighbours; unchecked when the caller knows the whole template lies >= 1 px
// inside the image (then neither can trigger).
template <bool CHECKED>
__device__ __forceinline__ uint32_t template_sample(const uint8_t *__restrict__ img, int rows, int cols, int64_t pitch,
                                                    double row, double col, int order) {
    if (CHECKED) {
        if (!(row >= 0.0 && row <= (double)(rows - 1) && col >= 0.0 && col <= (double)(cols - 1))) return 0;
    }
    if (order == 0) {
        int ri = __double2int_rd(__dadd_rn(row, 0.5));
        int ci = __double2int_rd(__dadd_rn(col, 0.5));
        if (CHECKED) { ri = min(ri, rows - 1); ci = min(ci, cols - 1); }
        return __ldg(img + (int64_t)ri * pitch + ci);
    }
    const double fr = floor(row), fc = floor(col);
    const int r0 = (int)fr, c0 = (int)fc;
    const double fy = __dsub_rn(row, fr), fx = __dsub_rn(col, fc);
    const double wy0 = __dsub_rn(1.0, fy), wx0 = __dsub_rn(1.0, fx);
    int r1 = r0 + 1, c1 = c0 + 1;
    if (CHECKED) { r1 = min(r1, rows - 1); c1 = min(c1, cols - 1); }
    const uint8_t *p0 = img + (int64_t)r0 * pitch, *p1 = img + (int64_t)r1 * pitch;
    double t = 0.0;
    t = __dadd_rn(t, __dmul_rn(__dmul_rn((double)__ldg(p0 + c0), wy0), wx0));
    t = __dadd_rn(t, __dmul_rn(__dmul_rn((double)__ldg(p0 + c1), wy0), fx));
    t = __dadd_rn(t, __dmul_rn(__dmul_rn((double)__ldg(p1 + c0), fy), wx0));
    t = __dadd_rn(t, __dmul_rn(__dmul_rn((double)__ldg(p1 + c1), fy), fx));
    t = t > 0.0 ? __dadd_rn(t, 0.5) : 0.0;
    if (t > 255.0) t = 255.0;
    return (uint32_t)t;
}
__device__ __forceinline__ uint8_t template_pixel(const uint8_t *__restrict__ img, int rows, int cols, int64_t pitch,
                                                  double off0, double off1, double cs, double sn,
                                                  int i, int j, int order) {
    double row, col;
    template_coord(off0, off1, cs, sn, i, j, row, col);
    return (uint8_t)template_sample<true>(img, rows, cols, pitch, row, col, order);
}
// true when all four template corners map >= 1 px inside the image: the affine map of the
// s x s index square is a parallelogram, so every sample is then strictly inside.
__device__ __forceinline__ bool template_inside(int rows, int cols, double off0, double off1, double cs, double sn, int s) {
    bool in = true;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        double row, col;
        template_coord(off0, off1, cs, sn, (c & 1) ? s - 1 : 0, (c & 2) ? s - 1 : 0, row, col);
        in = in && row >= 1.0 && row <= (double)(rows - 2) && col >= 1.0 && col <= (double)(cols - 2);
    }
    return in;
}

// same test, one corner per lane (lanes 0..3), result uniform over the warp
__device__ __forceinline__ bool template_inside_warp(int rows, int cols, double off0, double off1, double cs, double sn, int s) {
    const int c = threadIdx.x & 3;
    double row, col;
    template_coord(off0, off1, cs, sn, (c & 1) ? s - 1 : 0, (c & 2) ? s - 1 : 0, row, col);
    const bool in = row >= 1.0 && row <= (double)(rows - 2) && col >= 1.0 && col <= (double)(cols - 2);
    return __all_sync(0xffffffffu, in);
}

// ---------------------------------------------------------------- Hessian pieces
// np.gradient along one axis (unit spacing, edge_order=1) at position `i` of a line
// of `n` float32 samples spaced `stride` apart.
__device__ __forceinline__ float grad_at(const float *__restrict__ line, int n, int stride, int i) {
    if (i == 0) return __fsub_rn(line[stride], line[0]);
    if (i == n - 1) return __fsub_rn(line[(n - 1) * stride], line[(n - 2) * stride]);
    return __fmul_rn(__fsub_rn(line[(i + 1) * stride], line[(i - 1) * stride]), 0.5f);
}
// gradient of the gradient along the same axis
__device__ __forceinline__ float grad2_at(const float *__restrict__ line, int n, int stride, int i) {
    if (i >= 2 && i <= n - 3) {          // interior: both neighbouring first derivatives are central differences
        const float c = line[i * stride];
        const float gp = __fmul_rn(__fsub_rn(line[(i + 2) * stride], c), 0.5f);
        const float gm = __fmul_rn(__fsub_rn(c, line[(i - 2) * stride]), 0.5f);
        return __fmul_rn(__fsub_rn(gp, gm), 0.5f);
    }
    if (i == 0) return __fsub_rn(grad_at(line, n, stride, 1), grad_at(line, n, stride, 0));
    if (i == n - 1) return __fsub_rn(grad_at(line, n, stride, n - 1), grad_at(line, n, stride, n - 2));
    return __fmul_rn(__fsub_rn(grad_at(line, n, stride, i + 1), grad_at(line, n, stride, i - 1)), 0.5f);
}
// hes = hypot(d2/dx2, d2/dy2) at (y, x) of a rows x cols map
__device__ __forceinline__ float hessian_at(const float *__restrict__ f, int rows, int cols, int y, int x) {
    const double a = (double)grad2_at(f + (size_t)y * cols, cols, 1, x);
    const double b = (double)grad2_at(f + x, rows, cols, y);
    return __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b))));
}
__device__ __forceinline__ int reflect_index(int i, int n) {
    // scipy 'reflect': (d c b a | a b c d | d c b a)
    while (i < 0 || i >= n) {
        if (i < 0) i = -i - 1;
        if (i >= n) i = 2 * n - 1 - i;
    }
    return i;
}
// one pass of gaussian_filter(sigma=1) (9 taps, weights gw[0..4] = centre..edge) along `axis`
__device__ __forceinline__ float gauss_at(const float *__restrict__ f, int rows, int cols, int y, int x, int axis,
                                          const double *gw) {
    double acc = __dmul_rn(gw[0], (double)f[(size_t)y * cols + x]);
#pragma unroll
    for (int k = 1; k <= 4; ++k) {
        double a, b;
        if (axis == 0) {
            a = (double)f[(size_t)reflect_index(y - k, rows) * cols + x];
            b = (double)f[(size_t)reflect_index(y + k, rows) * cols + x];
        } else {
            a = (double)f[(size_t)y * cols + reflect_index(x - k, cols)];
            b = (double)f[(size_t)y * cols + reflect_index(x + k, cols)];
        }
        acc = __dadd_rn(acc, __dmul_rn(gw[k], __dadd_rn(a, b)));
    }
    return __double2float_rn(acc);
}

// ---- fast path of peak_statistics: hes_norm only, maps of at least 5 x 5 with an odd number of elements, CTAs of 128 / 256 /
// 512 threads, a 2048-word shared-memory histogram.  Same values as the general path below, three sweeps over the map
// instead of six: the Hessian sweep also accumulates the sum (np.std's mean) and the first radix-select histogram; the
// second sweep accumulates the squared deviations and the second histogram; a third sweep collects the (<= 64) values
// sharing the median's upper 20 bits.  hypot() is never negative, so a value's bit pattern is its sortable key (digits:
// bits 30..21 | 20..11 | 10..0).  The FP64 sums of float32 addends are exact for the map sizes of the split tail whatever the
// order and differ from the sequential order by < 1 ulp(double) for the largest maps -- far below the float32 rounding that
// follows -- which is why the kernels and the CPU restatement used by the tests agree bit for bit.
// Rank search over 1024 bins (1024 / blockDim.x per thread): the thread owning the bin of rank kk writes sel = {bin, rank
// inside it, population of the bin, 0}.  Two barriers inside.
__device__ __forceinline__ void fast_rank_search(const uint32_t *__restrict__ hist, uint32_t kk, BlockScratch &bs) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int per = 1024 / nt;                       // 8, 4 or 2
    uint32_t h[8];
    uint32_t sum = 0;
    if (per == 8) {
        const uint4 h0 = reinterpret_cast<const uint4 *>(hist)[2 * tid], h1 = reinterpret_cast<const uint4 *>(hist)[2 * tid + 1];
        h[0] = h0.x; h[1] = h0.y; h[2] = h0.z; h[3] = h0.w; h[4] = h1.x; h[5] = h1.y; h[6] = h1.z; h[7] = h1.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) h[j] = j < per ? hist[tid * per + j] : 0u;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) sum += h[j];
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) bs.wtot[warp] = incl;
    __syncthreads();
    uint32_t excl = incl - sum;
    for (int w = 0; w < warp; ++w) excl += bs.wtot[w];
    if (kk >= excl && kk < excl + sum) {
        uint32_t c = excl;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (kk >= c && kk < c + h[j]) { bs.sel[0] = (uint32_t)(tid * per + j); bs.sel[1] = kk - c; bs.sel[2] = h[j]; bs.sel[3] = 0u; }
            c += h[j];
        }
    }
    __syncthreads();
}

// `hist`: 2048 words of shared memory (any contents).  Returns (hes[peak] - median(hes)) / std(hes) and the median and std
// it used; every thread calls it.
__device__ float hes_norm_fast(const float *__restrict__ map, int rows, int cols, int peak_idx, float *__restrict__ hes,
                               uint32_t *__restrict__ hist, BlockScratch &bs, float &med_out, float &sd_out) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5, n = rows * cols;
    for (int k = tid; k < 512; k += nt) reinterpret_cast<uint4 *>(hist)[k] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    double dsum = 0.0;
    // one Hessian value per lane and call (all 32 lanes call together): store, sum, first histogram (warp-aggregated:
    // the values of a map fall into a handful of the 1024 exponent bins)
    auto emit = [&](bool valid, int k, float v) {
        uint32_t bin = 0xffffffffu;
        if (valid) { hes[k] = v; dsum += (double)v; bin = __float_as_uint(v) >> 21; }
        const uint32_t peers = __match_any_sync(0xffffffffu, bin);
        if (valid && lane == (__ffs(peers) - 1)) atomicAdd(&hist[bin & 1023u], (uint32_t)__popc(peers));
    };
    {   // interior: branch-free 5-point stencils, the rounding sequence of np.gradient(np.gradient(.)) away from the edges
        const int iw = cols - 4, ni = (rows - 4) * iw;
        const int idy = nt / iw, idx = nt - idy * iw;
        int y = tid / iw, x = tid - y * iw;
        for (int k = tid; k - tid < ni; k += nt) {
            const bool valid = k < ni;
            float v = 0.0f;
            const int o = (y + 2) * cols + (x + 2);
            if (valid) {
                const float *p = map + o;
                const float c = p[0];
                const float gxp = __fmul_rn(__fsub_rn(p[2], c), 0.5f), gxm = __fmul_rn(__fsub_rn(c, p[-2]), 0.5f);
                const float gyp = __fmul_rn(__fsub_rn(p[2 * cols], c), 0.5f), gym = __fmul_rn(__fsub_rn(c, p[-2 * cols]), 0.5f);
                const double a2 = (double)__fmul_rn(__fsub_rn(gxp, gxm), 0.5f), b2 = (double)__fmul_rn(__fsub_rn(gyp, gym), 0.5f);
                v = __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(a2, a2), __dmul_rn(b2, b2))));
            }
            emit(valid, o, v);
            x += idx; y += idy; if (x >= iw) { x -= iw; ++y; }
        }
        // border frame: two rows top and bottom, two columns left and right
        const int nb = 4 * cols + 4 * (rows - 4);
        for (int k = tid; k - tid < nb; k += nt) {
            const bool valid = k < nb;
            int yy = 0, xx = 0;
            if (k < 4 * cols) { const int r = k / cols; xx = k - r * cols; yy = r < 2 ? r : rows - 4 + r; }
            else { const int q = k - 4 * cols, r = q >> 2, ci = q & 3; yy = r + 2; xx = ci < 2 ? ci : cols - 4 + ci; }
            float v = 0.0f;
            if (valid) v = hessian_at(map, rows, cols, yy, xx);
            emit(valid, yy * cols + xx, v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
    if (lane == 0) bs.red[warp] = dsum;
    __syncthreads();                                   // hes, hist[0..1023] and red are complete
    double tot = 0.0;
    for (int w = 0; w < nw; ++w) tot += bs.red[w];
    const float mean = __double2float_rn(tot / (double)n);
    fast_rank_search(hist, (uint32_t)(n / 2), bs);
    const uint32_t b1 = bs.sel[0], kk1 = bs.sel[1];
    // second sweep: squared deviations (np.std) + second histogram over the values in bin b1
    double q = 0.0;
    for (int i = tid; i < n; i += nt) {
        const float v = hes[i];
        const float dv = __fsub_rn(v, mean);
        q += (double)__fmul_rn(dv, dv);
        const uint32_t u = __float_as_uint(v);
        if ((u >> 21) == b1) atomicAdd(&hist[1024u + ((u >> 11) & 1023u)], 1u);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    if (lane == 0) bs.red[16 + warp] = q;
    __syncthreads();
    double qt = 0.0;
    for (int w = 0; w < nw; ++w) qt += bs.red[16 + w];
    const float sd = __fsqrt_rn(__double2float_rn(qt / (double)n));
    fast_rank_search(hist + 1024, kk1, bs);
    const uint32_t prefix = (b1 << 10) | bs.sel[0], kk2 = bs.sel[1], pop = bs.sel[2];
    float med;
    if (pop <= 64u) {
        for (int i = tid; i < n; i += nt) {
            const uint32_t u = __float_as_uint(hes[i]);
            if ((u >> 11) == prefix) bs.cand[atomicAdd(&bs.sel[3], 1u)] = u;
        }
        __syncthreads();
        if (tid < (int)pop) {
            const uint32_t mine = bs.cand[tid];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < pop; ++j) {
                const uint32_t o = bs.cand[j];
                rank += (o < mine) || (o == mine && j < (uint32_t)tid);
            }
            if (rank == kk2) bs.sel[0] = mine;
        }
        __syncthreads();
        med = __uint_as_float(bs.sel[0]);
        __syncthreads();                               // bs.sel is free again
    } else {
        med = block_select_wide(hes, n, n / 2, hist, bs);          // many values share 20 bits (flat maps): the general select
    }
    med_out = med;
    sd_out = sd;
    return __fdiv_rn(__fsub_rn(hes[peak_idx], med), sd);
}

// Tail of rotate_and_match (reference pmlib.py:167-172): Hessian at the peak and the
// optional normalisations.  `best` is the winning NCC map; tmp_a/tmp_b/hes are scratch
// maps of the same size.  Every thread of the CTA calls this; results valid in all.  On return `best` is unchanged and
// `hes` holds the Hessian map (of the smoothed map with hes_smth) before normalisation; hmed / hsd (hes_norm) and rmed /
// rsd (mcc_norm) are the median and std that normalised h and r, so SID_PEAKS normalises its secondary peaks with them.
struct PeakStats { float h; float r; float hmed, hsd, rmed, rsd; };
__device__ PeakStats peak_statistics(const float *__restrict__ best, int rows, int cols, int peak_idx, float peak_r,
                                     unsigned flags, const double *gw,
                                     float *__restrict__ tmp_a, float *__restrict__ tmp_b, float *__restrict__ hes,
                                     BlockScratch &bs, uint32_t *wide_hist = nullptr) {
    const int tid = threadIdx.x, nt = blockDim.x, n = rows * cols;
    if ((flags & 7u) == 1u && wide_hist != nullptr && rows >= 5 && cols >= 5 && (n & 1) && (nt == 128 || nt == 256 || nt == 512)) {
        PeakStats fast;
        fast.r = peak_r;
        fast.h = hes_norm_fast(best, rows, cols, peak_idx, hes, wide_hist, bs, fast.hmed, fast.hsd);
        fast.rmed = 0.0f; fast.rsd = 1.0f;
        return fast;
    }
    const int y_first = tid / cols, x_first = tid - y_first * cols, dy = nt / cols, dx = nt - dy * cols;
    const float *src = best;
    if (flags & 2u) {               // hes_smth
        for (int k = tid, y = y_first, x = x_first; k < n; k += nt) {
            tmp_a[k] = gauss_at(best, rows, cols, y, x, 0, gw);
            x += dx; y += dy; if (x >= cols) { x -= cols; ++y; }
        }
        __syncthreads();
        for (int k = tid, y = y_first, x = x_first; k < n; k += nt) {
            tmp_b[k] = gauss_at(tmp_a, rows, cols, y, x, 1, gw);
            x += dx; y += dy; if (x >= cols) { x -= cols; ++y; }
        }
        __syncthreads();
        src = tmp_b;
    }
    if (rows >= 5 && cols >= 5) {
        // interior (2 <= y < rows-2, 2 <= x < cols-2): branch-free 5-point stencils, same rounding sequence as
        // np.gradient(np.gradient(.)) away from the edges
        const int iw = cols - 4, ni = (rows - 4) * iw;
        const int iy_first = tid / iw, ix_first = tid - iy_first * iw, idy = nt / iw, idx = nt - idy * iw;
        for (int k = tid, y = iy_first, x = ix_first; k < ni; k += nt) {
            const float *p = src + (size_t)(y + 2) * cols + (x + 2);
            const float c = p[0];
            const float gxp = __fmul_rn(__fsub_rn(p[2], c), 0.5f), gxm = __fmul_rn(__fsub_rn(c, p[-2]), 0.5f);
            const float gyp = __fmul_rn(__fsub_rn(p[2 * cols], c), 0.5f), gym = __fmul_rn(__fsub_rn(c, p[-2 * cols]), 0.5f);
            const double a2 = (double)__fmul_rn(__fsub_rn(gxp, gxm), 0.5f), b2 = (double)__fmul_rn(__fsub_rn(gyp, gym), 0.5f);
            hes[(size_t)(y + 2) * cols + (x + 2)] =
                __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(a2, a2), __dmul_rn(b2, b2))));
            x += idx; y += idy; if (x >= iw) { x -= iw; ++y; }
        }
        // border frame: two rows top and bottom, two columns left and right
        const int nb = 4 * cols + 4 * (rows - 4);
        for (int k = tid; k < nb; k += nt) {
            int y, x;
            if (k < 4 * cols) { const int r = k / cols; x = k - r * cols; y = r < 2 ? r : rows - 4 + r; }
            else { const int q = k - 4 * cols, r = q >> 2, cidx = q & 3; y = r + 2; x = cidx < 2 ? cidx : cols - 4 + cidx; }
            hes[(size_t)y * cols + x] = hessian_at(src, rows, cols, y, x);
        }
    } else {
        for (int k = tid, y = y_first, x = x_first; k < n; k += nt) {
            hes[k] = hessian_at(src, rows, cols, y, x);
            x += dx; y += dy; if (x >= cols) { x -= cols; ++y; }
        }
    }
    __syncthreads();
    PeakStats ps;
    ps.h = hes[peak_idx];
    ps.r = peak_r;
    ps.hmed = 0.0f; ps.hsd = 1.0f; ps.rmed = 0.0f; ps.rsd = 1.0f;
    if (flags & 1u) {               // hes_norm
        const float med = block_median(hes, n, bs, wide_hist);
        const float sd = block_std(hes, n, bs);
        ps.h = __fdiv_rn(__fsub_rn(ps.h, med), sd);
        ps.hmed = med; ps.hsd = sd;
    }
    if (flags & 4u) {               // mcc_norm
        const float med = block_median(best, n, bs, wide_hist);
        const float sd = block_std(best, n, bs);
        ps.r = __fdiv_rn(__fsub_rn(peak_r, med), sd);
        ps.rmed = med; ps.rsd = sd;
    }
    return ps;
}

// Sub-pixel offsets of the peak (SID_SUBPIXEL): the vertex of the parabola through the peak b and its neighbours a (lower
// index) and c (higher index), one axis at a time, on the RAW float32 map of the winning angle (the map peak_statistics
// reads, never the smoothed one).  p = b - a, q = b - c, d = (p - q) / (2 (p + q)) in FP64 intrinsics without
// contraction, so a NumPy float64 restatement is bit-identical.  A peak on the first or last column (row)
// gives +0.0 on that axis.  No guard is needed: the map is finite (flat template -> 1, tiny variance -> 0) and (bi, bj) is
// np.argmax's FIRST maximum, so the lower-index neighbour is strictly smaller and the other one no larger: p > 0,
// q >= 0, p + q > 0.  |p - q| <= p + q survives monotone rounding, so |d| <= 0.5 exactly, and d = +0.5 exactly when the
// higher-index neighbour ties the peak.  Called by the one thread that writes the row.
struct PeakOffsets { double dx, dy; };
__device__ __forceinline__ double parabola_vertex(float a, float b, float c) {
    const double p = __dsub_rn((double)b, (double)a), q = __dsub_rn((double)b, (double)c);
    return __ddiv_rn(__dsub_rn(p, q), __dmul_rn(2.0, __dadd_rn(p, q)));
}
__device__ __forceinline__ PeakOffsets peak_offsets(const float *map, int rows, int cols, int bi, int bj) {
    const float *pk = map + (size_t)bi * cols + bj;
    PeakOffsets d;
    d.dx = (bj > 0 && bj < cols - 1) ? parabola_vertex(pk[-1], pk[0], pk[1]) : 0.0;
    d.dy = (bi > 0 && bi < rows - 1) ? parabola_vertex(pk[-cols], pk[0], pk[cols]) : 0.0;
    return d;
}

// ---------------------------------------------------------------- TMA (cp.async.bulk.tensor) + mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 2-D tile of a uint8 image -> shared memory; (x, y) = element coordinates of the tile's first byte
__device__ __forceinline__ void tma_load_2d(void *dst, const void *tmap, int x, int y, unsigned long long *bar) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // earlier generic-proxy accesses to dst are done
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------- argmax helpers
// key = (sortable value << 32) | (~flat_index): max() gives the largest value and,
// among equal values, the lowest row-major index (np.argmax semantics).
__device__ __forceinline__ unsigned long long peak_key(float v, uint32_t idx) {
    return ((unsigned long long)f32_key(v) << 32) | (unsigned long long)(0xffffffffu - idx);
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, k, o);
        k = other > k ? other : k;
    }
    return k;
}

// Secondary peaks (SID_PEAKS, rule in include/sid_b200.h): the SID_N_PEAKS best local maxima of the raw winning map other
// than the primary (flat index peak_idx), and their records c2, r2, r, h, computed as the row computes its own.  One sweep
// over the map; every thread keeps a sorted top 3 of peak_key()s (value, then lowest index), then three rounds of a
// block-wide maximum pop the best ones.  `hes` and ps: what peak_statistics left.  (c2fg, r2fg): the point's first guess;
// H x W: its window.  Every thread of the CTA calls this after peak_statistics; thread 0 writes the 3 x 4 doubles at dst
// (NaN records where fewer peaks exist).  bs.red is reused.
constexpr int N_PEAKS = 3;
__device__ __noinline__ void store_secondary_peaks(double *dst, const float *map, const float *hes, int rows, int cols,
                                                   int peak_idx, const PeakStats ps, unsigned flags, double c2fg,
                                                   double r2fg, int H, int W, int s, BlockScratch &bs) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = (nt + 31) >> 5, n = rows * cols;
    unsigned long long t0 = 0ull, t1 = 0ull, t2 = 0ull;
    for (int p = tid; p < n; p += nt) {
        if (p == peak_idx) continue;
        const int i = p / cols, j = p - i * cols;
        const float v = map[p];
        // lower flat index (row above, left neighbour): strictly smaller; higher (right neighbour, row below): not larger
        bool pk = true;
        if (j > 0) pk = pk && map[p - 1] < v;
        if (j < cols - 1) pk = pk && map[p + 1] <= v;
        if (i > 0) {
            const float *u = map + p - cols;
            pk = pk && u[0] < v && (j == 0 || u[-1] < v) && (j == cols - 1 || u[1] < v);
        }
        if (i < rows - 1) {
            const float *d = map + p + cols;
            pk = pk && d[0] <= v && (j == 0 || d[-1] <= v) && (j == cols - 1 || d[1] <= v);
        }
        if (!pk) continue;
        const unsigned long long k = peak_key(v, (uint32_t)p);
        if (k > t2) {
            if (k > t1) { t2 = t1; if (k > t0) { t1 = t0; t0 = k; } else t1 = k; }
            else t2 = k;
        }
    }
    unsigned long long *red = reinterpret_cast<unsigned long long *>(bs.red);
    unsigned long long top[N_PEAKS];
#pragma unroll
    for (int r = 0; r < N_PEAKS; ++r) {
        const unsigned long long m = warp_max_u64(t0);
        __syncthreads();                                   // the previous reads of bs.red are done
        if (lane == 0) red[warp] = m;
        __syncthreads();
        unsigned long long best = 0ull;
        for (int w = 0; w < nw; ++w) best = red[w] > best ? red[w] : best;
        if (best != 0ull && t0 == best) { t0 = t1; t1 = t2; t2 = 0ull; }     // keys are unique: one thread pops
        top[r] = best;
    }
    if (tid != 0) return;
#pragma unroll
    for (int r = 0; r < N_PEAKS; ++r) {
        double *o = dst + 4 * r;
        if (top[r] == 0ull) { o[0] = o[1] = o[2] = o[3] = nan(""); continue; }
        const int p = (int)(0xffffffffu - (uint32_t)(top[r] & 0xffffffffull));
        const int i = p / cols, j = p - i * cols;
        double c2 = c2fg + ((double)j - (double)(W - s) / 2.0);
        double r2 = r2fg + ((double)i - (double)(H - s) / 2.0);
        if (flags & 8u) {                                  // SID_SUBPIXEL: p > 0 and q >= 0 as for the primary
            const PeakOffsets d = peak_offsets(map, rows, cols, i, j);
            c2 = __dadd_rn(c2, d.dx);
            r2 = __dadd_rn(r2, d.dy);
        }
        float rv = map[p], hv = hes[p];
        if (flags & 4u) rv = __fdiv_rn(__fsub_rn(rv, ps.rmed), ps.rsd);
        if (flags & 1u) hv = __fdiv_rn(__fsub_rn(hv, ps.hmed), ps.hsd);
        o[0] = c2; o[1] = r2; o[2] = (double)rv; o[3] = (double)hv;
    }
}

}  // namespace sid
