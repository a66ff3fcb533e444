// sid_single_kernels.cuh -- kernels behind the single-call entry points
// (sid_get_template, sid_match_template, sid_get_hessian, sid_rotate_and_match).
// They work on maps of any size in global memory and share every arithmetic helper
// with the fused batched kernel, so both paths give identical numbers.
#pragma once
#include "sid_common.cuh"
#include "sid_pm_kernel.cuh"

namespace sid {

// ---- get_template for n_angles angles of one point: out[a][s][s], stats[a] = {sum, sqsum, has_zero}
__global__ void __launch_bounds__(256) templates_kernel(const uint8_t *__restrict__ img, int rows, int cols, long long pitch,
                                                        double c, double r, const double *__restrict__ tab, int s, int order,
                                                        uint8_t *__restrict__ out, uint32_t *__restrict__ stats) {
    const int a = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const double *tb = tab + 4 * a;
    const double cs = tb[0], sn = tb[1];
    const double off0 = __dsub_rn(r, tb[2]), off1 = __dsub_rn(c, tb[3]);
    uint32_t lsum = 0, lsq = 0, lzero = 0;
    const int ss = s * s;
    for (int k = tid; k < ss; k += blockDim.x) {
        const int i = k / s, j = k - i * s;
        const uint32_t v = template_pixel(img, rows, cols, pitch, off0, off1, cs, sn, i, j, order);
        out[(size_t)a * ss + k] = (uint8_t)v;
        lsum += v; lsq += v * v; lzero |= (v == 0);
    }
    for (int o = 16; o > 0; o >>= 1) {
        lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        lsq += __shfl_xor_sync(0xffffffffu, lsq, o);
        lzero |= __shfl_xor_sync(0xffffffffu, lzero, o);
    }
    if (lane == 0) {
        atomicAdd(&stats[3 * a + 0], lsum);
        atomicAdd(&stats[3 * a + 1], lsq);
        if (lzero) atomicOr(&stats[3 * a + 2], 1u);
    }
}

// ---- sum / sum of squares of an arbitrary template (th x tw, pitch tp) -> stats[0..1]
__global__ void __launch_bounds__(256) template_sums_kernel(const uint8_t *__restrict__ tpl, int th, int tw, long long tp,
                                                            uint32_t *__restrict__ stats) {
    uint32_t lsum = 0, lsq = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < th * tw; k += gridDim.x * blockDim.x) {
        const uint32_t v = tpl[(size_t)(k / tw) * tp + (k % tw)];
        lsum += v; lsq += v * v;
    }
    for (int o = 16; o > 0; o >>= 1) {
        lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        lsq += __shfl_xor_sync(0xffffffffu, lsq, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&stats[0], lsum); atomicAdd(&stats[1], lsq); }
}

// ---- integral images (uint32, wrap-around arithmetic: window sums stay < 2^32)
// isum/isq are (H+1) x (W+1); pass 1 = prefix along each row, pass 2 = prefix down each column.
__global__ void integral_rows_kernel(const uint8_t *__restrict__ img, int H, int W, long long pitch,
                                     uint32_t *__restrict__ isum, uint32_t *__restrict__ isq) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y > H) return;
    uint32_t *rs = isum + (size_t)y * (W + 1), *rq = isq + (size_t)y * (W + 1);
    rs[0] = 0; rq[0] = 0;
    if (y == 0) { for (int x = 1; x <= W; ++x) { rs[x] = 0; rq[x] = 0; } return; }
    const uint8_t *row = img + (size_t)(y - 1) * pitch;
    uint32_t s = 0, q = 0;
    for (int x = 0; x < W; ++x) { const uint32_t v = row[x]; s += v; q += v * v; rs[x + 1] = s; rq[x + 1] = q; }
}
__global__ void integral_cols_kernel(int H, int W, uint32_t *__restrict__ isum, uint32_t *__restrict__ isq) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x > W) return;
    uint32_t s = 0, q = 0;
    for (int y = 0; y <= H; ++y) {
        const size_t k = (size_t)y * (W + 1) + x;
        s += isum[k]; q += isq[k]; isum[k] = s; isq[k] = q;
    }
}

// ---- tiled TM_CCOEFF_NORMED: each CTA computes MT_ROWS x MT_COLS outputs
constexpr int MT_TX = 8;
constexpr int MT_ROWS = 32;
constexpr int MT_COLS = 4 * MT_TX * 2;   // 64
struct MtArgs {
    const uint8_t *img; int H, W; long long pitch;          // pitch % 4 == 0, base 4-aligned
    const uint8_t *tpl; int th, tw; long long tp;
    const uint32_t *isum, *isq;                              // (H+1) x (W+1)
    const uint32_t *tstats;                                  // sum, sqsum of the template
    double inv_area, sqrt_inv_area;
    float *out;                                              // RH x RW
    int wpw, tpw;                                            // smem pitches in words
};
__global__ void __launch_bounds__(256) match_template_kernel(const MtArgs a) {
    extern __shared__ __align__(16) unsigned char mt_smem[];
    const int tid = threadIdx.x;
    const int RH = a.H - a.th + 1, RW = a.W - a.tw + 1;
    const int ty0 = blockIdx.y * MT_ROWS, tx0 = blockIdx.x * MT_COLS;
    const int rows_in = min(MT_ROWS, RH - ty0) + a.th - 1;
    uint32_t *win32 = reinterpret_cast<uint32_t *>(mt_smem);
    uint32_t *tpl32 = win32 + (MT_ROWS + a.th - 1) * a.wpw + PM_WIN_SLACK;
    // stage window tile (tx0 is a multiple of 4 -> already word aligned); columns past the image read as 0
    for (int t = tid; t < rows_in * a.wpw; t += blockDim.x) {
        const int y = t / a.wpw, k = t - y * a.wpw;
        const long long gx = (long long)tx0 + 4 * k;
        uint32_t v = 0;
        const uint8_t *row = a.img + (size_t)(ty0 + y) * a.pitch;
        if (gx + 3 < a.W) v = __ldg(reinterpret_cast<const uint32_t *>(row + gx));
        else { for (int b = 0; b < 4; ++b) if (gx + b < a.W) v |= (uint32_t)row[gx + b] << (8 * b); }
        win32[t] = v;
    }
    for (int t = tid; t < a.th * a.tpw; t += blockDim.x) {
        const int i = t / a.tpw, k = t - i * a.tpw;
        uint32_t v = 0;
        for (int b = 0; b < 4; ++b) { const int j = 4 * k + b; if (j < a.tw) v |= (uint32_t)a.tpl[(size_t)i * a.tp + j] << (8 * b); }
        tpl32[t] = v;
    }
    __syncthreads();
    const TemplStats st = templ_stats(a.tstats[0], a.tstats[1], a.inv_area, a.sqrt_inv_area);
    const int nchunk = (a.tw + 15) / 16;
    // 256 threads = 32 rows x 4 classes x 2 column groups
    const int p = tid & 3, y = (tid >> 2) & 31, cg = tid >> 7;
    const int oy = ty0 + y;
    if (oy >= RH) return;
    unsigned acc[MT_TX];
#pragma unroll
    for (int k = 0; k < MT_TX; ++k) acc[k] = 0u;
    const int q0 = cg * MT_TX;
    mac_rows_any<MT_TX>(win32 + y * a.wpw + q0, a.wpw, tpl32, a.tpw, a.th, nchunk, 8 * p, acc);
    const int IW = a.W + 1;
#pragma unroll
    for (int tx = 0; tx < MT_TX; ++tx) {
        const int ox = tx0 + 4 * (q0 + tx) + p;
        if (ox < RW) {
            const size_t k00 = (size_t)oy * IW + ox, k10 = (size_t)(oy + a.th) * IW + ox;
            const uint32_t ws = a.isum[k00] - a.isum[k00 + a.tw] - a.isum[k10] + a.isum[k10 + a.tw];
            const uint32_t wq = a.isq[k00] - a.isq[k00 + a.tw] - a.isq[k10] + a.isq[k10 + a.tw];
            a.out[(size_t)oy * RW + ox] = ncc_value((long long)acc[tx], ws, window_den(ws, wq, a.inv_area), st);
        }
    }
}

// ---- np.argmax of a map: single CTA, result key (see peak_key)
__global__ void __launch_bounds__(1024) argmax_kernel(const float *__restrict__ map, int n, unsigned long long *__restrict__ out) {
    __shared__ unsigned long long sk[32];
    unsigned long long key = 0ull;
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const unsigned long long k2 = peak_key(map[k], (uint32_t)k);
        key = k2 > key ? k2 : key;
    }
    key = warp_max_u64(key);
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x < 32) {
        key = threadIdx.x < (blockDim.x >> 5) ? sk[threadIdx.x] : 0ull;
        key = warp_max_u64(key);
        if (threadIdx.x == 0) *out = key;
    }
}

// ---- tail of rotate_and_match on a map in global memory: out[0] = r, out[1] = h; with SID_SUBPIXEL also
// offsets[0] = dx, offsets[1] = dy (peak_offsets)
struct PeakArgs { const float *best; int rows, cols, idx; float r; unsigned flags; double gw[5]; float *tmp_a, *tmp_b, *hes; float *out; double *offsets; };
__global__ void __launch_bounds__(1024) peak_stats_kernel(const PeakArgs a) {
    __shared__ BlockScratch bs;
    if (threadIdx.x == 0 && (a.flags & 8u)) {
        const int bi = a.idx / a.cols;
        const PeakOffsets d = peak_offsets(a.best, a.rows, a.cols, bi, a.idx - bi * a.cols);
        a.offsets[0] = d.dx; a.offsets[1] = d.dy;
    }
    const PeakStats ps = peak_statistics(a.best, a.rows, a.cols, a.idx, a.r, a.flags, a.gw, a.tmp_a, a.tmp_b, a.hes, bs);
    if (threadIdx.x == 0) { a.out[0] = ps.r; a.out[1] = ps.h; }
}

// ---- get_hessian of a whole map: out = hes or (hes - median) / std
struct HesArgs { const float *ccm; int rows, cols; unsigned flags; double gw[5]; float *tmp_a, *tmp_b; float *out; };
__global__ void __launch_bounds__(1024) hessian_map_kernel(const HesArgs a) {
    __shared__ BlockScratch bs;
    const int tid = threadIdx.x, nt = blockDim.x, n = a.rows * a.cols;
    const float *src = a.ccm;
    if (a.flags & 2u) {
        for (int k = tid; k < n; k += nt) a.tmp_a[k] = gauss_at(a.ccm, a.rows, a.cols, k / a.cols, k % a.cols, 0, a.gw);
        __syncthreads();
        for (int k = tid; k < n; k += nt) a.tmp_b[k] = gauss_at(a.tmp_a, a.rows, a.cols, k / a.cols, k % a.cols, 1, a.gw);
        __syncthreads();
        src = a.tmp_b;
    }
    for (int k = tid; k < n; k += nt) a.out[k] = hessian_at(src, a.rows, a.cols, k / a.cols, k % a.cols);
    __syncthreads();
    if (a.flags & 1u) {
        const float med = block_median(a.out, n, bs);
        const float sd = block_std(a.out, n, bs);
        __syncthreads();
        for (int k = tid; k < n; k += nt) a.out[k] = __fdiv_rn(__fsub_rn(a.out[k], med), sd);
    }
}

}  // namespace sid
