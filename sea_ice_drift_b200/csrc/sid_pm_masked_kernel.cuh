// sid_pm_masked_kernel.cuh -- masked correlation (SID_MASKED) for the rows the reference returns as NaN because a
// template holds a 0 pixel (land, no-data, samples outside image 1).
//
// For one angle's template T (s x s) the mask is M = (T > 0), n = sum M, St = sum T, Stt = sum T^2.  At map position p,
// over the window patch W (window zeros are data, only the template is masked):
//   C = sum T W,  Sw = sum M W,  Sww = sum M W^2                          (exact: u8 x u8 products, < 2^32)
//   num = n C - St Sw,  vt = n Stt - St^2,  vw = n Sww - Sw^2             (exact int64)
//   r = (double)num / (sqrt((double)vt) * sqrt((double)vw)), clamped to [-1, 1], rounded to float32;  vw = 0 -> r = 0
// i.e. the Pearson correlation over the valid template pixels, what cv2.matchTemplate(..., TM_CCOEFF_NORMED,
// mask=(T > 0)) computes.  A row is matched this way when every angle's template has n >= ceil(s^2 / 2) and vt > 0.
//
// The sums come from IDP.4A on the CUDA cores: a thread owns one map position and walks the template four bytes at a
// time, with the window bytes masked by M first (V = W & M), so that C = dp4a(V, T), Sw = dp4a(V, 1) and
// Sww = dp4a(V, V).  Template and mask words sit in shared memory and are read as broadcasts; the window is read from
// global memory (L1) as aligned words, so any window size is taken.  Masked rows are a minority of a grid: the kernel
// favours simplicity over throughput.
#pragma once
#include "sid_common.cuh"
#include "sid_pm_kernel.cuh"

namespace sid {

constexpr int PM_MASKED_THREADS = 256;
constexpr int PM_MASKED_MAX_NW = 32;                // template row words at img_size 128

// Template of one angle for the masked rule: byte j of word q of row i is T[i][4q + j] (0 beyond s), its mask word has
// 0xFF where T > 0.  n / St / Stt accumulate in *stats (zeroed by the caller).  Every sample goes through template_pixel
// (template_sample's bounds).
__device__ __forceinline__ void masked_template(const uint8_t *__restrict__ img, int rows, int cols, long long pitch,
                                                double c, double r, const double *__restrict__ tab, int s, int order,
                                                uint32_t *__restrict__ tw, uint32_t *__restrict__ mw, uint32_t *stats) {
    const double cs = tab[0], sn = tab[1];
    const double off0 = __dsub_rn(r, tab[2]), off1 = __dsub_rn(c, tab[3]);
    const int nw = (s + 3) >> 2;
    uint32_t ln = 0, lsum = 0, lsq = 0;
    unsigned char *tb = reinterpret_cast<unsigned char *>(tw), *mb = reinterpret_cast<unsigned char *>(mw);
    for (int k = threadIdx.x; k < s * s; k += blockDim.x) {
        const int i = k / s, j = k - i * s;
        const uint32_t v = template_pixel(img, rows, cols, pitch, off0, off1, cs, sn, i, j, order);
        tb[i * nw * 4 + j] = (unsigned char)v;
        mb[i * nw * 4 + j] = v ? 0xFFu : 0u;
        ln += v != 0; lsum += v; lsq += v * v;
    }
    ln = __reduce_add_sync(0xffffffffu, ln);
    lsum = __reduce_add_sync(0xffffffffu, lsum);
    lsq = __reduce_add_sync(0xffffffffu, lsq);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&stats[0], ln); atomicAdd(&stats[1], lsum); atomicAdd(&stats[2], lsq); }
}

// The masked correlation at the window patch whose top-left byte is `win` (row pitch `pitch`, a multiple of 4).  Reads
// whole aligned words: up to 3 bytes before the patch and 6 bytes past its last column, inside the same rows (the
// resident layout pads every row by >= 16 bytes), where the zero template and mask bytes cancel them.
__device__ __forceinline__ float masked_ncc_at(const uint8_t *win, long long pitch, const uint32_t *__restrict__ tw,
                                               const uint32_t *__restrict__ mw, int s, long long n, long long st,
                                               double sqrt_vt) {
    const int nw = (s + 3) >> 2;
    const int sh = (int)((uintptr_t)win & 3u) * 8;
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(win - ((uintptr_t)win & 3u));
    const long long pw = pitch >> 2;
    uint32_t c = 0, sw = 0, sww = 0;
    for (int i = 0; i < s; ++i) {
        uint32_t lo = __ldg(wp);
        for (int q = 0; q < nw; ++q) {
            const uint32_t hi = __ldg(wp + q + 1);
            const uint32_t v = __funnelshift_r(lo, hi, sh) & mw[i * nw + q];
            lo = hi;
            c = __dp4a(v, tw[i * nw + q], c);
            sw = __dp4a(v, 0x01010101u, sw);
            sww = __dp4a(v, v, sww);
        }
        wp += pw;
    }
    const long long num = n * (long long)c - st * (long long)sw;
    const long long vw = n * (long long)sww - (long long)sw * (long long)sw;
    if (vw == 0) return 0.0f;
    double rr = __ddiv_rn((double)num, __dmul_rn(sqrt_vt, __dsqrt_rn((double)vw)));
    rr = fmin(fmax(rr, -1.0), 1.0);
    return __double2float_rn(rr);
}

__host__ __device__ inline bool masked_template_ok(int s, long long n, long long st, long long stt) {
    return 2 * n >= (long long)s * s && n * stt - st * st > 0;
}

// Candidate rows of the masked pass: the points the correlation launches left with status 0 (SID_PT_NAN)
__global__ void masked_candidates_kernel(const int *__restrict__ status, long long n, int *__restrict__ cand,
                                         unsigned *__restrict__ count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool take = i < n && status[i] == 0;
    const unsigned m = __ballot_sync(0xffffffffu, take);
    const int lane = threadIdx.x & 31;
    unsigned base = 0;
    if (lane == 0 && m) base = atomicAdd(count, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (take) cand[base + __popc(m & ((1u << lane) - 1u))] = (int)i;
}

struct PmMaskedShared {
    uint32_t tw[128 * PM_MASKED_MAX_NW], mw[128 * PM_MASKED_MAX_NW];
    uint32_t hist[2048];                 // peak_statistics' wide histogram
    BlockScratch bs;
    uint32_t stats[3];
    unsigned long long key;
    unsigned item;
    int ok;
};

// One candidate row per CTA (work stealing over a.order[0 .. *n_cand)).  The winning angle's float map goes through the
// existing peak_statistics / peak_offsets / pm_store_map / pm_store_template.  Per-CTA global scratch: two map slots (the
// best so far and the current angle), the Hessian map and a smoothing temporary, max_rr floats each.
// PEAKS: SID_PEAKS, a separate instantiation as for pm_points_kernel.
template <bool PEAKS>
__global__ void __launch_bounds__(PM_MASKED_THREADS) pm_masked_kernel(const PmArgs a, const unsigned *__restrict__ n_cand) {
    __shared__ PmMaskedShared S;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, s = a.s;
    float *slab = reinterpret_cast<float *>(a.scratch + (size_t)blockIdx.x * a.scratch_per_cta);
    auto slot = [&](int k) { return slab + (size_t)k * a.max_rr; };
    float *hes = slab + 2 * (size_t)a.max_rr, *tmp_b = slab + 3 * (size_t)a.max_rr;
    for (int k = tid; k < 128 * PM_MASKED_MAX_NW; k += nt) { S.tw[k] = 0u; S.mw[k] = 0u; }     // padding bytes stay 0
    const long long total = min((long long)*n_cand, a.n);
    for (;;) {
        __syncthreads();
        if (tid == 0) S.item = atomicAdd(a.counter, 1u);
        __syncthreads();
        if ((long long)S.item >= total) break;
        const long long pt = a.order[S.item];
        const double c1 = a.c1[pt], r1 = a.r1[pt], c2 = a.c2fg[pt], r2 = a.r2fg[pt];
        long long x0, y0;
        int W, H;
        if (!pm_window_rect(a, c1, r1, c2, r2, a.border[pt], x0, y0, W, H)) continue;   // not a NaN row of the rule
        const int RH = H - s + 1, RW = W - s + 1, RR = RH * RW;
        if (RR > a.max_rr) continue;
        // 1. every angle's template must qualify
        if (tid == 0) S.ok = 1;
        for (int an = 0; an < a.n_angles; ++an) {
            __syncthreads();                                    // the previous angle's statistics have been read
            if (tid < 3) S.stats[tid] = 0u;
            __syncthreads();
            masked_template(a.img1, a.rows1, a.cols1, a.pitch1, c1, r1, a.tab + 4 * an, s, a.rot_order, S.tw, S.mw, S.stats);
            __syncthreads();
            if (tid == 0 && !masked_template_ok(s, S.stats[0], S.stats[1], S.stats[2])) S.ok = 0;
        }
        __syncthreads();
        if (!S.ok) continue;
        // 2. the masked map of every angle; first maximum of each, a later angle wins on strict '>'
        const uint8_t *win0 = a.img2 + y0 * a.pitch2 + x0;
        float best_r = -INFINITY;
        int best_a = -1, best_idx = 0, best_slot = 0, cur = 0;
        for (int an = 0; an < a.n_angles; ++an) {
            __syncthreads();                                    // the previous angle's key has been read
            if (tid < 3) S.stats[tid] = 0u;
            if (tid == 0) S.key = 0ull;
            __syncthreads();
            masked_template(a.img1, a.rows1, a.cols1, a.pitch1, c1, r1, a.tab + 4 * an, s, a.rot_order, S.tw, S.mw, S.stats);
            __syncthreads();
            const long long n = S.stats[0], st = S.stats[1], stt = S.stats[2];
            const double sqrt_vt = __dsqrt_rn((double)(n * stt - st * st));
            float *map = slot(cur);
            unsigned long long key = 0ull;
            for (int p = tid; p < RR; p += nt) {
                const int y = p / RW, x = p - y * RW;
                const float v = masked_ncc_at(win0 + (long long)y * a.pitch2 + x, a.pitch2, S.tw, S.mw, s, n, st, sqrt_vt);
                map[p] = v;
                const unsigned long long k2 = peak_key(v, (uint32_t)p);
                key = k2 > key ? k2 : key;
            }
            key = warp_max_u64(key);
            if (lane == 0 && key) atomicMax(&S.key, key);
            __syncthreads();
            const float v = key_f32((uint32_t)(S.key >> 32));      // the same in every thread
            if (v > best_r) {
                best_r = v; best_a = an; best_slot = cur; cur ^= 1;
                best_idx = (int)(0xffffffffu - (uint32_t)(S.key & 0xffffffffull));
            }
        }
        if (best_a < 0) continue;
        // 3. the tail of every other path on the winning float map
        const float *best = slot(best_slot);
        __syncthreads();
        if (a.maps_out) pm_store_map(a, pt, best, RR);
        const PeakStats ps = peak_statistics(best, RH, RW, best_idx, best_r, a.flags, a.gw, slot(best_slot ^ 1), tmp_b, hes,
                                             S.bs, S.hist);
        if (tid == 0) {
            const int bi = best_idx / RW, bj = best_idx - bi * RW;
            double *o = a.out + 5 * pt;
            o[0] = c2 + ((double)bj - (double)(W - s) / 2.0);
            o[1] = r2 + ((double)bi - (double)(H - s) / 2.0);
            if (a.flags & 8u) {             // SID_SUBPIXEL
                const PeakOffsets d = peak_offsets(best, RH, RW, bi, bj);
                o[0] = __dadd_rn(o[0], d.dx);
                o[1] = __dadd_rn(o[1], d.dy);
            }
            o[2] = a.angles[best_a];
            o[3] = (double)ps.r;
            o[4] = (double)ps.h;
            if (a.status) a.status[pt] = 2;                 // SID_PT_MASKED
        }
        if constexpr (PEAKS) store_secondary_peaks(a.peaks + 12 * pt, best, hes, RH, RW, best_idx, ps, a.flags, c2, r2, H, W, s, S.bs);
        if (a.tpl_out) pm_store_template(a, pt, best_a);
    }
}

// Per-CTA global scratch of pm_masked_kernel (bytes)
__host__ __device__ inline size_t pm_masked_scratch_bytes(int max_rr) { return ((size_t)max_rr * 4 * 4 + 255) & ~(size_t)255; }

// sid_rotate_and_match: the masked map of one angle over an explicit window (H x W at `img`, any size); template bytes
// tpl (s x s) with its statistics n / St / Stt computed on the host
__global__ void __launch_bounds__(256) masked_map_kernel(const uint8_t *__restrict__ img, int H, int W, long long pitch,
                                                         const uint8_t *__restrict__ tpl, int s, long long n, long long st,
                                                         long long stt, float *__restrict__ out) {
    __shared__ uint32_t tw[128 * PM_MASKED_MAX_NW], mw[128 * PM_MASKED_MAX_NW];
    const int nw = (s + 3) >> 2;
    for (int k = threadIdx.x; k < s * nw; k += blockDim.x) {
        const int i = k / nw, q = k - i * nw;
        uint32_t t = 0u, m = 0u;
        for (int b = 0; b < 4; ++b) {
            const int j = 4 * q + b;
            const uint32_t v = j < s ? tpl[i * s + j] : 0u;
            t |= v << (8 * b);
            m |= (v ? 0xFFu : 0u) << (8 * b);
        }
        tw[k] = t; mw[k] = m;
    }
    __syncthreads();
    const int RW = W - s + 1, RR = (H - s + 1) * RW;
    const double sqrt_vt = __dsqrt_rn((double)(n * stt - st * st));
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < RR; p += gridDim.x * blockDim.x) {
        const int y = p / RW, x = p - y * RW;
        out[p] = masked_ncc_at(img + (long long)y * pitch + x, pitch, tw, mw, s, n, st, sqrt_vt);
    }
}

}  // namespace sid
