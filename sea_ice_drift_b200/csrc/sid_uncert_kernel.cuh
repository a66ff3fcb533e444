// sid_uncert_kernel.cuh -- per-vector covariance of the sub-pixel offsets (SID_UNCERT) by correlation statistics
// (Wieneke 2015, "PIV uncertainty quantification from correlation statistics", Meas. Sci. Technol. 26, 074002).
//
// The rule is written out in include/sid_b200.h.  In short, for a VALID or MASKED row with winning template T, mask M,
// integer peak P0 = (bi, bj) and its four neighbours X-, X+ (along the row) and Y-, Y+ (down the column):
//   t_k = M_k (n T_k - St),  w_k(P) = M_k (n W_P,k - Sw(P)),  x_k(P) = t_k w_k(P)               (exact int32 / int64)
//   A(P) = sum x_k(P),  V(P) = sum w_k(P)^2,  Vt = sum t_k^2,  S(P, Q) = sum x_k(P) x_k(Q)       (exact int64 / int128)
//   K(P, Q) = D(n S - A(P) A(Q)) / (((D(n) D(Vt)) sqrt(D(V(P)))) sqrt(D(V(Q))))                   (IEEE double)
// K is the population covariance of the per-pixel contributions to the Pearson correlation at P and Q, times n.  The
// covariance of (dx, dy) is K propagated linearly through the parabola vertex of SID_SUBPIXEL.
//
// The pass runs after every other launch of a call and reads only what they left: the table (winning angle, c2, r2) and
// the status.  It changes none of them.  One row per CTA (grid-stride), UNC_THREADS threads:
//   1. the winning template into shared memory (template_pixel, as pm_store_template), with n, St and Stt;
//   2. the integer peak among the at most 2 x 2 integer positions within 0.5 + 1e-6 of the table's sub-pixel position:
//      the largest recomputed map value, ties to the lowest flat index (the map's first global maximum is among them);
//   3. the map values at P0, X-, X+, Y-, Y+ (the parabola's inputs) and Sw at each;
//   4. one sweep over the template's pixels for A, V, Vt and the 15 S sums; thread 0 finishes the record.
// Map values are recomputed from exact integer sums with the arithmetic of the kernels that made the map (templ_stats,
// window_den and ncc_finish for VALID rows, masked_ncc_at's for MASKED rows), so they are the map's bits.
#pragma once
#include "sid_common.cuh"
#include "sid_pm_kernel.cuh"

namespace sid {

constexpr int UNC_THREADS = 128;
constexpr int UNC_WARPS = UNC_THREADS / 32;
constexpr int UNC_NPOS = 5;                          // P0, X-, X+, Y-, Y+
constexpr int UNC_NPAIR = UNC_NPOS * (UNC_NPOS + 1) / 2;
constexpr int UNC_NWORDS = 2 * UNC_NPAIR + 2 * UNC_NPOS + 1;   // S (int128) | A | V | Vt, 64-bit words

struct UncShared {
    uint8_t tpl[128 * 128];
    unsigned long long red[UNC_WARPS][UNC_NWORDS];
    uint32_t stats[3];                               // n (T > 0), St, Stt of the template
    uint32_t sums[UNC_NPOS][3];                      // per position: sum T W, sum M W, sum M W^2
    int bi, bj;                                      // the integer peak, chosen by thread 0
};

// Correctly rounded (ties to even) signed 128-bit integer -> double: the top 64 bits with the bits below them folded
// into a sticky bit 0, rounded by the hardware conversion, then scaled exactly.
__device__ __forceinline__ double i128_to_double_rn(__int128 v) {
    const bool neg = v < 0;
    const unsigned __int128 u = neg ? (unsigned __int128)0 - (unsigned __int128)v : (unsigned __int128)v;
    const unsigned long long hi = (unsigned long long)(u >> 64), lo = (unsigned long long)u;
    double d;
    if (hi == 0ull) {
        d = __ull2double_rn(lo);
    } else {
        const int sh = 64 - __clzll((long long)hi);          // 1 ... 64
        const unsigned long long top = (unsigned long long)(u >> sh) | ((lo << (64 - sh)) != 0ull ? 1ull : 0ull);
        d = scalbn(__ull2double_rn(top), sh);
    }
    return neg ? -d : d;
}

__device__ __forceinline__ __int128 shfl_down_i128(__int128 v, int o) {
    const unsigned long long lo = __shfl_down_sync(0xffffffffu, (unsigned long long)v, o);
    const unsigned long long hi = __shfl_down_sync(0xffffffffu, (unsigned long long)((unsigned __int128)v >> 64), o);
    return (__int128)(((unsigned __int128)hi << 64) | lo);
}

// Sums at up to UNC_NPOS map positions (py[p], px[p]) of the window at `win`: sum T W, sum M W, sum M W^2 with M = 1
// (VALID) or T > 0 (MASKED).  Every product and sum fits uint32 (s <= 128).  Block-wide; the totals land in S.sums.
__device__ __forceinline__ void unc_position_sums(UncShared &S, int s, bool masked, const uint8_t *win,
                                                  long long pitch, const int (&py)[UNC_NPOS], const int (&px)[UNC_NPOS],
                                                  int np) {
    uint32_t acc[UNC_NPOS][3];
#pragma unroll
    for (int p = 0; p < UNC_NPOS; ++p) acc[p][0] = acc[p][1] = acc[p][2] = 0u;
    for (int k = threadIdx.x; k < s * s; k += blockDim.x) {
        const int i = k / s, j = k - i * s;
        const uint32_t t = S.tpl[k];
        const bool m = !masked || t != 0u;
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) {
            if (p < np) {
                const uint32_t w = __ldg(win + (long long)(py[p] + i) * pitch + (px[p] + j));
                const uint32_t wm = m ? w : 0u;
                acc[p][0] += t * w;
                acc[p][1] += wm;
                acc[p][2] += wm * wm;
            }
        }
    }
#pragma unroll
    for (int p = 0; p < UNC_NPOS; ++p)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint32_t v = __reduce_add_sync(0xffffffffu, acc[p][c]);
            if ((threadIdx.x & 31) == 0 && p < np) atomicAdd(&S.sums[p][c], v);
        }
}

// The raw float32 map value from a position's exact sums: VALID rows as every correlation kernel (templ_stats /
// window_den / ncc_finish, a flat template gives 1), MASKED rows as masked_ncc_at
__device__ __forceinline__ float unc_map_value(const uint32_t (&sm)[3], bool masked, const TemplStats &ts, double inv_area,
                                               long long n, long long st, double sqrt_vt) {
    if (!masked) {
        if (ts.flat) return 1.0f;
        const double num = __dsub_rn((double)sm[0], __dmul_rn((double)sm[1], ts.mean));
        return __double2float_rn(ncc_finish(num, __dmul_rn(window_den(sm[1], sm[2], inv_area), ts.norm)));
    }
    const long long num = n * (long long)sm[0] - st * (long long)sm[1];
    const long long vw = n * (long long)sm[2] - (long long)sm[1] * (long long)sm[1];
    if (vw == 0) return 0.0f;
    double rr = __ddiv_rn((double)num, __dmul_rn(sqrt_vt, __dsqrt_rn((double)vw)));
    rr = fmin(fmax(rr, -1.0), 1.0);
    return __double2float_rn(rr);
}

// ∂d/∂(a, b, c) of the parabola vertex d = (p - q) / (2 (p + q)), p = b - a, q = b - c
__device__ __forceinline__ void unc_vertex_grad(float a, float b, float c, double (&g)[3]) {
    const double p = __dsub_rn((double)b, (double)a), q = __dsub_rn((double)b, (double)c);
    const double w = __dmul_rn(__dadd_rn(p, q), __dadd_rn(p, q));
    g[0] = __ddiv_rn(-q, w);
    g[1] = __ddiv_rn(__dsub_rn(q, p), w);
    g[2] = __ddiv_rn(p, w);
}

// g^T K(u, v) g' over u in ul, v in vl: h_u = (K(u, v0) g'0 + K(u, v1) g'1) + K(u, v2) g'2, then (g0 h0 + g1 h1) + g2 h2
__device__ __forceinline__ double unc_quad(const double (&K)[UNC_NPOS][UNC_NPOS], const int (&ul)[3], const double (&g)[3],
                                           const int (&vl)[3], const double (&gp)[3]) {
    double h[3];
#pragma unroll
    for (int u = 0; u < 3; ++u)
        h[u] = __dadd_rn(__dadd_rn(__dmul_rn(K[ul[u]][vl[0]], gp[0]), __dmul_rn(K[ul[u]][vl[1]], gp[1])),
                         __dmul_rn(K[ul[u]][vl[2]], gp[2]));
    return __dadd_rn(__dadd_rn(__dmul_rn(g[0], h[0]), __dmul_rn(g[1], h[1])), __dmul_rn(g[2], h[2]));
}

// One row per CTA, grid-stride over rows 0 .. a.n - 1.  Writes unc[3 pt ...] = var_c, var_r, cov_cr for every row (NaN
// for rows that are neither VALID nor MASKED, and per the rule's NaN cases).  Reads a.out and a.status only.
__global__ void __launch_bounds__(UNC_THREADS) uncert_kernel(const PmArgs a, double *__restrict__ unc) {
    __shared__ UncShared S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, s = a.s;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    for (long long pt = blockIdx.x; pt < a.n; pt += gridDim.x) {
        const int status = a.status[pt];
        const double *row = a.out + 5 * pt;
        const double c1 = a.c1[pt], r1 = a.r1[pt], c2fg = a.c2fg[pt], r2fg = a.r2fg[pt];
        long long x0, y0;
        int W, H, an = -1;
        bool go = (status == 1 || status == 2) && pm_window_rect(a, c1, r1, c2fg, r2fg, a.border[pt], x0, y0, W, H);
        if (go) {
            const double ang = row[2];
            for (int k = 0; k < a.n_angles && an < 0; ++k) if (a.angles[k] == ang) an = k;
            go = an >= 0;
        }
        if (!go) {                                              // uniform over the CTA
            if (tid == 0) { unc[3 * pt] = qnan; unc[3 * pt + 1] = qnan; unc[3 * pt + 2] = qnan; }
            continue;
        }
        const bool masked = status == 2;
        const int RH = H - s + 1, RW = W - s + 1;
        const uint8_t *win = a.img2 + y0 * a.pitch2 + x0;
        __syncthreads();                                        // the previous row's shared state has been read
        if (tid < 3) S.stats[tid] = 0u;
        if (tid < UNC_NPOS * 3) S.sums[tid / 3][tid % 3] = 0u;
        __syncthreads();
        // 1. the winning template and its statistics
        {
            const double *tab = a.tab + 4 * an;
            const double cs = tab[0], sn = tab[1];
            const double off0 = __dsub_rn(r1, tab[2]), off1 = __dsub_rn(c1, tab[3]);
            uint32_t ln = 0, lsum = 0, lsq = 0;
            for (int k = tid; k < s * s; k += UNC_THREADS) {
                const int i = k / s, j = k - i * s;
                const uint32_t v = template_pixel(a.img1, a.rows1, a.cols1, a.pitch1, off0, off1, cs, sn, i, j, a.rot_order);
                S.tpl[k] = (uint8_t)v;
                ln += v != 0u; lsum += v; lsq += v * v;
            }
            ln = __reduce_add_sync(0xffffffffu, ln);
            lsum = __reduce_add_sync(0xffffffffu, lsum);
            lsq = __reduce_add_sync(0xffffffffu, lsq);
            if (lane == 0) { atomicAdd(&S.stats[0], ln); atomicAdd(&S.stats[1], lsum); atomicAdd(&S.stats[2], lsq); }
        }
        // 2. peak candidates: the integers within 0.5 + 1e-6 of the table's position in map coordinates
        const double ec = __dadd_rn(__dsub_rn(row[0], c2fg), (double)(W - s) / 2.0);
        const double er = __dadd_rn(__dsub_rn(row[1], r2fg), (double)(H - s) / 2.0);
        const int j_lo = max(0, (int)ceil(__dsub_rn(ec, 0.5 + 1e-6))), j_hi = min(RW - 1, (int)floor(__dadd_rn(ec, 0.5 + 1e-6)));
        const int i_lo = max(0, (int)ceil(__dsub_rn(er, 0.5 + 1e-6))), i_hi = min(RH - 1, (int)floor(__dadd_rn(er, 0.5 + 1e-6)));
        int py[UNC_NPOS] = {0, 0, 0, 0, 0}, px[UNC_NPOS] = {0, 0, 0, 0, 0}, np = 0;
        for (int i = i_lo; i <= i_hi && i <= i_lo + 1; ++i)
            for (int j = j_lo; j <= j_hi && j <= j_lo + 1; ++j) { py[np] = i; px[np] = j; ++np; }
        if (!(isfinite(ec) && isfinite(er)) || np == 0) {
            if (tid == 0) { unc[3 * pt] = qnan; unc[3 * pt + 1] = qnan; unc[3 * pt + 2] = qnan; }
            continue;
        }
        __syncthreads();                                        // template and statistics complete
        const long long n = masked ? (long long)S.stats[0] : (long long)s * s;
        const long long st = S.stats[1], stt = S.stats[2];
        const TemplStats ts = templ_stats(S.stats[1], S.stats[2], a.inv_area, a.sqrt_inv_area);
        const double sqrt_vt = __dsqrt_rn((double)(n * stt - st * st));
        unc_position_sums(S, s, masked, win, a.pitch2, py, px, np);
        __syncthreads();
        if (tid == 0) {                                         // candidates in flat order, strict '>': the first maximum
            float best = -INFINITY;
            int bp = 0;
            for (int p = 0; p < np; ++p) {
                const uint32_t sm[3] = {S.sums[p][0], S.sums[p][1], S.sums[p][2]};
                const float v = unc_map_value(sm, masked, ts, a.inv_area, n, st, sqrt_vt);
                if (v > best) { best = v; bp = p; }
            }
            S.bi = py[bp]; S.bj = px[bp];
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p) S.sums[p][0] = S.sums[p][1] = S.sums[p][2] = 0u;
        }
        __syncthreads();
        // 3. the five positions: P0, X-, X+, Y-, Y+ (an axis whose peak is on the map's edge is not refined: unused)
        const int bi = S.bi, bj = S.bj;
        const bool ux = bj > 0 && bj < RW - 1, uy = bi > 0 && bi < RH - 1;
        const int qy[UNC_NPOS] = {bi, bi, bi, bi - 1, bi + 1}, qx[UNC_NPOS] = {bj, bj - 1, bj + 1, bj, bj};
        const bool used[UNC_NPOS] = {true, ux, ux, uy, uy};
        // unused positions are evaluated at P0 (always inside the map) and ignored
        int ey[UNC_NPOS], ex[UNC_NPOS];
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) { ey[p] = used[p] ? qy[p] : bi; ex[p] = used[p] ? qx[p] : bj; }
        unc_position_sums(S, s, masked, win, a.pitch2, ey, ex, UNC_NPOS);
        __syncthreads();
        int swp[UNC_NPOS];
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) swp[p] = (int)S.sums[p][1];
        // 4. A, V, Vt and S over the template's pixels
        __int128 acc_s[UNC_NPAIR];
        long long acc_a[UNC_NPOS], acc_v[UNC_NPOS], acc_t = 0;
#pragma unroll
        for (int q = 0; q < UNC_NPAIR; ++q) acc_s[q] = 0;
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) { acc_a[p] = 0; acc_v[p] = 0; }
        const int n32 = (int)n, st32 = (int)st;
        for (int k = tid; k < s * s; k += UNC_THREADS) {
            const int i = k / s, j = k - i * s;
            const int tv = S.tpl[k];
            const bool m = !masked || tv != 0;
            const int t = m ? n32 * tv - st32 : 0;
            long long x[UNC_NPOS];
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p) {
                int w = 0;
                if (m && used[p]) w = n32 * (int)__ldg(win + (long long)(ey[p] + i) * a.pitch2 + (ex[p] + j)) - swp[p];
                x[p] = (long long)t * w;
                acc_a[p] += x[p];
                acc_v[p] += (long long)w * w;
            }
            acc_t += (long long)t * t;
            int q = 0;
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p)
#pragma unroll
                for (int r = p; r < UNC_NPOS; ++r) acc_s[q++] += (__int128)x[p] * x[r];
        }
        // block reduction: warp shuffles, then thread 0 over the warps
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int q = 0; q < UNC_NPAIR; ++q) acc_s[q] += shfl_down_i128(acc_s[q], o);
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p) {
                acc_a[p] += __shfl_down_sync(0xffffffffu, acc_a[p], o);
                acc_v[p] += __shfl_down_sync(0xffffffffu, acc_v[p], o);
            }
            acc_t += __shfl_down_sync(0xffffffffu, acc_t, o);
        }
        if (lane == 0) {
            unsigned long long *r = S.red[warp];
#pragma unroll
            for (int q = 0; q < UNC_NPAIR; ++q) {
                r[2 * q] = (unsigned long long)acc_s[q];
                r[2 * q + 1] = (unsigned long long)((unsigned __int128)acc_s[q] >> 64);
            }
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p) {
                r[2 * UNC_NPAIR + p] = (unsigned long long)acc_a[p];
                r[2 * UNC_NPAIR + UNC_NPOS + p] = (unsigned long long)acc_v[p];
            }
            r[2 * UNC_NPAIR + 2 * UNC_NPOS] = (unsigned long long)acc_t;
        }
        __syncthreads();
        if (tid != 0) continue;
        // 5. thread 0: K, the vertex gradients and the record
        for (int w = 1; w < UNC_WARPS; ++w) {
            const unsigned long long *r = S.red[w];
#pragma unroll
            for (int q = 0; q < UNC_NPAIR; ++q) acc_s[q] += (__int128)(((unsigned __int128)r[2 * q + 1] << 64) | r[2 * q]);
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p) {
                acc_a[p] += (long long)r[2 * UNC_NPAIR + p];
                acc_v[p] += (long long)r[2 * UNC_NPAIR + UNC_NPOS + p];
            }
            acc_t += (long long)r[2 * UNC_NPAIR + 2 * UNC_NPOS];
        }
        // K(P, Q) once per unordered pair, P the earlier in the order P0, X-, X+, Y-, Y+
        double K[UNC_NPOS][UNC_NPOS];
        const double dnvt = __dmul_rn(__ll2double_rn(n), __ll2double_rn(acc_t));
        double sq[UNC_NPOS];
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) sq[p] = __dsqrt_rn(__ll2double_rn(acc_v[p]));
        {
            int q = 0;
#pragma unroll
            for (int p = 0; p < UNC_NPOS; ++p)
#pragma unroll
                for (int r = p; r < UNC_NPOS; ++r, ++q) {
                    double k = qnan;
                    if (used[p] && used[r] && acc_v[p] != 0 && acc_v[r] != 0) {
                        const __int128 num = (__int128)n * acc_s[q] - (__int128)acc_a[p] * acc_a[r];
                        k = __ddiv_rn(i128_to_double_rn(num), __dmul_rn(__dmul_rn(dnvt, sq[p]), sq[r]));
                    }
                    K[p][r] = k; K[r][p] = k;
                }
        }
        float mv[UNC_NPOS];
#pragma unroll
        for (int p = 0; p < UNC_NPOS; ++p) {
            const uint32_t sm[3] = {S.sums[p][0], S.sums[p][1], S.sums[p][2]};
            mv[p] = unc_map_value(sm, masked, ts, a.inv_area, n, st, sqrt_vt);
        }
        double gx[3], gy[3];
        unc_vertex_grad(mv[1], mv[0], mv[2], gx);
        unc_vertex_grad(mv[3], mv[0], mv[4], gy);
        const int lx[3] = {1, 0, 2}, ly[3] = {3, 0, 4};
        const double var_c = ux ? unc_quad(K, lx, gx, lx, gx) : qnan;
        const double var_r = uy ? unc_quad(K, ly, gy, ly, gy) : qnan;
        const double cov_cr = ux && uy ? unc_quad(K, lx, gx, ly, gy) : qnan;
        unc[3 * pt] = var_c;
        unc[3 * pt + 1] = var_r;
        unc[3 * pt + 2] = cov_cr;
    }
}

}  // namespace sid
