// sid_pm_kernel.cuh -- the fused, batched pattern-matching kernel (and its light tail kernel).
//
// One persistent CTA per grid point (work-stealing over a list ordered largest-window-first, next work
// item prefetched) does everything the reference's use_mcc (pmlib.py:176-212) does for that point:
//
//   1. stage the search window of image 2 (pmlib.py:200-202) in shared memory: one TMA 2-D tile load
//      (cp.async.bulk.tensor + mbarrier; the box must start 16-byte aligned, consumers absorb the 0..15
//      byte offset), requested during the previous point's tail; fallback for boxes wider than 256 bytes:
//      warp-per-row aligned loads re-aligned with a funnel shift;
//   2. window sums / sums of squares for every displacement with two sliding-sum passes (exact
//      integers), folded into sqrt(max(sq - s^2/N, 0)) once per point;
//   3. for every angle (batches held in shared memory together): gather the rotated template from
//      image 1 (get_template, pmlib.py:89-115), zero-pixel check (pmlib.py:152-154), then the exact
//      integer correlation numerators
//        - IMMA path (default): mma.sync.m16n8k32 u8 x u8 -> s32, A = raw window rows, B = Toeplitz band
//          of a template row built on the fly, one warp per 16 x 24 output tile and all resident angles;
//        - dp4a path: IDP.4A, one thread per output row / column class / TX outputs at stride 4;
//      OpenCV's TM_CCOEFF_NORMED normalisation in FP64 without FMA contraction; running argmax with
//      np.argmax tie rules; best angle with the reference's strict '>' rule (pmlib.py:158-165);
//   4. Hessian at the peak, median (radix select) / std normalisation, optional mcc_norm
//      (pmlib.py:167-172) and the displacement bookkeeping (pmlib.py:168-169, 209-210) -- inside this
//      kernel, or, for small result maps, in pm_tail_kernel at much higher occupancy (split tail).
//
// Result-sized arrays (window statistics, NCC maps) live in shared memory when window + templates +
// scratch fit in a third of an SM, else in a per-CTA global slab that stays L2-resident; either way only
// O(R^2) traffic per angle goes there, against O(R^2 s^2) integer MACs out of shared memory / registers.
#pragma once
#include <cuda.h>
#include "sid_common.cuh"

namespace sid {

constexpr int PM_THREADS = 256;
constexpr int PM_MAX_AB = 4;      // angles whose templates sit in shared memory together (dp4a path; IMMA: PM_IMMA_AB)
constexpr int PM_SEG = 16;        // outputs per horizontal sliding-sum work item
constexpr int PM_VSEG = 8;        // outputs per vertical sliding-sum work item
constexpr int PM_WIN_SLACK = 64;  // words readable past the staged window

// Hand-off from the fused kernel to pm_tail_kernel (one record per work item of the launch).
struct PmTailRec {
    int pt;            // point index, or -1 when the fused kernel already wrote the (NaN) row
    int RH, RW;        // result map shape
    int H, W;          // window shape (for the displacement bookkeeping)
    int best_idx;      // flat index of the peak
    int best_a;        // index of the winning angle
    float best_r;      // peak value
    int mode;          // 0: the work item's hand-off region holds the float map; 1 (pm_ws_kernel): the exact integers it is made
                       //    of -- numerators of the winning angle | window sums | window sums of squares (tail_stride words each)
    uint32_t tsum, tsq;   // mode 1: template sum / sum of squares of the winning angle
};
// words per work item of the hand-off region
__host__ __device__ inline size_t tail_item_words(int tail_stride, int mode) { return (size_t)tail_stride * (mode ? 3 : 1); }

struct PmArgs {
    const uint8_t *img1; int rows1, cols1; long long pitch1;
    const uint8_t *img2; int rows2, cols2; long long pitch2;
    long long n;
    const double *c1, *r1, *c2fg, *r2fg, *border;
    const int *order;             // optional processing order (largest windows first)
    int s;                        // img_size
    int n_angles;
    const double *angles;         // device, n_angles
    const double *tab;            // device, n_angles x 4
    int rot_order;
    unsigned flags;
    double inv_area, sqrt_inv_area;
    double gw[5];                 // gaussian_filter(sigma=1) weights, centre..edge
    double *out;                  // n x 5
    int *status;                  // optional
    unsigned char *scratch;
    unsigned long long scratch_per_cta;
    int max_rr;                   // capacity of one result map (elements)
    int max_hrw;                  // capacity of the horizontal-sum arrays
    int win_words;                // capacity of the staged window (32-bit words, incl. slack)
    int tpw;                      // template row pitch in words (multiple of 4)
    int ab;                       // angles per batch
    int tpl_off;                  // byte offset of template column 0 inside a template row (IMMA path: 8)
    int nc;                       // IMMA path: 32-byte K chunks per template row = ceil((s + 7) / 32)
    int tma;                      // 1: stage the window with a TMA 2-D tile load (box = tma_wpw*4 x tma_rows bytes)
    int tma_wpw, tma_rows;
    unsigned int *counter;        // work-stealing cursor
    // split tail (small result maps): the fused kernel stores the winning map + a record per work item and
    // pm_tail_kernel computes the peak statistics at much higher occupancy
    int split_tail;
    float *tail_maps;             // n x tail_stride
    int tail_stride;              // floats per handed-over map: max_rr rounded up to 4 (16-byte rows for the tail's vector loads)
    PmTailRec *tail_recs;         // n
    // sid_run_maps only (null otherwise): the winning angle's raw NCC map of point pt goes to maps_out + map_off[pt],
    // its template (s x s) to tpl_out + pt * s * s when tpl_out is set
    float *maps_out;
    const long long *map_off;
    uint8_t *tpl_out;
    // SID_PEAKS only (null otherwise): the secondary peaks of point pt go to peaks + 12 * pt (store_secondary_peaks)
    double *peaks;
};

__host__ __device__ inline int pm_window_pitch_words(int W, bool imma = false) {
    if (imma) {
        int w = (W + 4 + 3) / 4;
        while ((w & 15) != 8) ++w;             // pitch == 8 (mod 16) words
        return w;
    }
    int n16 = (W + 4 + 15) / 16;          // 16-byte units, with room for the shifted tail
    if ((n16 & 1) == 0) ++n16;            // odd multiple of 16 B -> 8 consecutive rows hit 8 distinct bank groups
    return n16 * 4;
}
constexpr int PM_IMMA_THREADS = 192;      // 6 warps: 3 CTAs/SM at <= 112 registers
constexpr int PM_IMMA_AB = 3;             // angles per batch on the tensor-core path (36 accumulators per thread)
constexpr int PM_IMMA_ROW_SLACK = 16;     // window rows readable past H (padded 16-row output blocks)

// ---- correlation numerators for one thread tile -----------------------------------
// acc[tx] += sum_i sum_jj dp4a(window word (row y+i, word q0+tx+jj, byte shift p), template word (i, jj))
template <int TX, int NW>
__device__ __forceinline__ void mac_rows(const uint32_t *__restrict__ wrow, int wpw,
                                         const uint32_t *__restrict__ trow, int tpw,
                                         int s, int sh, unsigned (&acc)[TX]) {
    for (int i = 0; i < s; ++i) {
        uint32_t w[TX + NW];
#pragma unroll
        for (int k = 0; k < TX + NW; ++k) w[k] = wrow[k];
#pragma unroll
        for (int k = 0; k < TX + NW - 1; ++k) w[k] = __funnelshift_r(w[k], w[k + 1], sh);
        uint32_t t[(NW + 3) / 4 * 4];
#pragma unroll
        for (int k = 0; k < (NW + 3) / 4; ++k) {
            const uint4 v = *reinterpret_cast<const uint4 *>(trow + 4 * k);
            t[4 * k] = v.x; t[4 * k + 1] = v.y; t[4 * k + 2] = v.z; t[4 * k + 3] = v.w;
        }
#pragma unroll
        for (int jj = 0; jj < NW; ++jj)
#pragma unroll
            for (int tx = 0; tx < TX; ++tx) acc[tx] = __dp4a(w[tx + jj], t[jj], acc[tx]);
        wrow += wpw;
        trow += tpw;
    }
}

// any template width: 16 template bytes (4 words) at a time
template <int TX>
__device__ __forceinline__ void mac_rows_any(const uint32_t *__restrict__ wrow, int wpw,
                                             const uint32_t *__restrict__ trow, int tpw,
                                             int s, int nchunk, int sh, unsigned (&acc)[TX]) {
    for (int i = 0; i < s; ++i) {
        for (int c = 0; c < nchunk; ++c) {
            uint32_t w[TX + 4];
#pragma unroll
            for (int k = 0; k < TX + 4; ++k) w[k] = wrow[4 * c + k];
#pragma unroll
            for (int k = 0; k < TX + 3; ++k) w[k] = __funnelshift_r(w[k], w[k + 1], sh);
            const uint4 v = *reinterpret_cast<const uint4 *>(trow + 4 * c);
            const uint32_t t[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                for (int tx = 0; tx < TX; ++tx) acc[tx] = __dp4a(w[tx + jj], t[jj], acc[tx]);
        }
        wrow += wpw;
        trow += tpw;
    }
}

struct PmShared {
    BlockScratch bs;
    TemplStats st[PM_MAX_AB];
    unsigned long long key[PM_MAX_AB];
    uint32_t tsum[PM_MAX_AB], tsq[PM_MAX_AB];
    int slot[PM_MAX_AB];
    int haszero;
    unsigned int point, next;
    unsigned int tma_for;         // work item whose window was requested during the previous point's tail (else ~0)
    int nok, nx0, ny0;            // next point: window valid for prefetch, TMA box origin
    float best_r;
    int best_a, best_idx, best_slot;
};

// All tiles of one angle batch.  NW > 0: compile-time template width in words.
template <int TX, int NW>
__device__ __forceinline__ void pm_tiles(const uint32_t *__restrict__ win32, int wpw,
                                         const uint32_t *__restrict__ tpl32, int tpw, int s,
                                         int nb, int RH, int RW, int ab,
                                         const uint32_t *__restrict__ wsum, const double *__restrict__ wden,
                                         float *__restrict__ maps, int max_rr, PmShared &S) {
    // `ab` (0..3): byte offset of window column 0 inside win32's first word (TMA staging starts 16-byte
    // aligned); tiles are laid out over shifted columns x' = x + ab and mapped back on output
    const int tid = threadIdx.x, lane = tid & 31, nt = blockDim.x;
    const int nwc = (RW + ab + 3) >> 2;
    const int ncg = (nwc + TX - 1) / TX;
    const int ntiles = nb * ncg * RH * 4;
    const int nchunk = (s + 15) / 16;
    for (int base = 0; base < ntiles; base += nt) {
        const int t = base + tid;
        int my_ai = -1;
        unsigned long long key = 0ull;
        if (t < ntiles) {
            const int p = t & 3;
            int u = t >> 2;
            const int y = u % RH; u /= RH;
            const int cg = u % ncg;
            const int ai = u / ncg;
            const int q0 = cg * TX;
            unsigned acc[TX];
#pragma unroll
            for (int k = 0; k < TX; ++k) acc[k] = 0u;
            const uint32_t *wrow = win32 + y * wpw + q0;
            const uint32_t *trow = tpl32 + ai * s * tpw;
            if (NW > 0) mac_rows<TX, (NW > 0 ? NW : 1)>(wrow, wpw, trow, tpw, s, 8 * p, acc);
            else mac_rows_any<TX>(wrow, wpw, trow, tpw, s, nchunk, 8 * p, acc);
            const TemplStats st = S.st[ai];
            float *map = maps + (size_t)S.slot[ai] * max_rr;
            my_ai = ai;
#pragma unroll
            for (int tx = 0; tx < TX; ++tx) {
                const int x = 4 * (q0 + tx) + p - ab;
                if (x >= 0 && x < RW) {
                    const int idx = y * RW + x;
                    const float v = ncc_value((long long)acc[tx], wsum[idx], wden[idx], st);
                    map[idx] = v;
                    const unsigned long long k2 = peak_key(v, (uint32_t)idx);
                    key = k2 > key ? k2 : key;
                }
            }
        }
        // per-angle running argmax: warp-aggregate, then one shared atomic per warp and angle
        for (int a2 = 0; a2 < nb; ++a2) {
            unsigned long long k2 = (my_ai == a2) ? key : 0ull;
            k2 = warp_max_u64(k2);
            if (lane == 0 && k2) atomicMax(&S.key[a2], k2);
        }
    }
}

template <int NW>
__device__ __forceinline__ void pm_tiles_dispatch(int tx, const uint32_t *win32, int wpw, const uint32_t *tpl32, int tpw,
                                                  int s, int nb, int RH, int RW, int ab, const uint32_t *wsum,
                                                  const double *wden, float *maps, int max_rr, PmShared &S) {
    switch (tx) {
        case 8: pm_tiles<8, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
        case 9: pm_tiles<9, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
        case 10: pm_tiles<10, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
        case 11: pm_tiles<11, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
        case 12: pm_tiles<12, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
        default: pm_tiles<13, NW>(win32, wpw, tpl32, tpw, s, nb, RH, RW, ab, wsum, wden, maps, max_rr, S); break;
    }
}

// ---- tensor-core path: exact u8 x u8 -> s32 correlation with mma.sync.m16n8k32 (IMMA.16832) ----------
// For one template row i:  C[y][x] += sum_k A[y][k] * B[k][x]  with
//   A = 16 window rows (y0+i .. y0+i+15) x 32 window columns, straight from the staged window (no im2col);
//   B = Toeplitz band of template row i:  B[k][x] = T[i][col(k) - x], zero outside [0, s).
// The K slots are permuted so that a thread's two A words of a row are adjacent in memory (one LDS.64) and
// its two B words are 8 consecutive bytes of the zero-padded template row at byte (32c + 8*tig - g): three
// aligned words and two funnel shifts.  A warp owns a 16 x 24 output tile for all NBA resident angles, so
// every window fragment feeds NBA MMAs.
__device__ __forceinline__ void mma_u8_16832(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                             uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <int NBA, int NC>   // NC > 0: compile-time number of 32-byte K chunks (2 covers img_size <= 57)
__device__ __forceinline__ void pm_tiles_imma(const uint32_t *__restrict__ win32, int wpw,
                                              const uint32_t *__restrict__ tpl32, int tpw, int s, int nc_rt,
                                              int RH, int RW, int ab,
                                              const uint32_t *__restrict__ wsum, const double *__restrict__ wden,
                                              float *__restrict__ maps, int max_rr, PmShared &S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int nxg = (RW + ab + 23) / 24;               // tiles over shifted columns x' = x + ab (see pm_tiles)
    const int ntiles = ((RH + 15) >> 4) * nxg;
    const int ob = 8 + 8 * tig - g;               // byte offset of this lane's B bytes inside a padded template row
    constexpr int A_LANE = 2, A_HI = 1, B_HI = 1;
    const int bw = ob >> 2, bsh = (ob & 3) * 8;
    unsigned long long key[NBA];
#pragma unroll
    for (int a = 0; a < NBA; ++a) key[a] = 0ull;
    for (int t = warp; t < ntiles; t += nwarps) {
        const int yb = t / nxg, xg = t - yb * nxg;
        const int y0 = yb * 16, x0 = xg * 24;
        int acc[NBA][3][4];
#pragma unroll
        for (int a = 0; a < NBA; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[a][b][e] = 0;
        const uint32_t *arow = win32 + (y0 + g) * wpw + (x0 >> 2) + A_LANE * tig;
        const uint32_t *trow = tpl32 + bw;
        const uint32_t *arow8 = arow + 8 * wpw;
        const int nc = NC > 0 ? NC : nc_rt;
        const int tstride = s * tpw;
        for (int i = 0; i < s; ++i) {
#pragma unroll
            for (int c = 0; c < nc; ++c) {
                // the four fragment words are loaded as scalars so that each lands directly in its
                // operand register (a0..a3 must be consecutive; paired 64-bit loads would need moves)
                uint32_t af[3][4];
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    af[b][0] = arow[8 * c + 2 * b];
                    af[b][1] = arow8[8 * c + 2 * b];
                    af[b][2] = arow[8 * c + 2 * b + A_HI];
                    af[b][3] = arow8[8 * c + 2 * b + A_HI];
                }
#pragma unroll
                for (int a = 0; a < NBA; ++a) {
                    const uint32_t *tr = trow + a * tstride + 8 * c;
                    const uint32_t w0 = tr[0], w1 = tr[1], w2 = tr[B_HI], w3 = tr[B_HI + 1];   // B_HI == 1: w2 is w1 again (one load)
                    const uint32_t b0 = __funnelshift_r(w0, w1, bsh), b1 = __funnelshift_r(w2, w3, bsh);
#pragma unroll
                    for (int b = 0; b < 3; ++b) mma_u8_16832(acc[a][b], af[b][0], af[b][1], af[b][2], af[b][3], b0, b1);
                }
            }
            arow += wpw;
            arow8 += wpw;
            trow += tpw;
        }
        // ---- epilogue, two steps.  (1) The raw correlation sums go to their map slots as integers: C fragment =
        //      rows g / g+8, columns 2*tig, 2*tig+1 of each 8-column block.
#pragma unroll
        for (int b = 0; b < 3; ++b)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int y = y0 + g + 8 * h, x = x0 + 8 * b + 2 * tig + e - ab;
                    if (y < RH && x >= 0 && x < RW) {
                        const int idx = y * RW + x;
#pragma unroll
                        for (int a = 0; a < NBA; ++a) maps[(size_t)S.slot[a] * max_rr + idx] = __int_as_float(acc[a][b][2 * h + e]);
                    }
                }
        __syncwarp();
        //      (2) One rolled loop normalises the warp's 16 x 24 tile in place, lanes along x (conflict-free, and the
        //      accumulators are dead, so the template statistics fit in registers): OpenCV's FP64 formula, then the
        //      running maximum per lane -- positions are visited in increasing flat index, so a strict '>' keeps
        //      the first maximum like np.argmax.
        {
            double mean[NBA], norm[NBA];
            int soff[NBA], flat[NBA];
            float bv[NBA];
            int bi[NBA];
#pragma unroll
            for (int a = 0; a < NBA; ++a) {
                mean[a] = S.st[a].mean; norm[a] = S.st[a].norm; flat[a] = S.st[a].flat;
                soff[a] = S.slot[a] * max_rr;
                bv[a] = -INFINITY; bi[a] = -1;
            }
#pragma unroll 1
            for (int p = lane; p < 16 * 24; p += 32) {
                const int ty = p / 24, tx = p - ty * 24;
                const int y = y0 + ty, x = x0 + tx - ab;
                if (y < RH && x >= 0 && x < RW) {
                    const int idx = y * RW + x;
                    const double ws = (double)wsum[idx];
                    const double wd = wden[idx];
#pragma unroll
                    for (int a = 0; a < NBA; ++a) {
                        const int c = __float_as_int(maps[soff[a] + idx]);
                        const double num = __dsub_rn((double)c, __dmul_rn(ws, mean[a]));
                        const float v = flat[a] ? 1.0f : __double2float_rn(ncc_finish(num, __dmul_rn(wd, norm[a])));
                        maps[soff[a] + idx] = v;
                        if (v > bv[a]) { bv[a] = v; bi[a] = idx; }
                    }
                }
            }
#pragma unroll
            for (int a = 0; a < NBA; ++a)
                if (bi[a] >= 0) {
                    const unsigned long long k2 = peak_key(bv[a], (uint32_t)bi[a]);
                    key[a] = k2 > key[a] ? k2 : key[a];
                }
        }
    }
#pragma unroll
    for (int a = 0; a < NBA; ++a) {
        const unsigned long long k2 = warp_max_u64(key[a]);
        if (lane == 0 && k2) atomicMax(&S.key[a], k2);
    }
}

// outputs per thread: the TX in [8,13] that wastes the fewest padded columns
__host__ __device__ inline int pm_pick_tx(int RW) {
    const int nwc = (RW + 3) >> 2;
    int best = 8, best_cost = 1 << 30;
    for (int tx = 8; tx <= 13; ++tx) {
        const int cost = (nwc + tx - 1) / tx * tx;
        if (cost <= best_cost) { best_cost = cost; best = tx; }
    }
    return best;
}

// Search window of one point: img2[int(r2-hws-b):int(r2+hws+b+1), int(c2-hws-b):int(c2+hws+b+1)] with NumPy's
// clipping of the far end (reference pmlib.py:200-202).  Returns false for windows the reference cannot process.
// The one definition of the rule, for the kernels (G = PmArgs) and for sid_map_layout on the host (G = WindowGeom).
struct WindowGeom { int s, rows2, cols2; };
template <class G>
__host__ __device__ __forceinline__ bool window_rect(const G &a, double c1, double r1, double c2, double r2, double brd,
                                                     long long &x0, long long &y0, int &W, int &H) {
    const int s = a.s, hws = s / 2;
    bool ok = isfinite(c1) && isfinite(r1) && isfinite(c2) && isfinite(r2) && isfinite(brd) &&
              fabs(c2) < 1e9 && fabs(r2) < 1e9 && fabs(brd) < 1e9;
    x0 = y0 = 0; W = H = 0;
    if (!ok) return false;
    long long y1, x1;
    y0 = (long long)(r2 - (double)hws - brd);
    y1 = (long long)(r2 + (double)hws + brd + 1.0);
    x0 = (long long)(c2 - (double)hws - brd);
    x1 = (long long)(c2 + (double)hws + brd + 1.0);
    if (y1 > a.rows2) y1 = a.rows2;      // numpy slicing clips the far end
    if (x1 > a.cols2) x1 = a.cols2;
    ok = y0 >= 0 && x0 >= 0 && (y1 - y0) >= s + 1 && (x1 - x0) >= s + 1;
    H = (int)(y1 - y0); W = (int)(x1 - x0);
    return ok;
}
__device__ __forceinline__ bool pm_window_rect(const PmArgs &a, double c1, double r1, double c2, double r2, double brd,
                                               long long &x0, long long &y0, int &W, int &H) {
    return window_rect(a, c1, r1, c2, r2, brd, x0, y0, W, H);
}

// sid_run_maps: store the winning angle's raw NCC map (RR floats at `map`), read before peak_statistics may smooth or
// reuse it.  Called by every thread of the CTA; ends with a barrier, so the caller may overwrite `map` afterwards.
__device__ __forceinline__ void pm_store_map(const PmArgs &a, long long pt, const float *map, int RR) {
    float *dst = a.maps_out + a.map_off[pt];
    for (int k = threadIdx.x; k < RR; k += blockDim.x) dst[k] = map[k];
    __syncthreads();
}
// sid_run_maps: the winning angle's template, regathered with template_pixel so that it is bit-identical to
// templates_kernel.  The fused kernels call it at the very end of a point, where little else is live (inside their
// tail it would raise the register pressure of the whole loop).
__device__ __forceinline__ void pm_store_template(const PmArgs &a, long long pt, int best_a) {
    const int s = a.s;
    const double *tab = a.tab + 4 * best_a;
    const double cs = tab[0], sn = tab[1];
    const double off0 = __dsub_rn(a.r1[pt], tab[2]), off1 = __dsub_rn(a.c1[pt], tab[3]);
    uint8_t *dst = a.tpl_out + (size_t)pt * s * s;
    for (int k = threadIdx.x; k < s * s; k += blockDim.x) {
        const int i = k / s, j = k - i * s;
        dst[k] = template_pixel(a.img1, a.rows1, a.cols1, a.pitch1, off0, off1, cs, sn, i, j, a.rot_order);
    }
}

// Scratch footprint of one CTA (bytes): wden f64[rr] | wsum u32[rr] | region, where the region
// holds the NCC maps and, before any map exists, the horizontal sums hs/hq u32[hrw] each.
__host__ __device__ inline size_t pm_scratch_bytes(int max_rr, int max_hrw, int ab, bool smth, bool split_tail = false) {
    // maps: ab + 1 angle slots (one always keeps the best so far), the Hessian map, and a second
    // smoothing temporary only when hes_smth is requested; none of the latter two with a split tail
    size_t maps = (size_t)(ab + 1 + (split_tail ? 0 : 1 + (smth ? 1 : 0))) * max_rr * 4, hsq = (size_t)max_hrw * 8;
    size_t b = (size_t)max_rr * 12 + (maps > hsq ? maps : hsq);
    return (b + 255) & ~(size_t)255;
}

// SMEM_SCRATCH: the per-point scratch sits in shared memory behind the templates (small search
// windows: no L2 round trips in the statistics / epilogue / Hessian / median phases); otherwise
// in this CTA's global slab (any window size).  PEAKS: SID_PEAKS (store_secondary_peaks after the row), a separate
// instantiation so that the kernels without it keep their registers.
template <int NW, bool SMEM_SCRATCH, bool IMMA, bool PEAKS>
__global__ void __launch_bounds__(IMMA ? PM_IMMA_THREADS : PM_THREADS, 3)
pm_points_kernel(const PmArgs a, const __grid_constant__ CUtensorMap tmap2) {
    extern __shared__ __align__(128) unsigned char pm_smem[];
    __shared__ PmShared S;
    __shared__ __align__(8) unsigned long long win_bar;
    unsigned win_phase = 0;
    uint32_t *win32 = reinterpret_cast<uint32_t *>(pm_smem);
    uint32_t *tpl32 = win32 + a.win_words;
    const int tid = threadIdx.x, lane = tid & 31, nt = blockDim.x;   // nt <= PM_THREADS, chosen by the host
    const int s = a.s, tpw = a.tpw, ab = a.ab;

    unsigned char *slab;
    if constexpr (SMEM_SCRATCH) slab = reinterpret_cast<unsigned char *>(tpl32 + ab * s * tpw);
    else slab = a.scratch + (size_t)blockIdx.x * a.scratch_per_cta;
    double *wden = reinterpret_cast<double *>(slab);
    uint32_t *wsum = reinterpret_cast<uint32_t *>(wden + a.max_rr);
    float *maps = reinterpret_cast<float *>(wsum + a.max_rr);   // (ab + 3) maps of max_rr floats
    uint32_t *hs = reinterpret_cast<uint32_t *>(maps);          // aliases the maps: dead before the first map is written
    uint32_t *hq = hs + a.max_hrw;

    if (tid == 0) {
        S.next = atomicAdd(a.counter, 1u);
        S.tma_for = 0xffffffffu;
        if (a.tma) mbar_init(&win_bar, 1);
    }
    for (;;) {
        __syncthreads();
        if (tid == 0) {
            S.point = S.next;
            if ((long long)S.point < a.n) S.next = atomicAdd(a.counter, 1u);   // prefetch the next work item
        }
        __syncthreads();
        const long long pi = (long long)S.point;
        if (pi >= a.n) break;
        const bool prefetched = a.tma && S.tma_for == S.point;  // its window is already on the way (or here)
        if (a.tma && tid == nt - 1) {
            // the last thread looks one work item ahead so that thread 0 can prefetch its window during this
            // point's tail (these loads overlap the wait for this point's own window)
            int nok = 0;
            const long long pn = (long long)S.next;
            if (pn < a.n) {
                const long long q = a.order ? (long long)a.order[pn] : pn;
                long long nx0, ny0; int nW, nH;
                if (pm_window_rect(a, a.c1[q], a.r1[q], a.c2fg[q], a.r2fg[q], a.border[q], nx0, ny0, nW, nH)) {
                    nok = 1; S.nx0 = (int)(nx0 - (nx0 & 15)); S.ny0 = (int)ny0;
                }
            }
            S.nok = nok;
        }
        const long long pt = a.order ? (long long)a.order[pi] : pi;
        const double c1 = a.c1[pt], r1 = a.r1[pt], c2 = a.c2fg[pt], r2 = a.r2fg[pt], brd = a.border[pt];
        double *o = a.out + 5 * pt;

        // ---- window rectangle
        long long x0, y0;
        int W, H;
        bool ok = pm_window_rect(a, c1, r1, c2, r2, brd, x0, y0, W, H);
        const int RH = H - s + 1, RW = W - s + 1, RR = RH * RW;
        const int wpw = a.tma ? a.tma_wpw : pm_window_pitch_words(W, IMMA);
        const int xoff = a.tma ? (int)(x0 & 15) : 0;          // byte offset of window column 0 inside a staged row
        const int xab = xoff & 3;
        const uint32_t *winx = win32 + (xoff >> 2);
        if (ok) ok = RR <= a.max_rr && H * RW <= a.max_hrw &&
                     (H + (IMMA ? PM_IMMA_ROW_SLACK : 0)) * wpw + PM_WIN_SLACK <= a.win_words;
        if (prefetched) {                                       // always consume the phase of a requested window
            mbar_wait(&win_bar, win_phase);
            win_phase ^= 1u;
        }
        if (!ok) {
            if (tid == 0) {
                o[0] = o[1] = o[2] = o[3] = o[4] = nan("");
                if (a.status) a.status[pt] = -1;
                if (a.split_tail) a.tail_recs[pi].pt = -1;
            }
            continue;
        }

        // ---- 1. stage the window.  TMA: one 2-D tile load of the uint8 image (any byte offset, out-of-image
        //         bytes read as 0) signalled on an mbarrier.  Otherwise: one warp per row, each lane loads one
        //         aligned word and takes its right neighbour by shuffle, four rows in flight per warp.
        if (a.tma) {
            if (tid == 0) {
                if (!prefetched) {
                    mbar_expect_tx(&win_bar, (unsigned)(a.tma_wpw * 4 * a.tma_rows));
                    tma_load_2d(win32, &tmap2, (int)x0 - xoff, (int)y0, &win_bar);   // innermost start must be 16-byte aligned
                }
                S.best_r = -INFINITY; S.best_a = -1; S.best_idx = 0; S.best_slot = -1;
            }
            if (!prefetched) {
                mbar_wait(&win_bar, win_phase);
                win_phase ^= 1u;
            }
        } else {
            const int al8 = 8 * (int)(x0 & 3);
            const unsigned char *g = a.img2 + y0 * a.pitch2 + (x0 - (x0 & 3));
            const int warp = tid >> 5, nwarps = nt >> 5;
            for (int kb = 0; kb < wpw; kb += 31) {                  // 31 output words per pass (lane 31 only feeds lane 30)
                const int k = kb + lane;
                const bool in_row = k <= wpw;                        // word wpw is read for the last shift only
                for (int y = warp; y < H; y += 4 * nwarps) {
                    uint32_t w[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int yy = y + u * nwarps;
                        w[u] = 0;
                        if (in_row && yy < H) w[u] = __ldg(reinterpret_cast<const uint32_t *>(g + (long long)yy * a.pitch2) + k);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int yy = y + u * nwarps;
                        const uint32_t nx = __shfl_down_sync(0xffffffffu, w[u], 1);
                        if (lane < 31 && k < wpw && yy < H) win32[yy * wpw + k] = __funnelshift_r(w[u], nx, al8);
                    }
                }
            }
            if (tid == 0) { S.best_r = -INFINITY; S.best_a = -1; S.best_idx = 0; S.best_slot = -1; }
        }
        __syncthreads();

        // ---- 2a. horizontal sliding sums over template width, every window row
        {
            const unsigned char *wb = reinterpret_cast<const unsigned char *>(win32);
            const int pitchb = wpw * 4;
            int seg = PM_SEG;                                         // one round: H * ceil(RW / seg) <= nt when possible
            while (H * ((RW + seg - 1) / seg) > nt && seg < RW) ++seg;
            const int nseg = (RW + seg - 1) / seg;
            for (int t = tid; t < H * nseg; t += nt) {
                const int y = t / nseg, xs = (t - y * nseg) * seg;
                const int xe = min(RW, xs + seg);
                const unsigned char *rowp = wb + y * pitchb + xoff;
                uint32_t sum = 0, sq = 0;
                for (int j = 0; j < s; ++j) { const uint32_t v = rowp[xs + j]; sum += v; sq += v * v; }
                for (int x = xs; x < xe; ++x) {
                    hs[y * RW + x] = sum; hq[y * RW + x] = sq;
                    const uint32_t va = rowp[x], vb = rowp[x + s];
                    sum += vb - va; sq += vb * vb - va * va;
                }
            }
        }
        __syncthreads();
        // ---- 2b. vertical sliding sums -> window sum and denominator per displacement
        {
            int vseg = PM_VSEG;                                       // one round: RW * ceil(RH / vseg) <= nt when possible
            while (RW * ((RH + vseg - 1) / vseg) > nt && vseg < RH) ++vseg;
            const int nseg = (RH + vseg - 1) / vseg;
            for (int t = tid; t < RW * nseg; t += nt) {
                const int sg = t / RW, x = t - sg * RW;
                const int ys = sg * vseg, ye = min(RH, ys + vseg);
                uint32_t sum = 0, sq = 0;
#pragma unroll 5
                for (int i = 0; i < s; ++i) { sum += hs[(ys + i) * RW + x]; sq += hq[(ys + i) * RW + x]; }
                for (int y = ys; y < ye; ++y) {
                    wsum[y * RW + x] = sum;
                    wden[y * RW + x] = window_den(sum, sq, a.inv_area);
                    if (y + 1 < ye) {
                        sum += hs[(y + s) * RW + x] - hs[y * RW + x];
                        sq += hq[(y + s) * RW + x] - hq[y * RW + x];
                    }
                }
            }
        }
        // (the barrier after the template gather below also orders these writes before their first use)

        // ---- 3. angle batches
        const int A = a.n_angles;
        const int nbatch = (A + ab - 1) / ab;
        const int per = (A + nbatch - 1) / nbatch;
        const int txsel = pm_pick_tx(RW + xab);
        bool has_zero = false;
        for (int a0 = 0; a0 < A; a0 += per) {
            const int nb = min(per, A - a0);
            for (int t = tid; t < nb * s * tpw; t += nt) tpl32[t] = 0u;
            if (tid < PM_MAX_AB) { S.tsum[tid] = 0; S.tsq[tid] = 0; S.key[tid] = 0ull; }
            if (tid == 0) S.haszero = 0;
            __syncthreads();
            // gather rotated templates (get_template): thread = (column j, row group); the j terms of the
            // coordinates are hoisted, and a corner test removes the per-pixel bounds checks
            {
                unsigned char *tb = reinterpret_cast<unsigned char *>(tpl32);
                const int rows_per_pass = nt / s;                    // >= 1 since s <= 128 <= nt
                const int gi = tid / s, gj = tid - gi * s;
                const bool active = gi < rows_per_pass;
                const double dj = (double)gj;
                for (int ai = 0; ai < nb; ++ai) {
                    const double *tab = a.tab + 4 * (a0 + ai);
                    const double cs = tab[0], sn = tab[1];
                    const double off0 = __dsub_rn(r1, tab[2]), off1 = __dsub_rn(c1, tab[3]);
                    const bool inside = template_inside_warp(a.rows1, a.cols1, off0, off1, cs, sn, s);
                    const bool fast0 = inside && a.rot_order == 0;      // common case: nearest neighbour, fully inside
                    const double jsn = __dmul_rn(dj, sn), jcs = __dmul_rn(dj, cs);
                    unsigned char *tdst = tb + (size_t)ai * s * tpw * 4 + a.tpl_off + gj;
                    uint32_t lsum = 0, lsq = 0; int lzero = 0;
                    // one specialised loop runs per template: nearest + inside (the common case), other inside, checked
                    auto sweep = [&](auto sample) {
                        for (int i0 = 0; i0 < s; i0 += 4 * rows_per_pass) {
                            uint32_t v[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int i = i0 + u * rows_per_pass + gi;
                                v[u] = 1u;
                                if (active && i < s) {
                                    const double di = (double)i;
                                    const double row = __dadd_rn(__dadd_rn(off0, __dmul_rn(di, cs)), jsn);
                                    const double col = __dadd_rn(__dadd_rn(off1, __dmul_rn(di, -sn)), jcs);
                                    v[u] = sample(row, col);
                                }
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int i = i0 + u * rows_per_pass + gi;
                                if (active && i < s) {
                                    tdst[i * tpw * 4] = (unsigned char)v[u];
                                    lsum += v[u]; lsq += v[u] * v[u]; lzero |= (v[u] == 0);
                                }
                            }
                        }
                    };
                    if (fast0) sweep([&](double row, double col) { return template_sample<false>(a.img1, a.rows1, a.cols1, a.pitch1, row, col, 0); });
                    else if (inside) sweep([&](double row, double col) { return template_sample<false>(a.img1, a.rows1, a.cols1, a.pitch1, row, col, 1); });
                    else sweep([&](double row, double col) { return template_sample<true>(a.img1, a.rows1, a.cols1, a.pitch1, row, col, a.rot_order); });
                    lsum = __reduce_add_sync(0xffffffffu, lsum);
                    lsq = __reduce_add_sync(0xffffffffu, lsq);
                    lzero = __any_sync(0xffffffffu, lzero);
                    if (lane == 0) {
                        atomicAdd(&S.tsum[ai], lsum); atomicAdd(&S.tsq[ai], lsq);
                        if (lzero) S.haszero = 1;
                    }
                }
            }
            __syncthreads();
            if (S.haszero) { has_zero = true; break; }
            // every thread derives the template statistics it needs; thread < nb publishes slot + stats
            if (tid < nb) {
                S.st[tid] = templ_stats(S.tsum[tid], S.tsq[tid], a.inv_area, a.sqrt_inv_area);
                int slot = tid;                 // tid-th slot that does not hold the best map so far
                if (S.best_slot >= 0 && slot >= S.best_slot) ++slot;
                S.slot[tid] = slot;
            }
            __syncthreads();
            if constexpr (IMMA) {
                if (a.nc == 2) {
                    if (nb == 1) pm_tiles_imma<1, 2>(winx, wpw, tpl32, tpw, s, 2, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                    else if (nb == 2) pm_tiles_imma<2, 2>(winx, wpw, tpl32, tpw, s, 2, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                    else pm_tiles_imma<3, 2>(winx, wpw, tpl32, tpw, s, 2, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                } else {
                    if (nb == 1) pm_tiles_imma<1, 0>(winx, wpw, tpl32, tpw, s, a.nc, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                    else if (nb == 2) pm_tiles_imma<2, 0>(winx, wpw, tpl32, tpw, s, a.nc, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                    else pm_tiles_imma<3, 0>(winx, wpw, tpl32, tpw, s, a.nc, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
                }
            } else {
                pm_tiles_dispatch<NW>(txsel, winx, wpw, tpl32, tpw, s, nb, RH, RW, xab, wsum, wden, maps, a.max_rr, S);
            }
            __syncthreads();
            if (tid == 0) {
                for (int ai = 0; ai < nb; ++ai) {           // angle order, strict '>'
                    const unsigned long long k = S.key[ai];
                    const float v = key_f32((uint32_t)(k >> 32));
                    if (v > S.best_r) {
                        S.best_r = v; S.best_a = a0 + ai;
                        S.best_idx = (int)(0xffffffffu - (uint32_t)(k & 0xffffffffull));
                        S.best_slot = S.slot[ai];
                    }
                }
            }
            __syncthreads();
        }
        if (has_zero || S.best_a < 0) {
            if (tid == 0) {
                o[0] = o[1] = o[2] = o[3] = o[4] = nan("");
                if (a.status) a.status[pt] = 0;
                if (a.split_tail) a.tail_recs[pi].pt = -1;
            }
            continue;
        }

        // ---- 4. peak statistics and bookkeeping.  The window buffer is dead from here on: request the next
        //         point's window now so that the load overlaps the whole tail.
        if (a.tma && tid == 0 && S.nok) {
            mbar_expect_tx(&win_bar, (unsigned)(a.tma_wpw * 4 * a.tma_rows));
            tma_load_2d(win32, &tmap2, S.nx0, S.ny0, &win_bar);
            S.tma_for = S.next;
        }
        const int best_slot = S.best_slot, best_idx = S.best_idx;
        const float *best = maps + (size_t)best_slot * a.max_rr;
        if (a.split_tail) {
            // hand the winning map to pm_tail_kernel and move on to the next point
            float *dst = a.tail_maps + (size_t)pi * a.tail_stride;
            for (int k = tid; k < RR; k += nt) dst[k] = best[k];
            if (tid == 0) {
                PmTailRec rec;
                rec.pt = (int)pt; rec.RH = RH; rec.RW = RW; rec.H = H; rec.W = W;
                rec.best_idx = best_idx; rec.best_a = S.best_a; rec.best_r = S.best_r;
                rec.mode = 0; rec.tsum = 0u; rec.tsq = 0u;
                a.tail_recs[pi] = rec;
            }
            continue;
        }
        if (a.maps_out) pm_store_map(a, pt, best, RR);
        float *tmp_a = maps + (size_t)(best_slot == 0 ? 1 : 0) * a.max_rr;
        float *hes = maps + (size_t)(ab + 1) * a.max_rr;
        float *tmp_b = maps + (size_t)(ab + 2) * a.max_rr;      // only allocated (and touched) with hes_smth
        uint32_t *wide_hist = nullptr;                      // 2048 bins on the window-statistics buffer (dead by now)
        if constexpr (SMEM_SCRATCH) { if ((size_t)a.max_rr * 8 >= 2048 * 4) wide_hist = reinterpret_cast<uint32_t *>(wden); }
        const PeakStats ps = peak_statistics(best, RH, RW, best_idx, S.best_r, a.flags, a.gw, tmp_a, tmp_b, hes, S.bs, wide_hist);
        if (tid == 0) {
            const int bi = best_idx / RW, bj = best_idx - bi * RW;
            const double dr = (double)bi - (double)(H - s) / 2.0;
            const double dc = (double)bj - (double)(W - s) / 2.0;
            o[0] = c2 + dc;
            o[1] = r2 + dr;
            if (a.flags & 8u) {         // SID_SUBPIXEL: peak_statistics leaves `best` intact
                const PeakOffsets d = peak_offsets(best, RH, RW, bi, bj);
                o[0] = __dadd_rn(o[0], d.dx);
                o[1] = __dadd_rn(o[1], d.dy);
            }
            o[2] = a.angles[S.best_a];
            o[3] = (double)ps.r;
            o[4] = (double)ps.h;
            if (a.status) a.status[pt] = 1;
        }
        if constexpr (PEAKS) store_secondary_peaks(a.peaks + 12 * pt, best, hes, RH, RW, best_idx, ps, a.flags, c2, r2, H, W, s, S.bs);
        if (a.tpl_out) pm_store_template(a, pt, S.best_a);
    }
}

// Peak statistics of one work item per CTA (reference pmlib.py:167-172, 209-210) on the map the fused kernel
// handed over.  Light on registers and shared memory, so ~10 CTAs are resident per SM.  PEAKS: SID_PEAKS, as in
// pm_points_kernel.
constexpr int PM_TAIL_THREADS = 128;            // small maps; 256 / 512 for larger ones (pm_tail_threads)
constexpr int PM_TAIL_MAX_THREADS = 512;
template <bool PEAKS>
__global__ void __launch_bounds__(PM_TAIL_MAX_THREADS) pm_tail_kernel(const PmArgs a) {
    extern __shared__ __align__(16) unsigned char tail_smem[];
    __shared__ BlockScratch bs;
    const PmTailRec rec = a.tail_recs[blockIdx.x];
    if (rec.pt < 0) return;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int RR = rec.RH * rec.RW;
    // wide_hist first: 16-byte aligned whatever max_rr is
    uint32_t *wide_hist = reinterpret_cast<uint32_t *>(tail_smem);
    float *map = reinterpret_cast<float *>(wide_hist + 2048);
    float *hes = map + a.tail_stride;
    float *tmp_a = hes + a.tail_stride;                                // only with hes_smth
    float *tmp_b = tmp_a + a.tail_stride;
    const float *item = a.tail_maps + (size_t)blockIdx.x * tail_item_words(a.tail_stride, rec.mode);
    // the producer wrote RR values per array; the up to 3 values behind them in the last vector are never used
    if (rec.mode == 0) {
        const float4 *src = reinterpret_cast<const float4 *>(item);
        for (int k = tid; k < (RR + 3) >> 2; k += nt) reinterpret_cast<float4 *>(map)[k] = src[k];
    } else {
        // the winning map from its exact integers, with the normalisation of every other path (pm_ws_kernel evaluated only
        // the positions that could hold the peak)
        const int4 *srcC = reinterpret_cast<const int4 *>(item);
        const uint4 *srcS = reinterpret_cast<const uint4 *>(item + a.tail_stride);
        const uint4 *srcQ = reinterpret_cast<const uint4 *>(item + 2 * a.tail_stride);
        const TemplStats st = templ_stats(rec.tsum, rec.tsq, a.inv_area, a.sqrt_inv_area);
        for (int k = tid; k < (RR + 3) >> 2; k += nt) {
            const int4 c = srcC[k];
            const uint4 ws = srcS[k], wq = srcQ[k];
            float4 v = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
            if (!st.flat) v = ncc_vec4(c, ws, wq, st, a.inv_area);
            reinterpret_cast<float4 *>(map)[k] = v;
        }
    }
    __syncthreads();
    if (a.maps_out) {
        pm_store_map(a, rec.pt, map, RR);
        if (a.tpl_out) pm_store_template(a, rec.pt, rec.best_a);
    }
    // hes_norm-only maps take peak_statistics' three-sweep fast path (sid_common.cuh) on the 2048-word histogram
    const PeakStats ps = peak_statistics(map, rec.RH, rec.RW, rec.best_idx, rec.best_r, a.flags, a.gw, tmp_a, tmp_b, hes, bs, wide_hist);
    if (tid == 0) {
        const int bi = rec.best_idx / rec.RW, bj = rec.best_idx - bi * rec.RW;
        const double dr = (double)bi - (double)(rec.H - a.s) / 2.0;
        const double dc = (double)bj - (double)(rec.W - a.s) / 2.0;
        double *o = a.out + 5 * (long long)rec.pt;
        double c2o = a.c2fg[rec.pt] + dc, r2o = a.r2fg[rec.pt] + dr;
        if (a.flags & 8u) {             // SID_SUBPIXEL: peak_statistics leaves `map` intact
            const PeakOffsets d = peak_offsets(map, rec.RH, rec.RW, bi, bj);
            c2o = __dadd_rn(c2o, d.dx);
            r2o = __dadd_rn(r2o, d.dy);
        }
        o[0] = c2o;
        o[1] = r2o;
        o[2] = a.angles[rec.best_a];
        o[3] = (double)ps.r;
        o[4] = (double)ps.h;
        if (a.status) a.status[rec.pt] = 1;
    }
    if constexpr (PEAKS)
        store_secondary_peaks(a.peaks + 12 * (long long)rec.pt, map, hes, rec.RH, rec.RW, rec.best_idx, ps, a.flags,
                              a.c2fg[rec.pt], a.r2fg[rec.pt], rec.H, rec.W, a.s, bs);
}
// CTA size of pm_tail_kernel by map size: a large map in shared memory leaves room for only two CTAs per SM, so each gets
// more warps (128 / 256 / 512 take peak_statistics' fast path)
inline int pm_tail_threads(int max_rr) {
    return max_rr <= 2560 ? 128 : (max_rr <= 6144 ? 256 : 512);
}
inline size_t pm_tail_smem_bytes(int max_rr, bool smth) { return (size_t)((max_rr + 3) & ~3) * 4 * (2 + (smth ? 2 : 0)) + 2048 * 4; }

}  // namespace sid
