// sid_pm_ws_kernel.cuh -- warp-specialised pattern-matching kernel (round 2, second tcgen05 formulation).
//
// Same per-point work and arithmetic contract as pm_tc_kernel / pm_points_kernel (reference pmlib.py:176-212 and
// everything it calls), organised as a pipeline of specialised warps over a stream of grid points, one persistent
// CTA per SM:
//
//   control (1 warp)   work stealing, window rectangle (pmlib.py:200-202), TMA of the window into a ring of 3 slots
//   gather  (4 warps)  get_template (pmlib.py:89-115): 4 pixels per thread -> compact rows; template sums / zero flag;
//                      then the Toeplitz EXPANSION of every pair of template rows into a ring of A-operand slots
//   mma     (4 warps)  one issuing thread each (one x block of 16 result columns each): tcgen05.mma kind::i8,
//                      A and B both from shared memory, accumulators in tensor memory (2 sets of 256 columns)
//   stats   (7 warps)  window sums / sums of squares (sliding, exact integers), also written to the tail hand-off
//   epilogue(2 x 4 warps, alternate points)  tcgen05.ld, combine the two row parities, FP32 screening of the angles
//                      from the exact integers, OpenCV's exact FP64 normalisation of the positions that can still hold
//                      the peak, argmax, hand-off of the winning angle's numerators to pm_tail_kernel (which rebuilds
//                      the float map from them)
//
// Formulation.  With x' = x + (x0 & 15) = 16 xq + dx (the window is staged from a 16-byte aligned column):
//
//   corr[a][y][x] = sum_i sum_j W[y+i][x'+j] T_a[i][j]
//   D_xq[(dx, a, ip)][n] += sum_k A_pr[(dx, a, ip)][k] * B_{pr,xq}[n][k]        pr = 0 .. ceil(s/2)-1  (row pairs)
//       A_pr[(dx, a, ip)][k] = T_a[2 pr + ip][k - dx]     (0 outside the row)   -- 16 byte shifts x 3 angles x 2 rows = 96
//       B_{pr,xq}[n][k]      = W[2 pr + n][16 xq + k]                           -- the staged window itself (16-byte
//                                                                                  column panels: no im2col, no copy)
//   corr[a][y][x] = D_xq[(dx,a,0)][y] + D_xq[(dx,a,1)][y+1]
//
// so the only operand that has to be GENERATED is 16 byte-shifted copies of each template row (per 4 template pixels:
// 2 loads, 3 byte permutes, 16 word stores), instead of one Toeplitz row per result column.  Per point and angle
// batch this is ~1.5 k warp instructions against ~16 k for the row loop of pm_tc_kernel.
//
// The exact FP64 normalisation (the most expensive per-output step) runs only where the peak can be: every position of
// every angle is first screened with an FP32 estimate whose error (< 1e-6, bound at WS_MARGIN) is far below the margin
// (4e-6); the positions whose estimate is within the margin of the best lower bound, and those the estimate cannot
// judge, are evaluated exactly, so the result is the same bit pattern the other kernels produce (strict '>' over angles,
// np.argmax inside a map).  The tail kernel rebuilds the whole winning map for the peak statistics.
#pragma once
#include "sid_pm_tc_kernel.cuh"

namespace sid {

constexpr int WS_THREADS = 896;           // 28 warps: control | 4 mma | 8 gather | 7 stats | 2 x 4 epilogue
constexpr int WS_W_MMA = 1, WS_W_GATHER = 5, WS_W_STATS = 13, WS_W_EPI = 20;
constexpr int WS_NST = 7 * 32;            // stats threads
constexpr int WS_NSTAT = 3;               // sets of window statistics (stats warps run up to 3 points ahead of the epilogue);
                                          // 2 where three do not fit the shared memory (PmWsCfg::nstat)
constexpr int WS_NG = 8;                  // gather warps
constexpr int WS_NWIN = 2;                // window ring (each slot: the search window of image 2 + the template patch of image 1)
constexpr int WS_NENT = 8;                // point entries / template records
constexpr int WS_MAX_SLOTS = 8;
constexpr int WS_ACC_COLS = 256;          // tensor-memory columns per accumulator set (4 x blocks x 64)
// Screening estimate of a non-special position (window variance v = N wsq - wsum^2 > N, template variance
// tv = N tsq - tsum^2 > 0, numerator n = N corr - wsum tsum; all exact in int64, N = s^2):
//     e = f32(n) * rsqrt.approx(f32(v)) * f32(1 / sqrt(tv))          (the real value is r = n / sqrt(v tv), |r| <= 1)
// Its relative error is at most 2^-24 (f32(n)) + 2^-25 (f32(v) under the root) + 2^-22 (rsqrt.approx, 2 ulp)
// + 2^-24 (the per-angle factor) + 2 * 2^-24 (two products) < 5.3e-7.  OpenCV's FP64 value differs from r by < 2e-7: v > N
// and tv >= N - 1 keep its denominator >= ~1 and window_den's argument >= 1, where the FP64 rounding of the numerator
// (< 4e-8 absolute) and of the denominator (< 6e-8 relative) stay tiny, plus 2^-25 for its float rounding.  So
// |e - exact| < ERR = 1e-6, and every position whose exact value can reach the peak has e >= (largest usable e) - 2 ERR.
// Positions with v <= N (window_den's 10 FLT_EPSILON threshold can apply: the exact value may be 0) or |e| >= WS_NEAR1
// (OpenCV's +-1 / 0 cases) are not estimated: they always go to the exact evaluation.
constexpr float WS_MARGIN = 4e-6f;        // >= 2 ERR
constexpr float WS_NEAR1 = 0.99f;
constexpr int WS_LIST = 256;              // positions evaluated exactly per epilogue group and batch (more: full exact pass)

// optional role profile (-DSID_WS_PROF): cycles per bucket, written to a.scratch as long long [cta][6 roles][8]
#ifdef SID_WS_PROF
#define WSP_DECL long long wsp[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long wsp_t = clock64();
#define WSP(k) { const long long now_ = clock64(); wsp[k] += now_ - wsp_t; wsp_t = now_; }
#define WSP_OUT(role) { long long *d_ = reinterpret_cast<long long *>(a.scratch) + ((size_t)blockIdx.x * 6 + (role)) * 8; \
                        for (int k_ = 0; k_ < 8; ++k_) d_[k_] = wsp[k_]; }
#else
#define WSP_DECL
#define WSP(k) {}
#define WSP_OUT(role) {}
#endif

struct PmWsCfg {
    int nab;          // angles per batch (<= 3)
    int ks;           // 32-byte K steps per A row
    int npairs;       // template row pairs = ceil(s / 2)
    int nwords;       // 32-bit words per compact template row = ceil(s / 4)
    int tw;           // compact row pitch (words) = nwords + 2 (a zero word either side)
    int nslots;       // A ring depth
    int nstat;        // sets of window statistics (3, or 2 for the largest maps)
    int lbo_a;        // bytes between K panels of an A slot
    int slot_bytes;
    int wrows;        // rows per window panel
    int npanels;      // panels per window slot
    int np_load;      // panels loaded per point
    int load_rows;    // TMA box height
    int win_bytes;    // one window slot
    int n16max;       // widest accumulator (<= 64)
    int hp;           // pitch of the transposed horizontal sums (odd)
    int cpl;          // words per angle plane of the combined correlation buffer
    int hs_words;     // words per transposed horizontal-sum array
    unsigned inv_nw1; // ceil(2^32 / (nwords + 1))
    int pbw, pbh;     // template patch of image 1 (TMA box, bytes x rows): every sample of every angle lies inside
    int prad;         // its half size: ceil(0.7072 s + 3)
    int patch_bytes;
    int off_a, off_tpl, tpl_buf_words, off_stat, stat_bytes, off_hs, off_c, off_emax, off_list, smem_bytes;
};

inline bool pm_ws_geometry(int s, int Rmax, int Wmax, int n_angles, int max_rr, PmWsCfg &g, int Rtyp = 0, int nstat = WS_NSTAT) {
    if (s < 2 || s > 112 || Rmax < 2) return false;
    if (Rmax + 1 > 64 || Rmax + 15 > 64 || Wmax > 256) return false;
    g.nab = n_angles < 3 ? n_angles : 3;
    g.npairs = (s + 1) / 2;
    g.nwords = (s + 3) / 4;
    g.tw = g.nwords + 2;
    g.ks = (g.nwords + 4 + 7) / 8;
    g.lbo_a = 2048 + 48;        // K panels 12 banks apart: the expansion's word stores of a warp spread over the banks (<= 2-way)
    g.slot_bytes = 2 * g.ks * g.lbo_a;
    g.nslots = WS_NG;          // >= the number of expanding warps: a warp's successive row pairs then reuse ONE slot, so it can never wait
                               // for a completion two phases ahead (a parity wait cannot tell phase k from phase k + 2)
    g.n16max = (Rmax + 1 + 15) & ~15;
    g.np_load = (Wmax + 15 + 15) / 16;
    g.npanels = 3 + 2 * g.ks;  // x block 3 reads panels 3 .. 2 + 2 ks
    if (g.npanels < g.np_load) g.npanels = g.np_load;
    g.load_rows = Wmax;
    g.wrows = (Wmax + 7) & ~7;
    g.prad = (int)(0.7072 * (double)s + 3.0) + 1;
    g.pbw = (2 * g.prad + 2 + 15 + 15) & ~15;        // the box starts at a 16-byte aligned column
    g.pbh = 2 * g.prad + 2;
    if (g.pbw > 256 || g.pbh > 256) return false;
    g.patch_bytes = (g.pbw * g.pbh + 127) & ~127;
    g.win_bytes = g.npanels * g.wrows * 16 + g.patch_bytes;
    g.hp = Wmax | 1;
    g.cpl = (max_rr + 31) & ~31;
    {   // Pad the angle planes of the combined correlation buffer so that the epilogue's stores -- per instruction 4 adjacent x
        // of 3 angles and 2 row parities (rows RW words apart) -- spread over the banks for the typical map width
        // (measured: planes a multiple of 32 words apart made every store 3-way conflicted, 8 % of all shared wavefronts)
        const int RW = Rtyp > 0 ? Rtyp : Rmax;
        int best_pad = 0, best_worst = 99, best_distinct = 0;
        for (int pad = 0; pad < 32; ++pad) {
            int cnt[32] = {0}, worst = 0, distinct = 0;
            for (int x = 0; x < 4; ++x) for (int aa = 0; aa < 3; ++aa) for (int ip = 0; ip < 2; ++ip) {
                const int b = ((x + pad * aa - RW * ip) % 32 + 32) % 32;
                if (++cnt[b] == 1) ++distinct;
                if (cnt[b] > worst) worst = cnt[b];
            }
            if (worst < best_worst || (worst == best_worst && distinct > best_distinct)) { best_worst = worst; best_distinct = distinct; best_pad = pad; }
        }
        g.cpl += best_pad;
    }
    g.inv_nw1 = (unsigned)((0x100000000ull + (unsigned)g.nwords) / (unsigned)(g.nwords + 1));
    g.tpl_buf_words = g.nab * s * g.tw;
    size_t off = (size_t)WS_NWIN * g.win_bytes;
    // the MMAs may read up to s + 64 rows of a panel: keep that inside the allocation behind the last window slot
    off = (off + 127) & ~(size_t)127;
    g.off_a = (int)off; off += (size_t)g.nslots * g.slot_bytes;
    off = (off + 127) & ~(size_t)127;
    g.off_tpl = (int)off; off += (size_t)2 * g.tpl_buf_words * 4;
    off = (off + 127) & ~(size_t)127;
    g.off_stat = (int)off;
    g.stat_bytes = (max_rr * 8 + 127) & ~127;            // wsq u32 | wsum u32
    g.nstat = nstat < 2 ? 2 : (nstat > WS_NSTAT ? WS_NSTAT : nstat);
    off += (size_t)g.nstat * g.stat_bytes;
    g.hs_words = Rmax * g.hp;
    g.off_hs = (int)off; off += (size_t)g.hs_words * 6;       // hq u32 | hs u16
    off = (off + 127) & ~(size_t)127;
    g.off_c = (int)off; off += (size_t)2 * g.nab * g.cpl * 4;
    g.off_emax = (int)off; off += (size_t)2 * max_rr * 4;     // per epilogue group: largest estimate over the angles per position
    g.off_list = (int)off; off += (size_t)2 * WS_LIST * 4;
    g.smem_bytes = (int)((off + 127) & ~(size_t)127);
    return true;
}

struct WsPoint { double c1, r1; long long pt, pi; int x0, y0, W, H; int done, px0, py0, pad; };
struct WsTplRec { long long pt, pi; int x0, W, H, zero; uint32_t tsum[3], tsq[3]; };
struct WsBars {
    unsigned long long win_full[WS_NWIN], win_empty[WS_NWIN];
    unsigned long long slot_full[WS_MAX_SLOTS], slot_empty[WS_MAX_SLOTS];
    unsigned long long acc_full[2], acc_empty[2];
    unsigned long long tpl_full[WS_NENT];
    unsigned long long stats_full[WS_NSTAT], stats_empty[WS_NSTAT];
};
struct WsEpi { TemplStats st[3]; float m[4]; unsigned long long key[4][3]; unsigned cnt; };

// try_wait spin with a watchdog: a protocol error becomes a trap (launch failure), never a hung GPU
#ifdef SID_WS_DEBUG
__device__ int g_ws_abort[1024], g_ws_msgs = 0;
__device__ unsigned g_ws_bar0 = 0;
__device__ int g_ws_prog[32];
#define WSD(code) { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) *(volatile int *)&g_ws_prog[threadIdx.x >> 5] = (code); }
#else
#define WSD(code) {}
#endif
// `ns`: back-off between polls (the hardware suspend of try_wait is only ~100 clk): long where the wait is long and not on the
// critical path, short where a role is about to continue
template <unsigned NS = 40u>
__device__ __forceinline__ void ws_wait(uint32_t bar, unsigned parity, int line = 0) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity), "r"(2000000u) : "memory");
    if (ok) return;
    const long long t0 = clock64();
    for (;;) {
        // up to 1024 polls in a 5-instruction loop, then one look at the watchdog clock
        asm volatile("{\n\t.reg .pred p, q;\n\t.reg .u32 n;\n\tmov.u32 n, 0;\n\t"
                     "WS_POLL_%=:\n\t"
                     "nanosleep.u32 %4;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
                     "@p bra WS_DONE_%=;\n\t"
                     "add.u32 n, n, 1;\n\t"
                     "setp.lt.u32 q, n, 1024;\n\t"
                     "@q bra WS_POLL_%=;\n\t"
                     "WS_DONE_%=:\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(2000000u), "r"(NS) : "memory");
        if (ok) return;
#ifdef SID_WS_DEBUG
        if (*(volatile int *)&g_ws_abort[blockIdx.x] || clock64() - t0 > 100000000LL) {
            if ((threadIdx.x & 31) == 0 && blockIdx.x == 0 && atomicAdd(&g_ws_msgs, 1) < 200)
                printf("[ws] block %d warp %d lane %d: wait timed out, barrier byte %d parity %u line %d\n", (int)blockIdx.x, (int)(threadIdx.x >> 5),
                       (int)(threadIdx.x & 31), (int)(bar - g_ws_bar0), parity, line);
            __nanosleep(1000000);
            g_ws_abort[blockIdx.x] = 1;
            return;
        }
#else
        // watchdog: a protocol error becomes a trap (launch failure), never a hung GPU
        if (clock64() - t0 > 8000000000LL) __trap();
#endif
    }
}
__device__ __forceinline__ void ws_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void ws_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// D[tmem] (+)= A[smem descriptor] * B[smem descriptor], u8 x u8 -> s32, M = 128
__device__ __forceinline__ void tc_mma_i8_ss(uint32_t d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}

// exact normalisation of one angle with a non-flat template (OpenCV's formula, bit for bit the other kernels' epilogue):
// this thread's part of the argmax key.  Only where the contender list overflows (flat or degenerate content).
__device__ __forceinline__ unsigned long long ws_exact_pass(const int32_t *__restrict__ Ca, const uint32_t *__restrict__ wsum,
                                                            const uint32_t *__restrict__ wsq, const TemplStats st, double inv_area,
                                                            int RR, int et) {
    float bv = -INFINITY;
    int bidx = -1;
    for (int base = 0; base < RR; base += 512) {
        int32_t cc[4];
        uint32_t s4[4], q4[4];
        float v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int idx = min(base + 128 * c + et, RR - 1);
            cc[c] = Ca[idx]; s4[c] = wsum[idx]; q4[c] = wsq[idx];
        }
        ncc_ints4(cc, s4, q4, st, inv_area, v);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int idx = base + 128 * c + et;
            if (idx < RR && v[c] > bv) { bv = v[c]; bidx = idx; }
        }
    }
    return bidx >= 0 ? peak_key(bv, (uint32_t)bidx) : 0ull;
}

// Screening sweep of one epilogue thread over the positions idx = et + 128 j of a batch of NB angles: stores per position the
// largest estimate over the angles, +inf where one of them cannot be estimated (flat window, |e| >= WS_NEAR1), and returns
// the largest estimate of the positions whose estimates are all usable (each is within ERR of an exact value).
template <int NB>
__device__ __forceinline__ float ws_screen(const int32_t *__restrict__ C, int cpl, const uint32_t *__restrict__ wsum,
                                           const uint32_t *__restrict__ wsq, float *__restrict__ emax, int RR, int et, unsigned N,
                                           const int (&tsm)[3], const float (&tinv)[3]) {
    float mx = -INFINITY;
#pragma unroll 2
    for (int idx = et; idx < RR; idx += 128) {
        const uint32_t ws = wsum[idx], wq = wsq[idx];
        const unsigned long long v = (unsigned long long)N * wq - (unsigned long long)ws * ws;     // >= 0 (Cauchy-Schwarz)
        float rv;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rv) : "f"((float)v));
        float hi = -INFINITY, lo = INFINITY;
#pragma unroll
        for (int k = 0; k < NB; ++k) {
            const long long n = (long long)(int)N * (long long)C[k * cpl + idx] - (long long)(int)ws * (long long)tsm[k];
            const float e = (float)n * rv * tinv[k];
            hi = fmaxf(hi, e); lo = fminf(lo, e);
        }
        const bool judged = v > (unsigned long long)N && hi < WS_NEAR1 && lo > -WS_NEAR1;
        emax[idx] = judged ? hi : INFINITY;
        mx = fmaxf(mx, judged ? hi : -INFINITY);
    }
    return mx;
}

__global__ void __launch_bounds__(WS_THREADS, 1)
pm_ws_kernel(const PmArgs a, const PmWsCfg g, const __grid_constant__ CUtensorMap tmapP, const __grid_constant__ CUtensorMap tmap1) {
    extern __shared__ __align__(128) unsigned char ws_smem[];
    __shared__ WsBars B;
    __shared__ WsPoint ent[WS_NENT];
    __shared__ WsTplRec trec[WS_NENT];
    __shared__ WsEpi epi[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ volatile int all_done_s;
    __shared__ volatile unsigned total_pts_s[2];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = a.s, nab = g.nab;
    const int PS = g.wrows * 16;
    const int A_ = a.n_angles;
    const int nbatch = (A_ + nab - 1) / nab;
    const int per = (A_ + nbatch - 1) / nbatch;
    uint8_t *sWin = ws_smem;
    uint8_t *sA = ws_smem + g.off_a;
    uint32_t *sTpl = reinterpret_cast<uint32_t *>(ws_smem + g.off_tpl);
    const uint32_t bar0 = smem_u32(&B);
#ifdef SID_WS_DEBUG
    if (threadIdx.x == 0 && blockIdx.x == 0) g_ws_bar0 = bar0;
#endif
    auto BAR = [&](const unsigned long long *p) -> uint32_t { return bar0 + (uint32_t)((const unsigned char *)p - (const unsigned char *)&B); };

    // ---- one-time setup: zero the A ring and the template buffers (their padding stays zero for good)
    for (int t = tid; t < (g.off_stat - g.off_a) / 4; t += WS_THREADS) reinterpret_cast<uint32_t *>(sA)[t] = 0u;
    if (tid < WS_NENT) { trec[tid].zero = 0; for (int k = 0; k < 3; ++k) { trec[tid].tsum[k] = 0u; trec[tid].tsq[k] = 0u; } }
    if (tid == 0) {
        for (int i = 0; i < WS_NWIN; ++i) { mbar_init(&B.win_full[i], 1); mbar_init(&B.win_empty[i], 4 + WS_NST / 32); }
        for (int i = 0; i < WS_MAX_SLOTS; ++i) { mbar_init(&B.slot_full[i], 1); mbar_init(&B.slot_empty[i], 4); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&B.acc_full[i], 4); mbar_init(&B.acc_empty[i], 4);
        }
        for (int i = 0; i < WS_NSTAT; ++i) { mbar_init(&B.stats_full[i], WS_NST / 32); mbar_init(&B.stats_empty[i], 4); }
        for (int i = 0; i < WS_NENT; ++i) mbar_init(&B.tpl_full[i], WS_NG);
        all_done_s = 0; total_pts_s[0] = 0u; total_pts_s[1] = 0u;
    }
    if (warp == 0) tc_alloc(&tmem_base_s, 512u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = tmem_base_s;

    if (warp == 0) {
        // ================================================================ control
        if (lane == 0) {
            const unsigned win_tx = (unsigned)(g.np_load * g.load_rows * 16 + g.pbw * g.pbh);
            const int patch_off = g.npanels * g.wrows * 16;
            unsigned P = 0;
            WSP_DECL
            unsigned pi = atomicAdd(a.counter, 1u);
            while ((long long)pi < a.n) {
                const long long pt = a.order ? (long long)a.order[pi] : (long long)pi;
                const double c1 = a.c1[pt], r1 = a.r1[pt], c2 = a.c2fg[pt], r2 = a.r2fg[pt], brd = a.border[pt];
                const unsigned pi_next = atomicAdd(a.counter, 1u);
                long long x0, y0; int W, H;
                bool ok = pm_window_rect(a, c1, r1, c2, r2, brd, x0, y0, W, H);
                if (ok) {
                    const int RH = H - s + 1, RW = W - s + 1, xoff = (int)(x0 & 15);
                    ok = RH * RW <= a.max_rr && H <= g.load_rows && W + xoff <= g.np_load * 16 && RH + 1 <= g.n16max &&
                         xoff + RW <= 64;
                }
                if (!ok) {
                    double *o = a.out + 5 * pt;
                    o[0] = o[1] = o[2] = o[3] = o[4] = nan("");
                    if (a.status) a.status[pt] = -1;
                    a.tail_recs[pi].pt = -1;
                } else {
                    const unsigned ws = P % WS_NWIN;
                    WSP(0)
                    if (P >= WS_NWIN) ws_wait<400u>(BAR(&B.win_empty[ws]), ((P / WS_NWIN) - 1u) & 1u, __LINE__);
                    WSP(1)
                    WsPoint &e = ent[P & (WS_NENT - 1)];
                    e.c1 = c1; e.r1 = r1; e.pt = pt; e.pi = (long long)pi;
                    e.x0 = (int)x0; e.y0 = (int)y0; e.W = W; e.H = H; e.done = 0;
                    const int pxa = ((int)floor(c1) - g.prad) & ~15, py = (int)floor(r1) - g.prad;
                    e.px0 = pxa; e.py0 = py;
                    mbar_expect_tx(&B.win_full[ws], win_tx);
                    const int xa = (int)x0 - (int)(x0 & 15);
                    for (int p = 0; p < g.np_load; ++p)
                        tma_load_2d(sWin + (size_t)ws * g.win_bytes + (size_t)p * PS, &tmapP, xa + 16 * p, (int)y0, &B.win_full[ws]);
                    // template patch of image 1 around (c1, r1); out-of-image bytes read 0 (the gather only uses it for points
                    // whose samples all lie inside the image)
                    tma_load_2d(sWin + (size_t)ws * g.win_bytes + patch_off, &tmap1, pxa, py, &B.win_full[ws]);
                    ++P;
                }
                pi = pi_next;
            }
            const unsigned ws = P % WS_NWIN;
            if (P >= WS_NWIN) ws_wait<400u>(BAR(&B.win_empty[ws]), ((P / WS_NWIN) - 1u) & 1u, __LINE__);
            ent[P & (WS_NENT - 1)].done = 1;
            ws_arrive(BAR(&B.win_full[ws]));
            WSP(0)
            WSP_OUT(0)
        }
    } else if (warp < WS_W_GATHER) {
        // ================================================================ mma issuers (x block w each)
        if (lane == 0) {
            const int w = warp - WS_W_MMA;
            unsigned P = 0, round = 0, use0 = 0, use1 = 0;
            int slot = 0;
            const uint64_t adesc0 = tc_smem_desc(smem_u32(sA), (uint32_t)g.lbo_a, 128u);
            uint64_t ad = adesc0;
            WSP_DECL
            for (;;) {
                const unsigned ws = P % WS_NWIN;
                WSP(0)
                ws_wait<100u>(BAR(&B.win_full[ws]), (P / WS_NWIN) & 1u, __LINE__);
                WSP(1)
                const WsPoint &e = ent[P & (WS_NENT - 1)];
                if (e.done) break;
                const int RH = e.H - s + 1, RW = e.W - s + 1, xoff = e.x0 & 15;
                const int nxq = (xoff + RW + 15) >> 4;
                const int n16 = (RH + 1 + 15) & ~15;
                const uint32_t idesc = tc_idesc_u8(n16);
                const unsigned set = P & 1u;
                const uint32_t dcol = tbase + set * WS_ACC_COLS + (uint32_t)(w * 64);
                const uint64_t bdesc0 = tc_smem_desc(smem_u32(sWin + (size_t)ws * g.win_bytes + (size_t)w * PS), (uint32_t)PS, 128u);
                const uint32_t b_slot_full = bar0 + (uint32_t)offsetof(WsBars, slot_full);
                const uint32_t b_slot_empty = bar0 + (uint32_t)offsetof(WsBars, slot_empty);
                const uint64_t a_step = (uint64_t)(g.slot_bytes >> 4), a_kk = (uint64_t)((2 * g.lbo_a) >> 4), b_kk = (uint64_t)((2 * PS) >> 4);
                const bool mine = w < nxq;
                for (int b = 0; b < nbatch; ++b) {
                    const unsigned use = set ? use1 : use0;
                    WSP(0)
                    if (use >= 1u) ws_wait<100u>(BAR(&B.acc_empty[set]), (use - 1u) & 1u, __LINE__);
                    WSP(2)
                    tc_fence_after();
                    uint64_t bd = bdesc0;
                    uint32_t accum = 0u;
                    for (int pr = 0; pr < g.npairs; ++pr) {
                        ws_wait<100u>(b_slot_full + 8u * (uint32_t)slot, round, __LINE__);
                        WSP(3)
                        tc_fence_after();
                        if (mine) {
                            tc_mma_i8_ss(dcol, ad, bd, idesc, accum);
                            uint64_t a2 = ad, b2 = bd;
#pragma unroll 1
                            for (int kk = 1; kk < g.ks; ++kk) {
                                a2 += a_kk; b2 += b_kk;
                                tc_mma_i8_ss(dcol, a2, b2, idesc, 1u);
                            }
                        }
                        accum = 1u;
                        bd += 2;
                        tc_commit_addr(b_slot_empty + 8u * (uint32_t)slot);
                        ad += a_step;
                        if (++slot == g.nslots) { slot = 0; round ^= 1u; ad = adesc0; }
                    }
                    tc_commit_addr(BAR(&B.acc_full[set]));
                    if (set) ++use1; else ++use0;
                }
                tc_commit_addr(BAR(&B.win_empty[ws]));
                ++P;
            }
            if (w == 0) WSP_OUT(1)
            if (w == 0) {
                total_pts_s[0] = (P + 1u) / 2u; total_pts_s[1] = P / 2u;
                __threadfence_block();
                all_done_s = 1;
                __threadfence_block();
            }
            // poison completion of both accumulator barriers (the epilogue groups leave on it)
            if (use0 >= 1u) ws_wait(BAR(&B.acc_empty[0]), (use0 - 1u) & 1u, __LINE__);
            ws_arrive(BAR(&B.acc_full[0]));
            if (use1 >= 1u) ws_wait(BAR(&B.acc_empty[1]), (use1 - 1u) & 1u, __LINE__);
            ws_arrive(BAR(&B.acc_full[1]));
        }
    } else if (warp < WS_W_STATS) {
        // ================================================================ gather + Toeplitz expansion
        const int gt = tid - WS_W_GATHER * 32, gw = warp - WS_W_GATHER;
        const int nwords = g.nwords, tw = g.tw;
        const int rows_per_pass = (32 * WS_NG) / nwords;
        const int gi = gt / nwords, wj = gt - gi * nwords;
        const bool active = gi < rows_per_pass;
        double djv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) djv[k] = (double)min(4 * wj + k, s - 1);     // columns past the row repeat the last one (discarded)
        // expansion tasks of this lane (two per row pair; task -> (angle, row parity, word) never changes)
        int ex_src[2], ex_ip[2], ex_dst[2][4];
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            const int t = lane + 32 * it;
            const int rest = t / (nwords + 1), wjj = t - rest * (nwords + 1);
            const int ai = rest >> 1, ip = rest & 1;
            ex_ip[it] = ip;
            ex_src[it] = (ai * s + ip) * tw + wjj;
#pragma unroll
            for (int ee = 0; ee < 4; ++ee) {
                const int wq = wjj + ee;
                ex_dst[it][ee] = (2 * ai + ip) * 16 + (wq >> 2) * g.lbo_a + (wq & 3) * 4 + ee * 512;
            }
        }
        unsigned P = 0, J = 0;
        int qslot = 0;                    // slot of the job's first row pair
        unsigned quse = 0;                // ... and how often that slot has been used before
        WSP_DECL
        for (;;) {
            const unsigned ws = P % WS_NWIN;
            WSP(0)
            ws_wait<100u>(BAR(&B.win_full[ws]), (P / WS_NWIN) & 1u, __LINE__);
            WSP(1)
            const WsPoint &e = ent[P & (WS_NENT - 1)];
            if (e.done) break;
            const double c1 = e.c1, r1 = e.r1;
            const long long e_pt = e.pt, e_pi = e.pi;
            const int e_x0 = e.x0, e_W = e.W, e_H = e.H;
            const uint8_t *patch = sWin + (size_t)ws * g.win_bytes + (size_t)g.npanels * PS - ((size_t)e.py0 * g.pbw + e.px0);
            for (int a0 = 0; a0 < A_; a0 += per, ++J) {
                const int nb = min(per, A_ - a0);
                uint32_t *buf = sTpl + (J & 1u) * g.tpl_buf_words;
                WsTplRec &tr = trec[J & (WS_NENT - 1)];
                // which angles can skip the bounds checks (warp-uniform)
                unsigned inside_mask = 0;
                // every sample lies within 0.7072 s + 2 px of (r1, c1) whatever the angle (the rotation keeps the template centre
                // within 1 px of it): a point that far from the image border needs no per-angle test
                {
                    const double rad = 0.7072 * (double)s + 3.0;
                    if (r1 >= rad && c1 >= rad && r1 <= (double)(a.rows1 - 1) - rad && c1 <= (double)(a.cols1 - 1) - rad) inside_mask = (1u << nb) - 1u;
                }
                if (inside_mask == 0u)
                for (int ai = 0; ai < nb; ++ai) {
                    const double *tab = a.tab + 4 * (a0 + ai);
                    if (template_inside_warp(a.rows1, a.cols1, __dsub_rn(r1, tab[2]), __dsub_rn(c1, tab[3]), tab[0], tab[1], s))
                        inside_mask |= 1u << ai;
                }
                const bool all_fast = a.rot_order == 0 && inside_mask == (1u << nb) - 1u;
                WSD(50)
                uint32_t ls0 = 0, ls1 = 0, ls2 = 0, lq0 = 0, lq1 = 0, lq2 = 0;
                int lzero = 0;
                auto account = [&](int ai, uint32_t word, int nvalid) {
                    // sums over the valid bytes of the word (the others are 0); zero test on the valid bytes only
                    const uint32_t sm_ = __dp4a(word, 0x01010101u, 0u), sq_ = __dp4a(word, word, 0u);
                    ls0 += ai == 0 ? sm_ : 0u; ls1 += ai == 1 ? sm_ : 0u; ls2 += ai == 2 ? sm_ : 0u;
                    lq0 += ai == 0 ? sq_ : 0u; lq1 += ai == 1 ? sq_ : 0u; lq2 += ai == 2 ? sq_ : 0u;
                    const uint32_t filled = nvalid >= 4 ? word : (word | (0xffffffffu << (8 * nvalid)));
                    // a zero byte among the valid ones: (x - 0x01010101) & ~x & 0x80808080
                    lzero |= (((filled - 0x01010101u) & ~filled & 0x80808080u) != 0u);
                };
                if (active) {
                    const int nrow = nb * s;
                    const int nvalid = min(4, s - 4 * wj);
                    if (all_fast) {
                        // four tasks (16 pixels) per step: all loads are in flight before the first is used
                        for (int R0 = gi; R0 < nrow; R0 += 4 * rows_per_pass) {
                            uint32_t v[4][4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int R = min(R0 + u * rows_per_pass, nrow - 1);
                                const int ai = (R >= s) + (R >= 2 * s), i = R - ai * s;
                                const double *tab = a.tab + 4 * (a0 + ai);
                                const double cs = tab[0], sn = tab[1];
                                const double off0 = __dsub_rn(r1, tab[2]), off1 = __dsub_rn(c1, tab[3]);
                                const double di = (double)i;
                                const double br = __dadd_rn(off0, __dmul_rn(di, cs));
                                const double bc = __dadd_rn(off1, __dmul_rn(di, -sn));
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    const double row = __dadd_rn(br, __dmul_rn(djv[k], sn));
                                    const double col = __dadd_rn(bc, __dmul_rn(djv[k], cs));
                                    // nearest sample (scipy order 0: floor(x + 0.5)) out of the staged patch of image 1
                                    const int ri = __double2int_rd(__dadd_rn(row, 0.5)), ci = __double2int_rd(__dadd_rn(col, 0.5));
                                    v[u][k] = patch[ri * g.pbw + ci];
                                }
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int R = R0 + u * rows_per_pass;
                                if (R < nrow) {
                                    const int ai = (R >= s) + (R >= 2 * s), i = R - ai * s;
                                    uint32_t word = v[u][0];
                                    if (nvalid > 1) word |= v[u][1] << 8;
                                    if (nvalid > 2) word |= v[u][2] << 16;
                                    if (nvalid > 3) word |= v[u][3] << 24;
                                    account(ai, word, nvalid);
                                    buf[(ai * s + i) * tw + 1 + wj] = word;
                                }
                            }
                        }
                    } else {
                        for (int R = gi; R < nrow; R += rows_per_pass) {
                            const int ai = (R >= s) + (R >= 2 * s), i = R - ai * s;
                            const double *tab = a.tab + 4 * (a0 + ai);
                            const double cs = tab[0], sn = tab[1];
                            const double off0 = __dsub_rn(r1, tab[2]), off1 = __dsub_rn(c1, tab[3]);
                            const double di = (double)i;
                            const double br = __dadd_rn(off0, __dmul_rn(di, cs));
                            const double bc = __dadd_rn(off1, __dmul_rn(di, -sn));
                            const bool inside = (inside_mask >> ai) & 1u;
                            uint32_t word = 0;
#pragma unroll 1
                            for (int k = 0; k < nvalid; ++k) {
                                const double row = __dadd_rn(br, __dmul_rn(djv[k], sn));
                                const double col = __dadd_rn(bc, __dmul_rn(djv[k], cs));
                                const uint32_t v = inside ? template_sample<false>(a.img1, a.rows1, a.cols1, a.pitch1, row, col, a.rot_order)
                                                          : template_sample<true>(a.img1, a.rows1, a.cols1, a.pitch1, row, col, a.rot_order);
                                word |= v << (8 * k);
                            }
                            account(ai, word, nvalid);
                            buf[(ai * s + i) * tw + 1 + wj] = word;
                        }
                    }
                }
                {   // template sums: one shared-memory atomic per warp, angle and quantity
                    ls0 = __reduce_add_sync(0xffffffffu, ls0); lq0 = __reduce_add_sync(0xffffffffu, lq0);
                    if (nb > 1) { ls1 = __reduce_add_sync(0xffffffffu, ls1); lq1 = __reduce_add_sync(0xffffffffu, lq1); }
                    if (nb > 2) { ls2 = __reduce_add_sync(0xffffffffu, ls2); lq2 = __reduce_add_sync(0xffffffffu, lq2); }
                    lzero = __any_sync(0xffffffffu, lzero);
                    if (lane == 0) {
                        atomicAdd(&tr.tsum[0], ls0); atomicAdd(&tr.tsq[0], lq0);
                        if (nb > 1) { atomicAdd(&tr.tsum[1], ls1); atomicAdd(&tr.tsq[1], lq1); }
                        if (nb > 2) { atomicAdd(&tr.tsum[2], ls2); atomicAdd(&tr.tsq[2], lq2); }
                        if (lzero) tr.zero = 1;
                    }
                }
                if (gt == 0) { tr.pt = e_pt; tr.pi = e_pi; tr.x0 = e_x0; tr.W = e_W; tr.H = e_H; }
                if (gt == 32) {          // clear the record of the next job (nobody reads it any more)
                    WsTplRec &nx = trec[(J + 1u) & (WS_NENT - 1)];
                    nx.zero = 0;
                    for (int k = 0; k < 3; ++k) { nx.tsum[k] = 0u; nx.tsq[k] = 0u; }
                }
                WSP(2)
                WSD(100)
                ws_bar(1, 32 * WS_NG);
                WSD(101)
                WSP(3)
                if (lane == 0) ws_arrive(BAR(&B.tpl_full[J & (WS_NENT - 1)]));
                // ---- expansion: row pair pr -> A slot (q + pr) % nslots
                const int ntask = 2 * nb * (nwords + 1);
                for (int pr = gw; pr < g.npairs; pr += WS_NG) {
                    int slot = qslot + pr;
                    unsigned use = quse;
                    while (slot >= g.nslots) { slot -= g.nslots; ++use; }
                    WSD(200 + pr)
                    WSP(4)
                    if (use >= 1u) ws_wait(bar0 + (uint32_t)offsetof(WsBars, slot_empty) + 8u * (uint32_t)slot, (use - 1u) & 1u, __LINE__);
                    WSP(5)
                    uint8_t *sl = sA + (size_t)slot * g.slot_bytes;
                    const uint32_t *bp = buf + 2 * pr * tw;
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        if (lane + 32 * it < ntask) {
                            uint32_t wlo = 0, whi = 0;
                            if (2 * pr + ex_ip[it] < s) { wlo = bp[ex_src[it]]; whi = bp[ex_src[it] + 1]; }
                            const uint32_t f1 = __byte_perm(wlo, whi, 0x6543), f2 = __byte_perm(wlo, whi, 0x5432), f3 = __byte_perm(wlo, whi, 0x4321);
#pragma unroll
                            for (int ee = 0; ee < 4; ++ee) {
                                uint8_t *pw = sl + ex_dst[it][ee];
                                *reinterpret_cast<uint32_t *>(pw) = whi;
                                *reinterpret_cast<uint32_t *>(pw + 128) = f1;
                                *reinterpret_cast<uint32_t *>(pw + 256) = f2;
                                *reinterpret_cast<uint32_t *>(pw + 384) = f3;
                            }
                        }
                    }
                    for (int t = lane + 64; t < ntask; t += 32) {           // wide templates: more than 64 tasks per pair
                        const int rest = (int)__umulhi((unsigned)t, g.inv_nw1);
                        const int wjj = t - rest * (nwords + 1);
                        const int ai = rest >> 1, ip = rest & 1;
                        const int i = 2 * pr + ip;
                        uint32_t wlo = 0, whi = 0;
                        if (i < s) {
                            const uint32_t *rowp = buf + (ai * s + i) * tw + wjj;
                            wlo = rowp[0]; whi = rowp[1];
                        }
                        uint32_t f[4];
                        f[0] = whi;
                        f[1] = __byte_perm(wlo, whi, 0x6543);
                        f[2] = __byte_perm(wlo, whi, 0x5432);
                        f[3] = __byte_perm(wlo, whi, 0x4321);
                        uint8_t *rowbase = sl + (2 * ai + ip) * 16;
#pragma unroll
                        for (int ee = 0; ee < 4; ++ee) {
                            const int wq = wjj + ee;
                            uint8_t *pw = rowbase + (wq >> 2) * g.lbo_a + (wq & 3) * 4 + ee * 4 * 128;
#pragma unroll
                            for (int c = 0; c < 4; ++c) *reinterpret_cast<uint32_t *>(pw + c * 128) = f[c];
                        }
                    }
                    WSD(300 + pr)
                    WSP(6)
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) ws_arrive(bar0 + (uint32_t)offsetof(WsBars, slot_full) + 8u * (uint32_t)slot);
                    WSP(7)
                    WSD(400 + pr)
                }
                WSD(500)
                qslot += g.npairs;
                while (qslot >= g.nslots) { qslot -= g.nslots; ++quse; }
                WSP(4)
            }
            ++P;
        }
        if (gt == 0) WSP_OUT(2)
    } else if (warp < WS_W_EPI) {
        // ================================================================ window statistics
        const int st_ = tid - WS_W_STATS * 32;
        uint32_t *hqT = reinterpret_cast<uint32_t *>(ws_smem + g.off_hs);
        uint16_t *hsT = reinterpret_cast<uint16_t *>(hqT + g.hs_words);        // a row sum of s bytes fits 16 bits (s <= 112)
        const int hp = g.hp;
        unsigned P = 0;
        WSP_DECL
        for (;;) {
            const unsigned ws = P % WS_NWIN;
            WSP(0)
            ws_wait<100u>(BAR(&B.win_full[ws]), (P / WS_NWIN) & 1u, __LINE__);
            WSP(1)
            const WsPoint &e = ent[P & (WS_NENT - 1)];
            if (e.done) break;
            const int W = e.W, H = e.H, xoff = e.x0 & 15;
            const int RH = H - s + 1, RW = W - s + 1;
            // the window sums also go to the work item's hand-off region, for pm_tail_kernel
            uint32_t *gsum = reinterpret_cast<uint32_t *>(a.tail_maps) + (size_t)e.pi * tail_item_words(a.tail_stride, 1) + a.tail_stride;
            uint32_t *gsq = gsum + a.tail_stride;
            const unsigned set = P % (unsigned)g.nstat;
            if (P >= (unsigned)g.nstat) ws_wait<200u>(BAR(&B.stats_empty[set]), ((P / (unsigned)g.nstat) - 1u) & 1u, __LINE__);
            WSP(2)
            uint32_t *wsq = reinterpret_cast<uint32_t *>(ws_smem + g.off_stat + (size_t)set * g.stat_bytes);
            uint32_t *wsum = wsq + a.max_rr;
            const uint8_t *win = sWin + (size_t)ws * g.win_bytes;
            // horizontal sliding sums: one (window row, x segment) per thread
            {
                int nsegx = WS_NST / H;
                if (nsegx < 1) nsegx = 1;
                if (nsegx > 4) nsegx = 4;
                const int Lx = (RW + nsegx - 1) / nsegx;
                for (int t = st_; t < H * nsegx; t += WS_NST) {
                    const int sg = t / H, r = t - sg * H;
                    const int xs = sg * Lx, xe = min(RW, xs + Lx);
                    if (xs >= xe) continue;
                    const uint8_t *rowp = win + 16 * r;
                    const int c0 = xs + xoff;                            // staged column of the segment's first window byte
                    // the first box sum from aligned words (two dot products per word), masked at both ends
                    uint32_t sum = 0, sq = 0;
                    {
                        const int cend = c0 + s;
                        int cw = c0 & ~3;                                // column of the current word
                        const int q = c0 >> 2;
                        const uint8_t *wp = rowp + (q >> 2) * PS + (q & 3) * 4;
                        int wleft = 4 - (q & 3);                         // words left in this 16-byte panel row
                        uint32_t mlo = 0xffffffffu << (8 * (c0 & 3));
                        while (cw < cend) {
                            uint32_t w = *reinterpret_cast<const uint32_t *>(wp) & mlo;
                            const int hi = cend - cw;                    // valid bytes of this word end at byte hi (>= 1)
                            if (hi < 4) w &= 0xffffffffu >> (8 * (4 - hi));
                            sum = __dp4a(w, 0x01010101u, sum);
                            sq = __dp4a(w, w, sq);
                            mlo = 0xffffffffu;
                            cw += 4; wp += 4;
                            if (--wleft == 0) { wp += PS - 16; wleft = 4; }
                        }
                    }
                    // two byte streams -- the column leaving the box and the column entering it -- read as aligned words, four
                    // columns per iteration (byte loads of 32 rows 16 bytes apart were 4-way bank conflicted: 13 % of all
                    // shared-memory wavefronts of the kernel); the word one ahead is always inside the slot (x + s <= W, and the
                    // staged panels are followed by the template patch)
                    const int c1 = c0 + s;
                    const uint8_t *pwo = rowp + (c0 >> 4) * PS + (c0 & 12);
                    const uint8_t *pwi = rowp + (c1 >> 4) * PS + (c1 & 12);
                    int wo_left = 4 - ((c0 >> 2) & 3), wi_left = 4 - ((c1 >> 2) & 3);      // words left in the 16-byte panel row
                    const unsigned sho = 8u * (unsigned)(c0 & 3), shi = 8u * (unsigned)(c1 & 3);
                    uint32_t wo = *reinterpret_cast<const uint32_t *>(pwo), wi = *reinterpret_cast<const uint32_t *>(pwi);
                    uint16_t *hsp = hsT + xs * hp + r;
                    uint32_t *hqp = hqT + xs * hp + r;
                    for (int x = xs; x < xe; x += 4) {
                        pwo += 4; if (--wo_left == 0) { pwo += PS - 16; wo_left = 4; }
                        pwi += 4; if (--wi_left == 0) { pwi += PS - 16; wi_left = 4; }
                        const uint32_t wo2 = *reinterpret_cast<const uint32_t *>(pwo), wi2 = *reinterpret_cast<const uint32_t *>(pwi);
                        const uint32_t out4 = __funnelshift_r(wo, wo2, sho), in4 = __funnelshift_r(wi, wi2, shi);
                        wo = wo2; wi = wi2;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if (x + j < xe) { *hsp = (uint16_t)sum; *hqp = sq; }
                            hsp += hp; hqp += hp;
                            const uint32_t va = (out4 >> (8 * j)) & 0xffu, vb = (in4 >> (8 * j)) & 0xffu;
                            const uint32_t d = vb - va;
                            sum += d; sq += d * (vb + va);
                        }
                    }
                }
            }
            WSP(3)
            ws_bar(2, WS_NST);
            WSP(4)
            if (lane == 0) ws_arrive(BAR(&B.win_empty[ws]));        // this warp is done with the window
            // vertical sliding sums -> window sum / sum of squares per displacement
            {
                int nseg = WS_NST / RW;
                if (nseg < 1) nseg = 1;
                if (nseg > RH) nseg = RH;
                const int L = (RH + nseg - 1) / nseg;
                for (int t = st_; t < RW * nseg; t += WS_NST) {
                    const int sg = t / RW, x = t - sg * RW;
                    const int ys = sg * L, ye = min(RH, ys + L);
                    if (ys >= ye) continue;
                    const uint16_t *hs = hsT + x * hp; const uint32_t *hq = hqT + x * hp;
                    uint32_t sum = 0, sq = 0;
                    for (int i = 0; i < s; ++i) { sum += hs[ys + i]; sq += hq[ys + i]; }
                    for (int y = ys; y < ye; ++y) {
                        const int idx = y * RW + x;
                        wsum[idx] = sum; wsq[idx] = sq;
                        gsum[idx] = sum; gsq[idx] = sq;
                        if (y + 1 < ye) { sum += (uint32_t)hs[y + s] - (uint32_t)hs[y]; sq += hq[y + s] - hq[y]; }
                    }
                }
            }
            WSP(5)
            __syncwarp();
            if (lane == 0) ws_arrive(BAR(&B.stats_full[set]));
            ws_bar(2, WS_NST);                                          // hsT / hqT are free again
            WSP(4)
            ++P;
        }
        if (st_ == 0) WSP_OUT(3)
    } else {
        // ================================================================ epilogue groups (points P = e, e + 2, ...)
        const int eg = (warp - WS_W_EPI) >> 2;
        const int et = tid - (WS_W_EPI + 4 * eg) * 32;
        const int ew = et >> 5;
        const int quarter = warp & 3;
        const int barid = 3 + eg;
        WsEpi &E = epi[eg];
        int32_t *C = reinterpret_cast<int32_t *>(ws_smem + g.off_c) + (size_t)eg * nab * g.cpl;
        const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
        const int dx = 4 * quarter + (lane >> 3), aa = (lane >> 1) & 3, ip = lane & 1;
        const int Ni = s * s;
        const long long Nll = (long long)Ni;
        uint32_t *list = reinterpret_cast<uint32_t *>(ws_smem + g.off_list) + eg * WS_LIST;
        float *emax = reinterpret_cast<float *>(ws_smem + g.off_emax) + (size_t)eg * a.max_rr;
        unsigned acc_use = 0;
        bool leave = false;
        WSP_DECL
        for (unsigned n = 0; !leave; ++n) {
            const unsigned P = (unsigned)eg + 2u * n;
            const unsigned sset = P % (unsigned)g.nstat;
            const uint32_t *wsq = reinterpret_cast<const uint32_t *>(ws_smem + g.off_stat + (size_t)sset * g.stat_bytes);
            const uint32_t *wsum = wsq + a.max_rr;
            float best_r = -INFINITY;
            int best_a = -1, best_idx = 0;
            uint32_t best_tsum = 0u, best_tsq = 0u;
            bool invalid = false;
            long long pt = 0, pi = 0;
            int W = 0, H = 0, xoff = 0, RH = 0, RW = 0, RR = 0;
            for (int b = 0; b < nbatch; ++b) {
                const unsigned J = P * (unsigned)nbatch + (unsigned)b;
                WSP(0)
                ws_wait<100u>(BAR(&B.acc_full[eg]), acc_use & 1u, __LINE__); ++acc_use;
                WSP(1)
                if (b == 0 && all_done_s && n == total_pts_s[eg]) { leave = true; break; }
                tc_fence_after();
                ws_wait(BAR(&B.tpl_full[J & (WS_NENT - 1)]), (J >> 3) & 1u, __LINE__);
                const WsTplRec &tr = trec[J & (WS_NENT - 1)];
                if (b == 0) {
                    pt = tr.pt; pi = tr.pi; W = tr.W; H = tr.H; xoff = tr.x0 & 15;
                    RH = H - s + 1; RW = W - s + 1; RR = RH * RW;
                    ws_wait<100u>(BAR(&B.stats_full[sset]), (P / (unsigned)g.nstat) & 1u, __LINE__);
                }
                WSP(2)
                const int a0 = b * per, nb = min(per, A_ - a0);
                const bool zero = tr.zero != 0;
                if (et < nb) E.st[et] = templ_stats(tr.tsum[et], tr.tsq[et], a.inv_area, a.sqrt_inv_area);
                // ---- combined correlation numerators -> C[a][y * RW + x]
                if (!invalid && !zero) {
                    const int nxq = (xoff + RW + 15) >> 4;
                    const int n16 = (RH + 1 + 15) & ~15;
                    const int ak = aa < nb ? aa : 0;
                    for (int xq = 0; xq < nxq; ++xq) {
                        const int xw = 16 * xq + 4 * quarter - xoff;            // first x of this warp's four dx
                        if (xw + 3 < 0 || xw >= RW) continue;                   // warp-uniform
                        const int x = 16 * xq + dx - xoff;
                        const bool lane_ok = x >= 0 && x < RW && aa < nb;
                        int32_t *cp = C + ak * g.cpl + (lane_ok ? x : 0) - ip * RW;     // row y = c0 + 2 t - ip
                        const uint32_t tad = tbase + (uint32_t)eg * WS_ACC_COLS + (uint32_t)(xq * 64) + lane_base;
                        uint32_t carry = 0;
                        for (int c0 = 0; c0 < n16; c0 += 16) {
                            uint32_t r[16];
                            tc_ld16(tad + (uint32_t)c0, r);
                            tc_ld_wait();
                            const int ylo = ip - c0, yhi = RH + ip - c0;           // valid 2 t: ylo <= 2 t < yhi
#pragma unroll
                            for (int t = 0; t < 8; ++t) {
                                const uint32_t send = ip ? r[2 * t + 1] : (t ? r[t ? 2 * t - 1 : 0] : carry);
                                const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 1);
                                if (lane_ok && 2 * t >= ylo && 2 * t < yhi) cp[(c0 + 2 * t) * RW] = (int32_t)(r[2 * t] + recv);
                            }
                            carry = r[15];
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) ws_arrive(BAR(&B.acc_empty[eg]));
                if (zero) invalid = true;
                WSP(3)
                ws_bar(barid, 128);
                WSP(4)
                if (invalid) continue;

                // ---- screening from the exact integers (the estimate and its error bound: WS_MARGIN above)
                float tinv[3];
                int tsm[3];
                unsigned flat = 0u;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const int kk = k < nb ? k : 0;
                    tsm[k] = (int)tr.tsum[kk];
                    const long long tv = Nll * (long long)tr.tsq[kk] - (long long)tsm[k] * (long long)tsm[k];
                    tinv[k] = tv > 0 ? (float)(1.0 / sqrt((double)tv)) : 0.0f;
                    if (k < nb && E.st[k].flat) flat |= 1u << k;
                }
                float mx = nb == 3 ? ws_screen<3>(C, g.cpl, wsum, wsq, emax, RR, et, (unsigned)Ni, tsm, tinv)
                         : nb == 2 ? ws_screen<2>(C, g.cpl, wsum, wsq, emax, RR, et, (unsigned)Ni, tsm, tinv)
                                   : ws_screen<1>(C, g.cpl, wsum, wsq, emax, RR, et, (unsigned)Ni, tsm, tinv);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                if (lane == 0) E.m[ew] = mx;
                if (et == 0) E.cnt = 0u;
                WSP(5)
                ws_bar(barid, 128);
                WSP(4)
                // ---- contenders.  The peak of the batch is >= the best lower bound (largest usable estimate - ERR, or 1 for a
                //      flat template, whose map is 1 everywhere); a position can hold it only if an estimate there is >= that
                //      - ERR, or if one cannot be estimated.  Those positions are evaluated exactly, for every angle.
                float Mx = fmaxf(fmaxf(E.m[0], E.m[1]), fmaxf(E.m[2], E.m[3]));
                if (flat) Mx = fmaxf(Mx, 1.0f);
                const float thr = fmaxf(Mx, best_r) - WS_MARGIN;
                for (int idx = et; idx < RR; idx += 128) {
                    if (emax[idx] >= thr) {
                        const unsigned slot = atomicAdd(&E.cnt, 1u);
                        if (slot < (unsigned)WS_LIST) list[slot] = (unsigned)idx;
                    }
                }
                ws_bar(barid, 128);
                unsigned long long key[3] = {0ull, 0ull, 0ull};
                const unsigned cnt = E.cnt;
                if (cnt <= (unsigned)WS_LIST) {
                    for (unsigned t = (unsigned)et; t < cnt * (unsigned)nb; t += 128u) {
                        const unsigned i = t / (unsigned)nb;
                        const int k = (int)(t - i * (unsigned)nb), idx = (int)list[i];
                        const TemplStats &sk = E.st[k];
                        const uint32_t ws = wsum[idx];
                        const double num = __dsub_rn((double)C[k * g.cpl + idx], __dmul_rn((double)ws, sk.mean));
                        const double tt = __dmul_rn(window_den(ws, wsq[idx], a.inv_area), sk.norm);
                        const unsigned long long kv = peak_key(__double2float_rn(ncc_finish(num, tt)), (uint32_t)idx);
#pragma unroll
                        for (int kk = 0; kk < 3; ++kk) if (kk == k && kv > key[kk]) key[kk] = kv;
                    }
                } else {
                    // flat or degenerate content: too many positions the estimates cannot separate -- every angle in full
                    for (int k = 0; k < nb; ++k)
                        if (!((flat >> k) & 1u)) {
                            const unsigned long long kv = ws_exact_pass(C + k * g.cpl, wsum, wsq, E.st[k], a.inv_area, RR, et);
#pragma unroll
                            for (int kk = 0; kk < 3; ++kk) if (kk == k) key[kk] = kv;
                        }
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    key[k] = warp_max_u64(key[k]);
                    if (lane == 0) E.key[ew][k] = key[k];
                }
                ws_bar(barid, 128);
                int pending = -1;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    unsigned long long k0 = E.key[0][k], k1 = E.key[1][k], k2 = E.key[2][k], k3 = E.key[3][k];
                    k0 = k0 > k1 ? k0 : k1; k2 = k2 > k3 ? k2 : k3;
                    unsigned long long kv = k0 > k2 ? k0 : k2;
                    if ((flat >> k) & 1u) kv = peak_key(1.0f, 0u);
                    if (kv == 0ull) continue;                   // no position of this angle listed
                    const float v = key_f32((uint32_t)(kv >> 32));
                    if (v > best_r) {
                        best_r = v; best_idx = (int)(0xffffffffu - (uint32_t)(kv & 0xffffffffull));
                        best_a = a0 + k; pending = k;
                    }
                }
                if (pending >= 0) {
                    // hand-off: the winning angle's numerators (pm_tail_kernel rebuilds its float map)
                    int32_t *gc = reinterpret_cast<int32_t *>(a.tail_maps) + (size_t)pi * tail_item_words(a.tail_stride, 1);
                    const int32_t *cs = C + pending * g.cpl;
                    for (int idx = et; idx < RR; idx += 128) gc[idx] = cs[idx];
                    best_tsum = tr.tsum[pending]; best_tsq = tr.tsq[pending];
                }
                WSP(6)
                ws_bar(barid, 128);          // C, E.st, E.key, the estimates and the list are free for the next batch
                WSP(4)
            }
            if (leave) {
                if (et == 0) WSP_OUT(4 + eg)
                break;
            }
            __syncwarp();
            if (lane == 0) ws_arrive(BAR(&B.stats_empty[sset]));
            if (et == 0) {
                if (invalid || best_a < 0) {
                    double *o = a.out + 5 * pt;
                    o[0] = o[1] = o[2] = o[3] = o[4] = nan("");
                    if (a.status) a.status[pt] = 0;
                    a.tail_recs[pi].pt = -1;
                } else {
                    PmTailRec rec;
                    rec.pt = (int)pt; rec.RH = RH; rec.RW = RW; rec.H = H; rec.W = W;
                    rec.best_idx = best_idx; rec.best_a = best_a; rec.best_r = best_r;
                    rec.mode = 1; rec.tsum = best_tsum; rec.tsq = best_tsq;
                    a.tail_recs[pi] = rec;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) { __syncwarp(); tc_dealloc(tbase, 512u); }
}

}  // namespace sid
