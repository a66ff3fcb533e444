// sid_pm_tc_kernel.cuh -- the fused pattern-matching kernel with the correlation on the 5th-generation tensor
// cores (tcgen05.mma kind::i8, u8 x u8 -> s32, accumulators in tensor memory).
//
// Same per-point work and the same arithmetic contract as pm_points_kernel (sid_pm_kernel.cuh; reference
// pmlib.py:176-212 and everything it calls); only the contraction is organised differently:
//
//   corr[a][y][x] = sum_i sum_j W[y+i][x+j] * T_a[i][j]
//                 = sum_i sum_k Toep_{a,i}[x][k] * W[y+i][k],      Toep_{a,i}[x][k] = T_a[i][k - x]   (0 outside)
//
//   D[(x,a)][y] (128 TMEM lanes x N columns)  +=  A_i[(x,a)][k] (TMEM, 128 lanes x K bytes)  *  B_i[y][k] (shared memory)
//
//   * B_i is the staged search window itself.  It sits in shared memory as 16-byte column panels (K-major, no
//     swizzle: rows 16 B apart, SBO = 128, LBO = panel stride), so "window rows i .. i+N-1" is the same matrix
//     descriptor with the start address advanced by 16*i -- no im2col, no copy.  Panels are written by TMA
//     (one 16-byte-wide box per panel, out-of-image bytes read as 0).
//   * A_i, the Toeplitz band of template row i for the <= 3 angles of a batch, is written into tensor memory by
//     the lane's own thread (tcgen05.st.32x32b: lane m = nab*x + a).  The byte shift x + (window offset) is
//     absorbed by keeping FOUR byte-shifted copies of every template row in shared memory, so a lane reads aligned
//     words only; a warp's rows are non-zero in a narrow band of K words, which is all it writes.
//   * Two warp groups (4 warps = the four TMEM lane quarters) alternate template rows; three A slots; after the
//     group barrier up to four warps issue one MMA each (measured: one thread issues at most one MMA per ~60-100
//     clk whatever its size, four issuers reach the pipe's 128*N/256 clk; profiles/r02_tcgen05_i8_rates.txt) and
//     commit to the slot's mbarrier.
//   * Epilogue: tcgen05.ld the lane's accumulator row (all y of one (x, a)), OpenCV's FP64 normalisation, map
//     store, running argmax -- y ascending is flat-index ascending for a fixed x, so a strict '>' is np.argmax.
//
// Result maps wider than 128/nab positions are processed in x tiles (the B descriptor moves by whole panels,
// the residual byte offset goes into the Toeplitz shift).
#pragma once
#include "sid_pm_kernel.cuh"

namespace sid {

constexpr int TC_THREADS = 256;
#ifndef SID_TC_OLD_TPL_LAYOUT
#define SID_TC_OLD_TPL_LAYOUT 0        // A/B switch: 1 = round-2 first template layout (copy stride 20 words, angle skew 4)
#endif

// Launch-uniform geometry of the tcgen05 path, computed on the host (pm_tc_geometry).
struct PmTcCfg {
    int nab;        // angles per batch == TMEM lanes per x position
    int xt;         // x positions per tile = 128 / nab
    int ks;         // K steps (32 bytes) per template row
    int nissue;     // issuing warps per warp group = min(ks, 4)
    int nb8;        // 8-word groups a warp writes per Toeplitz row (its band of non-zero K words)
    int slotc;      // TMEM columns per A slot
    int nslot;      // A slots shared by the two warp groups (3, or 2 when that keeps the allocation at 256 columns)
    int nacc;       // accumulators (K step ks adds into accumulator ks % nacc)
    int n16max;     // accumulator width: max N (result rows rounded up to 16)
    int tmem_cols;  // TMEM allocation (power of two)
    int wrows;      // rows per window panel (multiple of 8)
    int npanels;    // panels resident
    int np_load;    // panels loaded per point
    int load_rows;  // rows loaded per panel (TMA box height)
    int ctlw;       // left pad (words) of a template-row copy
    int tpw;        // words per template-row copy
    int tang;       // bytes per angle in the template area
    int win_bytes, tpl_bytes;
    unsigned par_mask;  // bit b: slot barrier b completes an ODD number of phases per tile (its parity flips from tile to tile)
    // window sums on the tensor cores (set by the host when shared memory / tensor memory allow it)
    int mma_sums;   // 1: horizontal box sums of v and v^2 by a ones-Toeplitz MMA, vertical sums from TMEM rows
    int n16hmax;    // accumulator width of those MMAs: window rows rounded up to 16
    int sq_off;     // byte offset (from the scratch slab) of the two squares windows (alias the result maps)
    int wsq_off;    // byte offset (from the scratch slab) of the u32 sums of squares
};

inline bool pm_tc_geometry(int s, int Rmax, int Wmax, int n_angles, PmTcCfg &g) {
    if (s < 2 || s > 128 || Rmax < 2 || Wmax > 256) return false;
    g.nab = n_angles < 3 ? n_angles : 3;
    g.xt = 128 / g.nab;
    const int xte = g.xt < Rmax ? g.xt : Rmax;
    g.ks = (xte + s - 1 + 15 + 31) / 32;
    g.nissue = g.ks < 4 ? g.ks : 4;
    const int xspan = g.nab == 1 ? 32 : 31 / g.nab + 2;             // distinct x positions among a warp's 32 lanes
    const int bandw = (3 + (xspan - 1) + (s - 1)) / 4 + 1;          // K words between a warp's first and last non-zero byte
    g.nb8 = (bandw + 7) / 8;
    g.ctlw = (3 + xspan - 1) / 4;
    // Bank layout of the template area: a warp's 32 lanes (11-12 x positions x 3 angles) read, per band word, from 12
    // (angle, copy) rows at 3-4 consecutive word offsets each.  Copy stride == 24 (mod 32) words puts the four copies on
    // banks 0 / 24 / 16 / 8 and an angle skew of 3 words interleaves the angles between them (the first layout, stride
    // 20 for both, made 3-way conflicts of every band load: 51 % of the kernel's shared wavefronts were replays).
    int tpw = g.ctlw + 8 * g.nb8;
    int askew = 16;
    if (tpw <= 24 && !SID_TC_OLD_TPL_LAYOUT) { tpw = 24; askew = 12; }
    else { tpw = (tpw + 3) & ~3; if ((tpw & 7) == 0) tpw += 4; }
    g.tpw = tpw;
    const int max_cw0 = (96 / g.nab + 15) >> 2;                     // first band word of the last warp, worst offset
    int slotc = max_cw0 + 8 * g.nb8;
    if (slotc < 8 * g.ks) slotc = 8 * g.ks;
    g.slotc = (slotc + 7) & ~7;
    g.n16max = (Rmax + 15) & ~15;
    if (g.n16max > 256) return false;
    // 256 columns keep two CTAs resident per SM: one accumulator per K step and three A slots if they fit, else one
    // accumulator, else two slots (measured on cfg2: accumulator count and slot depth change the kernel by < 3 %)
    g.nacc = g.ks; g.nslot = 3;
    if (g.nacc * g.n16max + g.nslot * g.slotc > 256) g.nacc = 1;
    if (g.nacc * g.n16max + g.nslot * g.slotc > 256) g.nslot = 2;
    if (g.nacc * g.n16max + g.nslot * g.slotc > 256) g.nslot = 3;           // one CTA per SM anyway
    const int need = g.nacc * g.n16max + g.nslot * g.slotc;
    if (need > 512) return false;
    g.tmem_cols = 32;
    while (g.tmem_cols < need) g.tmem_cols <<= 1;
    g.wrows = (s + g.n16max + 15) & ~15;                          // >= window rows rounded up to 16 (N of the sums MMAs)
    if (g.wrows < Wmax) g.wrows = (Wmax + 15) & ~15;
    const int ntiles = (Rmax + g.xt - 1) / g.xt;
    g.np_load = (Wmax + 15 + 15) / 16;
    const int p0max = ((ntiles - 1) * g.xt + 15) >> 4;
    g.npanels = p0max + 2 * g.ks;
    if (g.npanels < g.np_load) g.npanels = g.np_load;
    g.load_rows = Wmax;
    g.win_bytes = g.npanels * g.wrows * 16;
    g.tang = s * 4 * g.tpw * 4 + askew;
    // behind the last angle: a row of zeros (dead lanes), a row of ones and a row of 255s (window sums), 4 copies each
    g.tpl_bytes = (g.nab * g.tang + 12 * g.tpw * 4 + 127) & ~127;
    g.par_mask = 0;
    for (int b = 0; b < 2 * g.nslot; ++b)            // rows b, b + 2 nslot, ... of the s template rows commit to barrier b
        if (b < s && (((s - b + 2 * g.nslot - 1) / (2 * g.nslot)) & 1)) g.par_mask |= 1u << b;
    g.n16hmax = (Wmax + 15) & ~15;
    g.mma_sums = 0; g.sq_off = 0; g.wsq_off = 0;
    return true;
}

// ---------------------------------------------------------------- tcgen05 / TMEM primitives
__device__ __forceinline__ void tc_alloc(uint32_t *dst_smem, uint32_t ncols) {      // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_dealloc(uint32_t taddr, uint32_t ncols) {        // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem descriptor], u8 x u8 -> s32, M = 128
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t d, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tc_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// shared-memory matrix descriptor: K-major, no swizzle, sm_100 descriptor version 1
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3fffu) << 32) | ((uint64_t)1 << 46);
}
// instruction descriptor: D = s32, A = B = u8, both K-major, M = 128
__device__ __forceinline__ uint32_t tc_idesc_u8(int n) { return (2u << 4) | ((uint32_t)(n >> 3) << 17) | (8u << 24); }
__device__ __forceinline__ void mbar_wait_addr(uint32_t bar_addr, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar_addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_commit_addr(uint32_t bar_addr) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
}
// the 128 threads of one warp group (barrier 1 or 2; 0 is __syncthreads)
__device__ __forceinline__ void bar_sync_group(int wg) {
    if (wg == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
    else asm volatile("bar.sync 2, 128;" ::: "memory");
}

template <bool SMEM_SCRATCH>
__global__ void __launch_bounds__(TC_THREADS, 2)
pm_tc_kernel(const PmArgs a, const PmTcCfg g, const __grid_constant__ CUtensorMap tmapP) {
    extern __shared__ __align__(128) unsigned char pm_smem[];
    __shared__ PmShared S;
    __shared__ __align__(8) unsigned long long win_bar, slot_bar[6], done_bar[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ uint16_t sq_lut[256];
    __shared__ struct { double c1, r1, c2, r2; long long pt; int x0, y0, W, H, ok; } P;   // current point (written by thread 0)                            // v -> (v*v / 255) << 8 | (v*v % 255)
    unsigned win_phase = 0, done_phase = 0, slot_par = 0;       // slot_par: bit b = parity of completed phases of slot_bar[b]
    const int tid = threadIdx.x, lane = tid & 31, nt = TC_THREADS;
    const int wg = tid >> 7, wiw = (tid >> 5) & 3;              // warp group, warp in group == TMEM lane quarter
    const int s = a.s, nab = g.nab;
    uint8_t *sW = pm_smem;
    uint8_t *sT = pm_smem + g.win_bytes;
    const int PS = g.wrows * 16;                                 // panel stride (bytes)
    const int tpw4 = g.tpw * 4;                                  // bytes per template-row copy

    unsigned char *slab;
    if constexpr (SMEM_SCRATCH) slab = sT + g.tpl_bytes;
    else slab = a.scratch + (size_t)blockIdx.x * a.scratch_per_cta;
    double *wden = reinterpret_cast<double *>(slab);
    uint32_t *wsum = reinterpret_cast<uint32_t *>(wden + a.max_rr);
    float *maps = reinterpret_cast<float *>(wsum + a.max_rr);
    uint32_t *hs = reinterpret_cast<uint32_t *>(maps);
    uint32_t *hq = hs + a.max_hrw;
    uint8_t *sR = slab + g.sq_off, *sD = sR + (size_t)g.npanels * PS;      // squares windows: v^2 = 255 * d + r (mma_sums only)
    uint32_t *wsq = reinterpret_cast<uint32_t *>(slab + g.wsq_off);

    for (int t = tid; t < g.tpl_bytes / 4; t += nt) reinterpret_cast<uint32_t *>(sT)[t] = 0u;   // the padding stays zero for good
    {
        const uint32_t x = (uint32_t)tid * (uint32_t)tid, d = (x + 1u + (x >> 8)) >> 8;          // exact x / 255 for x < 65536
        sq_lut[tid] = (uint16_t)((d << 8) | (x - 255u * d));
    }
    __syncthreads();
    for (int t = tid; t < 8 * s; t += nt) {                      // constant rows: `s` bytes of 1 / of 255, byte-shifted copies
        const int j = t % s, c = (t / s) & 3, which = t / (4 * s);
        sT[(size_t)nab * g.tang + (size_t)(4 + 4 * which + c) * tpw4 + 4 * g.ctlw + c + j] = which ? 255 : 1;
    }
    if (tid == 0) {
        S.next = atomicAdd(a.counter, 1u);
        S.tma_for = 0xffffffffu;
        mbar_init(&win_bar, 1);
        for (int b = 0; b < 6; ++b) mbar_init(&slot_bar[b], g.nissue);
        mbar_init(&done_bar[0], g.nissue);
        mbar_init(&done_bar[1], g.nissue);
    }
    if (tid < 32) tc_alloc(&tmem_base_s, (uint32_t)g.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = tmem_base_s;
    const uint32_t lane_base = (uint32_t)(wiw * 32) << 16;
    const uint32_t tD = tbase, tA = tbase + (uint32_t)(g.nacc * g.n16max);
    const uint64_t bdesc0 = tc_smem_desc(smem_u32(sW), (uint32_t)PS, 128u);
    const unsigned win_tx = (unsigned)(g.np_load * g.load_rows * 16);
    // lane -> (x in tile, angle in batch)
    const int m = tid & 127, xi = m / nab, aa = m - xi * nab;
    const int xi_min = (wiw * 32) / nab;                         // first x of this warp's lanes

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            S.point = S.next;
            const long long pi0 = (long long)S.point;
            if (pi0 < a.n) {
                // issue order matters here (255 threads wait at the barrier below): the point's loads first, then the
                // work-stealing atomic, so that the two global round trips overlap instead of adding up
                const long long pt0 = a.order ? (long long)a.order[pi0] : pi0;
                const double c1 = a.c1[pt0], r1 = a.r1[pt0], c2 = a.c2fg[pt0], r2 = a.r2fg[pt0], brd = a.border[pt0];
                const unsigned int nxt = atomicAdd(a.counter, 1u);
                long long x0, y0; int W, H;
                bool ok = pm_window_rect(a, c1, r1, c2, r2, brd, x0, y0, W, H);
                const int RH0 = H - s + 1, RW0 = W - s + 1;
                if (ok) ok = RH0 * RW0 <= a.max_rr && H * RW0 <= a.max_hrw && H <= g.load_rows &&
                             W + (int)(x0 & 15) <= g.np_load * 16 && RH0 <= g.n16max;
                P.c1 = c1; P.r1 = r1; P.c2 = c2; P.r2 = r2; P.pt = pt0;
                P.x0 = (int)x0; P.y0 = (int)y0; P.W = W; P.H = H; P.ok = ok ? 1 : 0;
                S.next = nxt;
            }
        }
        __syncthreads();
        const long long pi = (long long)S.point;
        if (pi >= a.n) break;
        const bool prefetched = S.tma_for == S.point;
        if (tid == nt - 1) {                                     // look one work item ahead (window prefetch in the tail)
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
        const long long pt = P.pt;
        const double c1 = P.c1, r1 = P.r1, c2 = P.c2, r2 = P.r2;
        double *o = a.out + 5 * pt;
        const int x0 = P.x0, y0 = P.y0, W = P.W, H = P.H;
        const bool ok = P.ok != 0;
        const int RH = H - s + 1, RW = W - s + 1, RR = RH * RW;
        const int xoff = x0 & 15;
        if (prefetched) { mbar_wait(&win_bar, win_phase); win_phase ^= 1u; }
        if (!ok) {
            if (tid == 0) {
                o[0] = o[1] = o[2] = o[3] = o[4] = nan("");
                if (a.status) a.status[pt] = -1;
                if (a.split_tail) a.tail_recs[pi].pt = -1;
            }
            continue;
        }

        // ---- 1. stage the window: one 16-byte-wide TMA box per column panel
        if (tid == 0) {
            if (!prefetched) {
                mbar_expect_tx(&win_bar, win_tx);
                for (int p = 0; p < g.np_load; ++p) tma_load_2d(sW + p * PS, &tmapP, x0 - xoff + 16 * p, y0, &win_bar);
            }
            S.best_r = -INFINITY; S.best_a = -1; S.best_idx = 0; S.best_slot = -1;
        }
        if (!prefetched) { mbar_wait(&win_bar, win_phase); win_phase ^= 1u; }
        __syncthreads();

        if (g.mma_sums) {
            // ---- 2 (tensor cores).  Horizontal box sums of every window row as ONE Toeplitz MMA per quantity:
            //      Hs[x][r] = sum_k Ones[x][k] * W[r][k],   Hq[x][r] = sum_k Ones[x][k] * R[r][k] + 255s[x][k] * D[r][k]
            //      with v^2 = 255 * D + R split into two bytes (exact), then the vertical sliding sums run along each
            //      lane's own TMEM row (columns = window rows) in registers.
            const uint32_t inv_h = 0xffffffffu / (uint32_t)H + 1u;        // u / H == umulhi(u, inv_h) for u < 65536
            for (int t = tid; t < g.np_load * H * 4; t += nt) {
                const int w = t & 3, u = t >> 2, pnl = (int)__umulhi((uint32_t)u, inv_h), r = u - pnl * H;
                const int off = pnl * PS + r * 16 + 4 * w;
                const uint32_t v = *reinterpret_cast<const uint32_t *>(sW + off);
                const uint32_t t0 = sq_lut[v & 255u], t1 = sq_lut[(v >> 8) & 255u], t2 = sq_lut[(v >> 16) & 255u], t3 = sq_lut[v >> 24];
                *reinterpret_cast<uint32_t *>(sR + off) = __byte_perm(__byte_perm(t0, t1, 0x0040), __byte_perm(t2, t3, 0x0040), 0x5410);
                *reinterpret_cast<uint32_t *>(sD + off) = __byte_perm(__byte_perm(t0, t1, 0x0051), __byte_perm(t2, t3, 0x0051), 0x5410);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> visible to the tensor core
            const int n16h = (H + 15) & ~15;
            const uint32_t idesc_h = tc_idesc_u8(n16h);
            const uint32_t tQ = tD + (uint32_t)g.n16hmax;                    // second accumulator: sums of squares
            const uint32_t tOnes = tA + (uint32_t)((g.nslot - 2) * g.slotc), t255 = tA + (uint32_t)((g.nslot - 1) * g.slotc);
            const int ntile_s = (RW + g.xt - 1) / g.xt;
            for (int tile = 0; tile < ntile_s; ++tile) {
                const int xbase = tile * g.xt;
                const int RWt = min(g.xt, RW - xbase);
                const int col0 = xbase + xoff, p0 = col0 >> 4, offt = col0 & 15;
                const int q = xi + offt;
                const int cw0 = (xi_min + offt) >> 2;
                tc_fence_before();
                __syncthreads();
                tc_fence_after();
                {   // clear accumulators and slots
                    uint32_t z[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) z[c] = 0u;
                    const int ncol = g.nacc * g.n16max + g.nslot * g.slotc, half = ((ncol / 8 + 1) / 2) * 8;
                    const int cb = wg * half, ce = min(ncol, cb + half);
                    for (int c = cb; c < ce; c += 8) tc_st8(tD + lane_base + c, z);
                    tc_st_wait();
                    tc_fence_before();
                }
                __syncthreads();
                tc_fence_after();
                {   // warp group 0 writes the ones band, warp group 1 the 255s band (dead lanes: zeros)
                    const uint32_t *p = xi < RWt
                        ? reinterpret_cast<const uint32_t *>(sT + (size_t)nab * g.tang + (size_t)(4 + 4 * wg + (q & 3)) * tpw4) + g.ctlw - (q >> 2) + cw0
                        : reinterpret_cast<const uint32_t *>(sT + (size_t)nab * g.tang);
                    const uint32_t ta = (wg ? t255 : tOnes) + lane_base + (uint32_t)cw0;
                    for (int grp = 0; grp < g.nb8; ++grp) {
                        uint32_t v[8];
#pragma unroll
                        for (int c = 0; c < 8; ++c) v[c] = p[grp * 8 + c];
                        tc_st8(ta + grp * 8, v);
                    }
                    tc_st_wait();
                    tc_fence_before();
                }
                __syncthreads();
                if (lane == 0 && wiw < g.nissue) {
                    tc_fence_after();
                    const uint64_t toff = (uint64_t)((p0 * PS) >> 4);
                    const uint64_t dW = bdesc0 + toff;
                    const uint64_t dR = tc_smem_desc(smem_u32(sR), (uint32_t)PS, 128u) + toff;
                    const uint64_t dD = tc_smem_desc(smem_u32(sD), (uint32_t)PS, 128u) + toff;
                    for (int ks = wiw; ks < g.ks; ks += 4) {
                        const uint64_t kso = (uint64_t)(ks * ((2 * PS) >> 4));
                        if (wg == 0) {
                            tc_mma_i8_ts(tD, tOnes + (uint32_t)(ks * 8), dW + kso, idesc_h, 1u);
                        } else {
                            tc_mma_i8_ts(tQ, tOnes + (uint32_t)(ks * 8), dR + kso, idesc_h, 1u);
                            tc_mma_i8_ts(tQ, t255 + (uint32_t)(ks * 8), dD + kso, idesc_h, 1u);
                        }
                    }
                    tc_commit(&done_bar[wg]);
                }
                mbar_wait(&done_bar[0], done_phase);
                mbar_wait(&done_bar[1], done_phase);
                done_phase ^= 1u;
                tc_fence_after();
                {   // vertical sliding sums along the lane's TMEM row; each warp group takes half of the output rows
                    const int yh = (RH + 1) / 2, ys = wg * yh, ye = min(RH, ys + yh);
                    const bool emit = xi < RWt && aa == 0;
                    const int x = xbase + xi;
                    if (ys < ye) {
                        uint32_t sum = 0, sq = 0;
                        for (int c0 = 0; c0 < s; c0 += 8) {
                            uint32_t va[8], vb[8];
                            tc_ld8(tD + lane_base + (uint32_t)(ys + c0), va);
                            tc_ld8(tQ + lane_base + (uint32_t)(ys + c0), vb);
                            tc_ld_wait();
#pragma unroll
                            for (int c = 0; c < 8; ++c) if (c0 + c < s) { sum += va[c]; sq += vb[c]; }
                        }
                        if (emit) { wsum[ys * RW + x] = sum; wsq[ys * RW + x] = sq; }
                        for (int c0 = 0; ys + 1 + c0 < ye; c0 += 8) {
                            uint32_t na[8], oa[8], nq[8], oq[8];
                            tc_ld8(tD + lane_base + (uint32_t)(ys + s + c0), na);
                            tc_ld8(tD + lane_base + (uint32_t)(ys + c0), oa);
                            tc_ld8(tQ + lane_base + (uint32_t)(ys + s + c0), nq);
                            tc_ld8(tQ + lane_base + (uint32_t)(ys + c0), oq);
                            tc_ld_wait();
#pragma unroll
                            for (int c = 0; c < 8; ++c) {
                                const int y = ys + 1 + c0 + c;
                                sum += na[c] - oa[c]; sq += nq[c] - oq[c];
                                if (emit && y < ye) { wsum[y * RW + x] = sum; wsq[y * RW + x] = sq; }
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            for (int idx = tid; idx < RR; idx += nt) wden[idx] = window_den(wsum[idx], wsq[idx], a.inv_area);
        } else {
        // ---- 2a. horizontal sliding sums over the template width, every window row
            {
                int seg = PM_SEG;
                while (H * ((RW + seg - 1) / seg) > nt && seg < RW) ++seg;
                const int nseg = (RW + seg - 1) / seg;
                for (int t = tid; t < H * nseg; t += nt) {
                    const int y = t / nseg, xs = (t - y * nseg) * seg;
                    const int xe = min(RW, xs + seg);
                    const unsigned char *rowp = sW + y * 16;
                    auto wb = [&](int k) -> uint32_t { const int kk = k + xoff; return rowp[(kk >> 4) * PS + (kk & 15)]; };
                    uint32_t sum = 0, sq = 0;
                    for (int j = 0; j < s; ++j) { const uint32_t v = wb(xs + j); sum += v; sq += v * v; }
                    for (int x = xs; x < xe; ++x) {
                        hs[y * RW + x] = sum; hq[y * RW + x] = sq;
                        const uint32_t va = wb(x), vb = wb(x + s);
                        sum += vb - va; sq += vb * vb - va * va;
                    }
                }
            }
            __syncthreads();
            // ---- 2b. vertical sliding sums -> window sum and denominator per displacement
            {
                int vseg = PM_VSEG;
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
        }

        // ---- 3. angle batches
        const int A = a.n_angles;
        const int nbatch = (A + nab - 1) / nab;
        const int per = (A + nbatch - 1) / nbatch;
        const int n16 = (RH + 15) & ~15;
        const uint32_t idesc = tc_idesc_u8(n16);
        const int ntile = (RW + g.xt - 1) / g.xt;
        bool has_zero = false;
        for (int a0 = 0; a0 < A; a0 += per) {
            const int nb = min(per, A - a0);
            if (tid < PM_MAX_AB) { S.tsum[tid] = 0; S.tsq[tid] = 0; S.key[tid] = 0ull; }
            if (tid == 0) S.haszero = 0;
            __syncthreads();
            // gather the rotated templates (get_template), four byte-shifted copies of every row
            {
                const int rows_per_pass = nt / s;
                const int gi = tid / s, gj = tid - gi * s;
                const bool active = gi < rows_per_pass;
                const double dj = (double)gj;
                for (int ai = 0; ai < nb; ++ai) {
                    const double *tab = a.tab + 4 * (a0 + ai);
                    const double cs = tab[0], sn = tab[1];
                    const double off0 = __dsub_rn(r1, tab[2]), off1 = __dsub_rn(c1, tab[3]);
                    const bool inside = template_inside_warp(a.rows1, a.cols1, off0, off1, cs, sn, s);
                    const bool fast0 = inside && a.rot_order == 0;
                    const double jsn = __dmul_rn(dj, sn), jcs = __dmul_rn(dj, cs);
                    unsigned char *tdst = sT + (size_t)ai * g.tang + 4 * g.ctlw + gj;
                    uint32_t lsum = 0, lsq = 0; int lzero = 0;
                    // each thread owns column gj and rows gi, gi + rows_per_pass, ...: U rows, four loads in flight at a
                    // time, the remainder one by one (no predicated-off copies of the body).  (Measured: issuing all loads
                    // of the three angles before the first store is slightly SLOWER, 3.76 vs 3.68 ms on cfg2 -- registers.)
                    const int U = (s + rows_per_pass - 1) / rows_per_pass;
                    auto sweep = [&](auto sample) {
                        auto load = [&](int i) -> uint32_t {
                            if (!(active && i < s)) return 1u;
                            const double di = (double)i;
                            const double row = __dadd_rn(__dadd_rn(off0, __dmul_rn(di, cs)), jsn);
                            const double col = __dadd_rn(__dadd_rn(off1, __dmul_rn(di, -sn)), jcs);
                            return sample(row, col);
                        };
                        auto store = [&](int i, uint32_t v) {
                            if (active && i < s) {
                                unsigned char *d = tdst + (size_t)i * 4 * tpw4;
                                const unsigned char b = (unsigned char)v;
                                d[0] = b; d[tpw4 + 1] = b; d[2 * tpw4 + 2] = b; d[3 * tpw4 + 3] = b;
                                lsum += v; lsq += v * v; lzero |= (v == 0);
                            }
                        };
                        int u = 0;
                        for (; u + 4 <= U; u += 4) {
                            uint32_t v[4];
#pragma unroll
                            for (int w = 0; w < 4; ++w) v[w] = load((u + w) * rows_per_pass + gi);
#pragma unroll
                            for (int w = 0; w < 4; ++w) store((u + w) * rows_per_pass + gi, v[w]);
                        }
                        for (; u < U; ++u) store(u * rows_per_pass + gi, load(u * rows_per_pass + gi));
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
            if (tid < nb) {
                S.st[tid] = templ_stats(S.tsum[tid], S.tsq[tid], a.inv_area, a.sqrt_inv_area);
                int slot = tid;
                if (S.best_slot >= 0 && slot >= S.best_slot) ++slot;
                S.slot[tid] = slot;
            }
            __syncthreads();

            // ---- correlation on the tensor cores, one x tile at a time
            const bool my_angle = aa < nb;
            double t_mean = 0.0, t_norm = 0.0;
            int t_flat = 0;
            float *my_map = maps;
            if (my_angle) {
                t_mean = S.st[aa].mean; t_norm = S.st[aa].norm; t_flat = S.st[aa].flat;
                my_map = maps + (size_t)S.slot[aa] * a.max_rr;
            }
            unsigned long long key = 0ull;
            for (int tile = 0; tile < ntile; ++tile) {
                const int xbase = tile * g.xt;
                const int RWt = min(g.xt, RW - xbase);
                const int col0 = xbase + xoff, p0 = col0 >> 4, offt = col0 & 15;
                const bool live = my_angle && xi < RWt;
                const int q = xi + offt;
                const int cw0 = (xi_min + offt) >> 2;            // first K word of this warp's band
                const uint32_t *trow = reinterpret_cast<const uint32_t *>(sT + (size_t)aa * g.tang + (q & 3) * tpw4) +
                                       g.ctlw - (q >> 2) + cw0;
                // every warp is done reading the previous tile's accumulators (tcgen05.ld) before anything is cleared
                tc_fence_before();
                __syncthreads();
                tc_fence_after();
                // clear the accumulators and the A slots: each warp its lane quarter, each warp group half the columns
                {
                    uint32_t z[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) z[c] = 0u;
                    const int ncol = g.nacc * g.n16max + g.nslot * g.slotc, half = ((ncol / 8 + 1) / 2) * 8;
                    const int cb = wg * half, ce = min(ncol, cb + half);
                    for (int c = cb; c < ce; c += 8) tc_st8(tD + lane_base + c, z);
                    tc_st_wait();
                    tc_fence_before();
                }
                __syncthreads();
                tc_fence_after();
                // Row loop.  All index arithmetic is carried in running variables (i advances by 2): slot = i % nslot,
                // bi = i % (2 nslot) (the slot barrier this row commits to), bw = (i - nslot) % (2 nslot) and
                // kidx = (i - nslot) / (2 nslot) (barrier and completion index of the row that used this slot before).
                // Dead lanes read a row of zeros.
                {
                    const bool issuer = lane == 0 && wiw < g.nissue;
                    const uint32_t sbar = smem_u32(&slot_bar[0]);
                    const int row_words = 4 * g.tpw;
                    const uint32_t *p = live ? trow + (size_t)wg * row_words
                                             : reinterpret_cast<const uint32_t *>(sT + (size_t)nab * g.tang);
                    const int pstep = live ? 2 * row_words : 0;
                    // this thread's first MMA of a row (K step wiw); further K steps (ks >= 4) are rare
                    const uint32_t d0 = tD + (uint32_t)((wiw % g.nacc) * g.n16max);
                    const uint64_t b0 = bdesc0 + (uint64_t)((p0 * PS) >> 4) + (uint64_t)(wiw * ((2 * PS) >> 4));
                    const int nsl = g.nslot, per = 2 * g.nslot;
                    int slot = wg % nsl, bi = wg, bw = wg + nsl, kidx = -1;   // state for i = wg (bw, kidx describe row i - nslot)
                    if (g.nb8 == 2) {
                        // common case: 16 band words per row, held in registers one row ahead (the next row's shared-
                        // memory loads are in flight while this row's TMEM stores complete)
                        uint32_t v[16];
#pragma unroll
                        for (int c = 0; c < 16; ++c) v[c] = p[c];
                        for (int i = wg; i < s; i += 2) {
                            if (i >= nsl) {                      // MMAs of row i - nslot (same slot) done?
                                mbar_wait_addr(sbar + 8u * (uint32_t)bw, ((slot_par >> bw) + (unsigned)kidx) & 1u);
                                tc_fence_after();
                            }
                            const uint32_t ta = tA + lane_base + (uint32_t)(slot * g.slotc + cw0);
                            {
                                const uint32_t (&lo)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&v[0]);
                                const uint32_t (&hi)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&v[8]);
                                tc_st8(ta, lo);
                                tc_st8(ta + 8, hi);
                            }
                            p += pstep;
                            if (i + 2 < s) {
#pragma unroll
                                for (int c = 0; c < 16; ++c) v[c] = p[c];
                            }
                            tc_st_wait();
                            tc_fence_before();
                            bar_sync_group(wg);
                            if (issuer) {
                                tc_fence_after();
                                const uint32_t a0 = tA + (uint32_t)(slot * g.slotc);
                                tc_mma_i8_ts(d0, a0 + (uint32_t)(wiw * 8), b0 + (uint64_t)i, idesc, 1u);
                                for (int ks = wiw + 4; ks < g.ks; ks += 4)
                                    tc_mma_i8_ts(tD + (uint32_t)((ks % g.nacc) * g.n16max), a0 + (uint32_t)(ks * 8),
                                                 b0 + (uint64_t)(i + (ks - wiw) * ((2 * PS) >> 4)), idesc, 1u);
                                tc_commit_addr(sbar + 8u * (uint32_t)bi);
                            }
                            slot += 2; if (slot >= nsl) slot -= nsl;     // (slot + 2) % nslot
                            bi += 2; if (bi >= per) bi -= per;
                            bw += 2; if (bw >= per) { bw -= per; ++kidx; }
                        }
                    } else {
                    for (int i = wg; i < s; i += 2) {
                        if (i >= nsl) {                          // MMAs of row i - nslot (same slot) done?
                            mbar_wait_addr(sbar + 8u * (uint32_t)bw, ((slot_par >> bw) + (unsigned)kidx) & 1u);
                            tc_fence_after();
                        }
                        const uint32_t ta = tA + lane_base + (uint32_t)(slot * g.slotc + cw0);
                        for (int grp = 0; grp < g.nb8; ++grp) {
                            uint32_t v[8];
#pragma unroll
                            for (int c = 0; c < 8; ++c) v[c] = p[grp * 8 + c];
                            tc_st8(ta + grp * 8, v);
                        }
                        tc_st_wait();
                        tc_fence_before();
                        bar_sync_group(wg);
                        if (issuer) {
                            tc_fence_after();
                            const uint32_t a0 = tA + (uint32_t)(slot * g.slotc);
                            tc_mma_i8_ts(d0, a0 + (uint32_t)(wiw * 8), b0 + (uint64_t)i, idesc, 1u);
                            for (int ks = wiw + 4; ks < g.ks; ks += 4)
                                tc_mma_i8_ts(tD + (uint32_t)((ks % g.nacc) * g.n16max), a0 + (uint32_t)(ks * 8),
                                             b0 + (uint64_t)(i + (ks - wiw) * ((2 * PS) >> 4)), idesc, 1u);
                            tc_commit_addr(sbar + 8u * (uint32_t)bi);
                        }
                        p += pstep;
                        slot += 2; if (slot >= nsl) slot -= nsl;         // (slot + 2) % nslot
                        bi += 2; if (bi >= per) bi -= per;
                        bw += 2; if (bw >= per) { bw -= per; ++kidx; }
                    }
                    }
                }
                if (lane == 0 && wiw < g.nissue) tc_commit(&done_bar[wg]);
                slot_par ^= g.par_mask;                          // completions this tile added to each slot barrier (host-computed)
                mbar_wait(&done_bar[0], done_phase);
                mbar_wait(&done_bar[1], done_phase);
                done_phase ^= 1u;
                tc_fence_after();

                // epilogue: each warp group takes half of the rows (TMEM columns)
                {
                    const int halfn = n16 / 2;
                    const int x = xbase + xi;
                    float bv = -INFINITY;
                    int bidx = -1;
                    for (int c0 = wg * halfn; c0 < (wg + 1) * halfn; c0 += 8) {
                        if (c0 >= RH) break;
                        uint32_t acc[8];
                        tc_ld8(tD + lane_base + c0, acc);
                        if (g.nacc == 3) {
                            uint32_t v1[8], v2[8];
                            tc_ld8(tD + lane_base + (uint32_t)(g.n16max + c0), v1);
                            tc_ld8(tD + lane_base + (uint32_t)(2 * g.n16max + c0), v2);
                            tc_ld_wait();
#pragma unroll
                            for (int c = 0; c < 8; ++c) acc[c] += v1[c] + v2[c];
                        } else {
                            tc_ld_wait();
                            for (int k = 1; k < g.nacc; ++k) {
                                uint32_t v[8];
                                tc_ld8(tD + lane_base + (uint32_t)(k * g.n16max + c0), v);
                                tc_ld_wait();
#pragma unroll
                                for (int c = 0; c < 8; ++c) acc[c] += v[c];
                            }
                        }
                        if (live) {
#ifdef SID_TC_SERIAL_NCC
#pragma unroll
                            for (int c = 0; c < 8; ++c) {
                                const int y = c0 + c;
                                if (y < RH) {
                                    const int idx = y * RW + x;
                                    float v = 1.0f;
                                    if (!t_flat) {
                                        const double num = __dsub_rn((double)(int)acc[c], __dmul_rn((double)wsum[idx], t_mean));
                                        v = __double2float_rn(ncc_finish(num, __dmul_rn(wden[idx], t_norm)));
                                    }
                                    my_map[idx] = v;
                                    if (v > bv) { bv = v; bidx = idx; }
                                }
                            }
#else
                            // two batches of four outputs: the FP64 chains of a batch are independent and interleave
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                double num[4], tt[4];
                                float v[4];
                                int idx4[4];
#pragma unroll
                                for (int c = 0; c < 4; ++c) {
                                    const int y = min(c0 + 4 * h + c, RH - 1);          // rows past the map repeat the last row (discarded below)
                                    idx4[c] = y * RW + x;
                                    num[c] = __dsub_rn((double)(int)acc[4 * h + c], __dmul_rn((double)wsum[idx4[c]], t_mean));
                                    tt[c] = __dmul_rn(wden[idx4[c]], t_norm);
                                }
                                ncc_finish4(num, tt, v);
#pragma unroll
                                for (int c = 0; c < 4; ++c) {
                                    if (c0 + 4 * h + c < RH) {
                                        const float vv = t_flat ? 1.0f : v[c];
                                        my_map[idx4[c]] = vv;
                                        if (vv > bv) { bv = vv; bidx = idx4[c]; }
                                    }
                                }
                            }
#endif
                        }
                    }
                    if (bidx >= 0) {
                        const unsigned long long k2 = peak_key(bv, (uint32_t)bidx);
                        key = k2 > key ? k2 : key;
                    }
                }
                tc_fence_before();       // TMEM reads are done before the next tile's clears
            }
            for (int a2 = 0; a2 < nb; ++a2) {
                unsigned long long k2 = (aa == a2) ? key : 0ull;
                k2 = warp_max_u64(k2);
                if (lane == 0 && k2) atomicMax(&S.key[a2], k2);
            }
            __syncthreads();
            tc_fence_after();
            if (tid == 0) {
                for (int ai = 0; ai < nb; ++ai) {
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

        // ---- 4. peak statistics and bookkeeping; the window is dead: request the next point's now
        if (tid == 0 && S.nok) {
            mbar_expect_tx(&win_bar, win_tx);
            for (int p = 0; p < g.np_load; ++p) tma_load_2d(sW + p * PS, &tmapP, S.nx0 + 16 * p, S.ny0, &win_bar);
            S.tma_for = S.next;
        }
        const int best_slot = S.best_slot, best_idx = S.best_idx;
        const float *best = maps + (size_t)best_slot * a.max_rr;
        if (a.split_tail) {
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
        float *hes = maps + (size_t)(nab + 1) * a.max_rr;
        float *tmp_b = maps + (size_t)(nab + 2) * a.max_rr;
        // 2048-word histogram for the select of peak_statistics: the (dead) window statistics when the scratch is in shared
        // memory, else 8 KB of static shared memory (large maps: the scratch lives in the L2-resident slab)
        uint32_t *wide_hist = nullptr;
        if constexpr (SMEM_SCRATCH) { if ((size_t)a.max_rr * 8 >= 2048 * 4) wide_hist = reinterpret_cast<uint32_t *>(wden); }
        else { __shared__ __align__(16) uint32_t tail_hist_s[2048]; wide_hist = tail_hist_s; }
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
        if (a.peaks) store_secondary_peaks(a.peaks + 12 * pt, best, hes, RH, RW, best_idx, ps, a.flags, c2, r2, H, W, s, S.bs);
        if (a.tpl_out) pm_store_template(a, pt, S.best_a);
    }
    // a window requested for a work item that never ran (the list ended) must land before the CTA exits
    if (S.tma_for != 0xffffffffu && (long long)S.tma_for >= a.n) { /* never requested past the end: nok == 0 there */ }
    tc_fence_before();
    __syncthreads();
    if (tid < 32) tc_dealloc(tbase, (uint32_t)g.tmem_cols);
}

}  // namespace sid
