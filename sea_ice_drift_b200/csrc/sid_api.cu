// sid_api.cu -- C ABI (include/sid_b200.h) over the sm_100a kernels.
// No exceptions cross the boundary; every entry point returns a SID_* code.
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <new>
#include <string>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include <emmintrin.h>

#include "../../include/sid_b200.h"
#include "sid_common.cuh"
#include "sid_pm_kernel.cuh"
#include "sid_pm_tc_kernel.cuh"
#include "sid_pm_ws_kernel.cuh"
#include "sid_single_kernels.cuh"
#include "sid_knn_kernel.cuh"
#include "sid_defor_kernel.cuh"
#include "sid_fg_kernel.cuh"
#include "sid_downsample_kernel.cuh"
#include "sid_pm_masked_kernel.cuh"
#include "sid_uncert_kernel.cuh"

using namespace sid;

namespace {

constexpr size_t IMG_TAIL_SLACK = 4096;   // bytes readable past the last image row

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool owned = true;      // false: caller-owned memory adopted by sid_adopt_pair_device (never freed / grown here)
};

}  // namespace

// Persistent host threads for the staged upload of pageable images (creating 7 threads per band and image cost ~25 % of a
// band's copy time).  Owned by a context; the workers sleep on a condition variable between jobs.
class HostPool {
public:
    explicit HostPool(int workers) : nworkers_(workers) {
        for (int i = 0; i < workers; ++i) threads_.emplace_back([this, i] { loop(i); });
    }
    ~HostPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; }
        cv_.notify_all();
        for (std::thread &t : threads_) t.join();
    }
    int size() const { return nworkers_ + 1; }                 // the caller works too
    // fn(part) for part = 0 .. size() - 1, in parallel; returns when all parts are done
    void run(const std::function<void(int)> &fn) {
        { std::lock_guard<std::mutex> lk(m_); job_ = &fn; pending_ = nworkers_; ++gen_; }
        cv_.notify_all();
        fn(nworkers_);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
        job_ = nullptr;
    }
private:
    void loop(int id) {
        unsigned seen = 0;
        for (;;) {
            const std::function<void(int)> *job;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || gen_ != seen; });
                if (stop_) return;
                seen = gen_;
                job = job_;
            }
            (*job)(id);
            { std::lock_guard<std::mutex> lk(m_); if (--pending_ == 0) done_.notify_one(); }
        }
    }
    int nworkers_;
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    const std::function<void(int)> *job_ = nullptr;
    unsigned gen_ = 0;
    int pending_ = 0;
    bool stop_ = false;
};

struct sid_ctx {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;      // image upload, overlapped with compute (sid_run_pair)
    cudaStream_t band_stream[2] = {nullptr, nullptr};   // band launches alternate here so their tails overlap
    cudaEvent_t slot_event[3] = {};          // points uploaded, band stream 0 done, band stream 1 done
    cudaEvent_t band_event[17] = {};
    std::string err;
    long long launches = 0;
    // resident image pair (padded pitch, 16-byte multiple)
    DevBuf img1, img2;
    int rows1 = 0, cols1 = 0, rows2 = 0, cols2 = 0;
    long long pitch1 = 0, pitch2 = 0;
    bool have_pair = false;
    // per-call buffers
    DevBuf pts, order, out, status, angles, scratch, counter, misc, tail_maps, tail_recs, epi, fg;
    DevBuf maps, map_off, tpl;               // sid_run_maps: packed maps, their offsets, the templates
    DevBuf cand;                             // SID_MASKED: the candidate rows of the masked pass
    DevBuf peaks;                            // SID_PEAKS: n x SID_N_PEAKS x 4 doubles of the last sid_run* call
    long long peaks_n = -1;                  // its n, or -1 when the last sid_run* call did not set SID_PEAKS
    bool peaks_of_table = false;             // that call was the sid_run / sid_run_pair / sid_run_maps that left `out`
    DevBuf filt;                             // sid_filter_outliers
    DevBuf uncert;                           // SID_UNCERT: n x 3 doubles of the last sid_run* call
    long long uncert_n = -1;                 // its n, or -1 when the last sid_run* call did not set SID_UNCERT
    void *pin = nullptr;
    size_t pin_cap = 0;
    cudaEvent_t k_ev[2] = {};                // bracket the last fused-kernel launch (sid_last_kernel_ms)
    bool k_ev_valid = false;
    const char *k_name = "";
    HostPool *pool = nullptr;                // staged upload of pageable images
    long long table_n = -1;                  // rows of the result table the last sid_run / sid_run_pair left in `out`
    // staged upload of pageable host images (sid_run_pair): pinned double buffer + "slot free again" events
    void *stage = nullptr;
    size_t stage_cap = 0;
    cudaEvent_t stage_event[2] = {};
    void *encode_tiled = nullptr;            // cuTensorMapEncodeTiled, resolved through the runtime (no libcuda link)
    bool encode_tried = false;
};

namespace {

int fail(sid_ctx *c, int code, const std::string &msg) {
    if (c) c->err = msg;
    return code;
}
int cuda_fail(sid_ctx *c, cudaError_t e, const char *what) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    cudaGetLastError();
    return fail(c, SID_ECUDA, buf);
}
#define CU(call)                                                   \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call);   \
    } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-process, per-device property of the kernel (not of a
// context): raise it to the device's opt-in maximum, and re-assert it whenever some other context may have
// changed it -- setting it is cheap and idempotent.
int allow_max_smem(sid_ctx *ctx, const void *kernel) {
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, kernel));
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            ctx->max_smem_optin - (int)fa.sharedSizeBytes));
    return SID_OK;
}

int reserve(sid_ctx *ctx, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap && b.owned) return SID_OK;
    if (b.p && b.owned) cudaFree(b.p);
    b.p = nullptr; b.cap = 0; b.owned = true;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return fail(ctx, SID_ENOMEM, "device allocation failed"); }
    b.cap = want;
    return SID_OK;
}
int reserve_pinned(sid_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->pin_cap) return SID_OK;
    if (ctx->pin) { cudaFreeHost(ctx->pin); ctx->pin = nullptr; ctx->pin_cap = 0; }
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMallocHost(&ctx->pin, want);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(ctx, SID_ENOMEM, "pinned allocation failed"); }
    ctx->pin_cap = want;
    return SID_OK;
}

long long padded_pitch(int cols) { return ((long long)cols + 15) / 16 * 16 + 16; }

int upload_image(sid_ctx *ctx, DevBuf &buf, long long &pitch, const uint8_t *src, int rows, int cols,
                 long long src_pitch, cudaMemcpyKind kind) {
    if (!src || rows <= 0 || cols <= 0 || src_pitch < cols) return fail(ctx, SID_EINVAL, "bad image arguments");
    pitch = padded_pitch(cols);
    const size_t bytes = (size_t)pitch * rows + IMG_TAIL_SLACK;
    const bool fresh = bytes > buf.cap || !buf.owned;
    int rc = reserve(ctx, buf, bytes);
    if (rc) return rc;
    if (fresh) CU(cudaMemsetAsync(buf.p, 0, buf.cap, ctx->stream));
    CU(cudaMemcpy2DAsync(buf.p, (size_t)pitch, src, (size_t)src_pitch, (size_t)cols, (size_t)rows, kind, ctx->stream));
    return SID_OK;
}

void gaussian_weights(double gw[5]) {
    double w[9], sum = 0.0;
    for (int k = -4; k <= 4; ++k) { w[k + 4] = std::exp(-0.5 * (double)(k * k)); sum += w[k + 4]; }
    for (int k = 0; k < 9; ++k) w[k] /= sum;
    for (int k = 0; k <= 4; ++k) gw[k] = w[4 + k];
}

int check_common(sid_ctx *ctx, int img_size, int n_angles, const double *angle_tab, int rot_order, int mtype) {
    if (!ctx) return SID_EINVAL;
    if (img_size < 2 || img_size > 128) return fail(ctx, SID_EUNSUPPORTED, "img_size must be in [2, 128]");
    if (n_angles <= 0 || !angle_tab) return fail(ctx, SID_EINVAL, "need at least one angle and its table");
    if (rot_order != 0 && rot_order != 1)
        return fail(ctx, SID_EUNSUPPORTED, "rot_order must be 0 or 1 (higher spline orders need a full-image prefilter)");
    if (mtype != SID_TM_CCOEFF_NORMED) return fail(ctx, SID_EUNSUPPORTED, "only TM_CCOEFF_NORMED (5) is implemented");
    return SID_OK;
}

// SID_UNCERT propagates through the sub-pixel estimator, so it needs SID_SUBPIXEL
int check_uncert(sid_ctx *ctx, unsigned flags) {
    if ((flags & SID_UNCERT) && !(flags & SID_SUBPIXEL)) return fail(ctx, SID_EINVAL, "SID_UNCERT needs SID_SUBPIXEL");
    return SID_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// uint8 2-D tensor map over image 2 with a box of box_w x box_h bytes (TMA window staging).
bool make_window_tensor_map(sid_ctx *ctx, CUtensorMap *map, int box_w, int box_h, int which = 2) {
    if (!ctx->encode_tried) {
        ctx->encode_tried = true;
        cudaDriverEntryPointQueryResult q;
        void *fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            ctx->encode_tiled = fn;
        else
            cudaGetLastError();
    }
    const long long pitch = which == 1 ? ctx->pitch1 : ctx->pitch2;
    if (!ctx->encode_tiled || box_w > 256 || box_h > 256 || (box_w & 15) || (pitch & 15)) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)(which == 1 ? ctx->cols1 : ctx->cols2), (cuuint64_t)(which == 1 ? ctx->rows1 : ctx->rows2)};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch};
    const cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = ((EncodeTiledFn)ctx->encode_tiled)(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, which == 1 ? ctx->img1.p : ctx->img2.p, gdim, gstride, box,
                                                         estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// ------------------------------------------------------------------ matching launches: plan, reserve, enqueue
// Largest shared-memory footprint of pm_tail_kernel for which the tail is split off the correlation kernel: at least 4 tail
// CTAs per SM; larger maps measured faster with the fused tail (cfg1: 1.10 vs 1.21 ms)
constexpr size_t TAIL_SPLIT_SMEM = 52 * 1024;

bool split_tail_fits(int max_rr, bool smth) {
    if (const char *e = getenv("SID_PM_SPLIT_TAIL")) if (e[0] == '0') return false;
    return pm_tail_smem_bytes(max_rr, smth) <= TAIL_SPLIT_SMEM;
}

// SID_PM_PATH: unset = pm_ws_kernel where it fits, else pm_tc_kernel where two CTAs per SM fit, else mma.sync; "ws", "tc"
// and "imma" force one of them where it fits (mma.sync otherwise), "dp4a" the integer-pipe kernel
bool ws_wanted() {
    const char *e = getenv("SID_PM_PATH");
    return !e || strcmp(e, "ws") == 0;
}

// pm_ws_kernel's shared-memory layout for borders up to `border` (typical map width rtyp, nstat sets of window statistics)
// fits one CTA with `headroom` bytes to spare: the one rule the planner and ws_border_limit share
bool ws_fits(const sid_ctx *ctx, int s, int border, int n_angles, int rtyp, int nstat, PmWsCfg &g, size_t headroom = 0) {
    const int Wmax = 2 * (s / 2) + 2 * border + 1, Rmax = Wmax - s + 1;
    return pm_ws_geometry(s, Rmax, Wmax, n_angles, Rmax * Rmax, g, rtyp, nstat) &&
           (size_t)g.smem_bytes + 2048 + headroom <= (size_t)ctx->max_smem_optin;
}

enum PmKernel { PM_WS, PM_TC, PM_POINTS, PM_MASKED, PM_UNCERT };
// What a launch is for: the correlation of a border class, the masked pass of SID_MASKED, the uncertainty pass of
// SID_UNCERT
enum PmPass { PASS_MATCH, PASS_MASKED, PASS_UNCERT };

// Everything a matching launch needs that does not depend on which points it takes: the kernel and its variant, its
// configuration and tensor maps, the geometry fields of PmArgs, the CTA shape and that of the split tail
struct PmPlan {
    PmKernel kernel;
    const void *kfn;
    const char *name;                // sid_last_kernel_name
    int kidx;                        // PM_TC / PM_POINTS: 8 + smem_scratch, or the index in the pm_points_kernel table
    bool smem_scratch;               // PM_TC / PM_POINTS: per-point scratch in shared memory (else a global slab per CTA)
    PmWsCfg wg;
    PmTcCfg tg;
    alignas(64) CUtensorMap tmap;    // image 2: the search windows
    alignas(64) CUtensorMap tmap1;   // image 1 (PM_WS): the patch the templates of a point are sampled from
    PmArgs args;                     // geometry only; the launch sets the pointers and the point count
    size_t smem;
    int threads, occ, occ_api;       // occ_api: what the occupancy API answered (SID_DEBUG)
    int tail_threads;
    size_t tail_smem;
};

// Kernel, variant and shape of a launch over points with borders up to max_border (typ_border: the typical point, which
// sizes the CTA and pads pm_ws_kernel's layout).  PASS_MASKED: the masked pass of SID_MASKED (pm_masked_kernel, any
// border, its own tail); PASS_UNCERT: the uncertainty pass of SID_UNCERT (uncert_kernel, every row of the call, after
// every other launch).  Host queries only: nothing is allocated or enqueued.
int plan_pm(sid_ctx *ctx, int s, int n_angles, unsigned flags, int max_border, int typ_border, PmPlan &p,
            PmPass pass = PASS_MATCH) {
    p = PmPlan{};
    const int hws = s / 2;
    const int Wmax = 2 * hws + 2 * max_border + 1;
    const int Rmax = Wmax - s + 1;
    if (Rmax < 2) return fail(ctx, SID_EINVAL, "search window not larger than the template");
    PmArgs &a = p.args;
    a.s = s; a.n_angles = n_angles; a.flags = flags;
    const double area = (double)s * (double)s;
    a.inv_area = 1.0 / area;
    a.sqrt_inv_area = std::sqrt(a.inv_area);
    gaussian_weights(a.gw);
    a.max_rr = Rmax * Rmax;
    a.max_hrw = Wmax * Rmax;
    if (pass == PASS_UNCERT) {
        p.kernel = PM_UNCERT;
        p.kfn = (const void *)uncert_kernel;
        p.name = "sid::uncert_kernel";
        p.threads = UNC_THREADS;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p.occ, p.kfn, p.threads, 0));
        if (p.occ < 1) return fail(ctx, SID_ECUDA, "uncert_kernel does not fit on an SM");
        p.occ_api = p.occ;
        return SID_OK;
    }
    if (pass == PASS_MASKED) {
        p.kernel = PM_MASKED;
        p.kfn = (flags & SID_PEAKS) ? (const void *)pm_masked_kernel<true> : (const void *)pm_masked_kernel<false>;
        p.name = "sid::pm_masked_kernel";
        p.threads = PM_MASKED_THREADS;
        a.scratch_per_cta = pm_masked_scratch_bytes(a.max_rr);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p.occ, p.kfn, p.threads, 0));
        if (p.occ < 1) return fail(ctx, SID_ECUDA, "pm_masked_kernel does not fit on an SM");
        p.occ_api = p.occ;
        return SID_OK;
    }
    // correlation path: tcgen05 tensor cores (default), legacy mma.sync (SID_PM_PATH=imma) or the integer pipe
    // (SID_PM_PATH=dp4a); all three give bit-identical results
    const char *path_env = getenv("SID_PM_PATH");
    const bool want_tc = !path_env || strcmp(path_env, "tc") == 0;
    const bool imma = !(path_env && strcmp(path_env, "dp4a") == 0);
    const bool smth = (flags & SID_HES_SMTH) != 0;
    const bool global_scratch = getenv("SID_PM_GLOBAL_SCRATCH") != nullptr;
    // Split tail: peak statistics in a second, light kernel when the result map fits its shared memory
    const bool split_tail = split_tail_fits(a.max_rr, smth);
    a.split_tail = split_tail ? 1 : 0;
    if (split_tail) a.tail_stride = (a.max_rr + 3) & ~3;
    p.tail_threads = pm_tail_threads(a.max_rr);
    p.tail_smem = pm_tail_smem_bytes(a.max_rr, smth);
    if (split_tail)
        if (int arc = allow_max_smem(ctx, (flags & SID_PEAKS) ? (const void *)pm_tail_kernel<true> : (const void *)pm_tail_kernel<false>))
            return arc;
    // warp-specialised pipeline kernel (sid_pm_ws_kernel.cuh): small result maps (geometry: radius <= 24; its shared-memory
    // layout fits 227 KB up to radius 20 at s = 35, 22 with two sets of window statistics), needs the split tail
    if (ws_wanted() && split_tail) {
        // three sets of window statistics where they fit the shared memory, else two (radius 21 ... 22 at img_size 35)
        const int rtyp = 2 * typ_border + (Wmax - 2 * max_border) - s + 1;
        bool fits = false;
        for (int nstat = WS_NSTAT; nstat >= 2 && !fits; --nstat) fits = ws_fits(ctx, s, max_border, n_angles, rtyp, nstat, p.wg);
        if (fits && make_window_tensor_map(ctx, &p.tmap, 16, p.wg.load_rows) && make_window_tensor_map(ctx, &p.tmap1, p.wg.pbw, p.wg.pbh, 1)) {
            p.kernel = PM_WS;
            p.kfn = (const void *)pm_ws_kernel;
            p.name = "sid::pm_ws_kernel";
            a.tma = 1; a.ab = p.wg.nab;
            p.smem = (size_t)p.wg.smem_bytes;
            p.threads = WS_THREADS;
            p.occ = 1;
            return allow_max_smem(ctx, p.kfn);
        }
    }
    bool use_tc = want_tc && pm_tc_geometry(s, Rmax, Wmax, n_angles, p.tg) && make_window_tensor_map(ctx, &p.tmap, 16, p.tg.load_rows);
    PmTcCfg &tg = p.tg;
    // Measured (profiles/r02_ab_tc_vs_imma.txt): with one CTA per SM (tensor memory > 256 columns: search radius ~100) the
    // latency-bound non-MAC phases make the tcgen05 kernel slower than the mma.sync kernel at three CTAs per SM, so the
    // default takes it only where two CTAs fit; SID_PM_PATH=tc forces it.
    if (use_tc && !path_env && tg.tmem_cols > 256) use_tc = false;
    int variant = 0;
    if (use_tc) {
        // window panels + four byte-shifted copies of the template rows (+ the per-point scratch when two CTAs
        // still fit on an SM)
        a.tma = 1;
        a.ab = tg.nab;
        const size_t base = (size_t)tg.win_bytes + (size_t)tg.tpl_bytes;
        const size_t scratch = pm_scratch_bytes(a.max_rr, a.max_hrw, a.ab, smth, split_tail);
        const size_t wsq_bytes = ((size_t)a.max_rr * 4 + 255) & ~(size_t)255;
        const size_t need = base + scratch + wsq_bytes;
        const size_t cap2 = 108 * 1024;
        if (need <= cap2 && !global_scratch) { p.smem_scratch = true; p.smem = need; }
        else p.smem = base;
        // window sums on the tensor cores: the two squares windows alias the result maps (dead until the first
        // epilogue), two accumulators of n16hmax columns + two A slots must fit the tensor-memory allocation
        if (p.smem_scratch) {
            const size_t maps_off = ((size_t)a.max_rr * 12 + 127) & ~(size_t)127;
            const size_t sq_bytes = 2 * (size_t)tg.npanels * (size_t)tg.wrows * 16;
            const bool fits_smem = maps_off + sq_bytes <= scratch;
            const bool fits_tmem = 2 * tg.n16hmax + 8 <= tg.nacc * tg.n16max + (tg.nslot - 2) * tg.slotc && tg.n16hmax <= tg.wrows;
            if (fits_smem && fits_tmem) {
                tg.mma_sums = 1; tg.sq_off = (int)maps_off; tg.wsq_off = (int)scratch;
            }
        }
        if (p.smem > (size_t)ctx->max_smem_optin - 4096 - (p.smem_scratch ? 0 : 8192)) use_tc = false;      // window too large: legacy kernels
                                                                          // (the global-scratch variant has 8 KB more static shared memory)
    }
    // [8 ... 15]: the same kernels with SID_PEAKS
    const void *ktab[16] = {(const void *)pm_points_kernel<9, false, false, false>, (const void *)pm_points_kernel<13, false, false, false>,
                            (const void *)pm_points_kernel<0, false, false, false>, (const void *)pm_points_kernel<9, true, false, false>,
                            (const void *)pm_points_kernel<13, true, false, false>, (const void *)pm_points_kernel<0, true, false, false>,
                            (const void *)pm_points_kernel<0, false, true, false>, (const void *)pm_points_kernel<0, true, true, false>,
                            (const void *)pm_points_kernel<9, false, false, true>, (const void *)pm_points_kernel<13, false, false, true>,
                            (const void *)pm_points_kernel<0, false, false, true>, (const void *)pm_points_kernel<9, true, false, true>,
                            (const void *)pm_points_kernel<13, true, false, true>, (const void *)pm_points_kernel<0, true, false, true>,
                            (const void *)pm_points_kernel<0, false, true, true>, (const void *)pm_points_kernel<0, true, true, true>};
    const int kpeaks = (flags & SID_PEAKS) ? 8 : 0;
    // the legacy kernel of this launch in ktab: mma.sync (imma) or a dp4a specialisation, per-point scratch in shared or global memory
    auto legacy_kidx = [&](bool smem_scr) { return imma ? (smem_scr ? 7 : 6) : variant + (smem_scr ? 3 : 0); };
    if (!use_tc) {
    // window staging by TMA when the padded window (+15 bytes: the box must start 16-byte aligned) fits one
    // box of <= 256 x 256 bytes
    memset(&p.tmap, 0, sizeof p.tmap);
    a.tma = 0;
    int wpw = pm_window_pitch_words(Wmax, imma);
    {
        const char *e = getenv("SID_PM_TMA");
        const int wpw_tma = pm_window_pitch_words(Wmax + 15, imma);
        if (!(e && e[0] == '0') && make_window_tensor_map(ctx, &p.tmap, wpw_tma * 4, Wmax)) {
            a.tma = 1; a.tma_wpw = wpw_tma; a.tma_rows = Wmax;
            wpw = wpw_tma;
        }
    }
    a.win_words = (Wmax + (imma ? PM_IMMA_ROW_SLACK : 0)) * wpw + PM_WIN_SLACK;
    const int nw = (s + 3) / 4;
    if (nw == 9) variant = 0; else if (nw == 13) variant = 1; else variant = 2;   // dp4a kernel specialisation by template width in words
    if (imma) {
        a.nc = (s + 7 + 31) / 32;
        a.tpw = (32 * a.nc + 16) / 4;
        a.tpl_off = 8;
        a.ab = std::min(n_angles, PM_IMMA_AB);
    } else {
        a.nc = 0;
        a.tpw = variant == 2 ? (s + 15) / 16 * 4 : (nw + 3) / 4 * 4;
        a.tpl_off = 0;
        a.ab = std::min(n_angles, PM_MAX_AB);
    }
    // Shared memory: window + templates (+ the per-point scratch when it all fits in a third of an SM).
    const size_t smem_cap_fast = 75 * 1024;
    auto base_smem = [&](int ab) { return ((size_t)a.win_words + (size_t)ab * s * a.tpw) * 4; };
    for (int ab = a.ab; ab >= 1 && !p.smem_scratch; --ab) {
        const size_t need = base_smem(ab) + pm_scratch_bytes(a.max_rr, a.max_hrw, ab, smth, split_tail);
        // fewer resident templates only pays if it keeps all angles in <= the same number of batches
        if (need <= smem_cap_fast && (n_angles + ab - 1) / ab == (n_angles + a.ab - 1) / a.ab) {
            p.smem_scratch = true; a.ab = ab; p.smem = need;
        }
    }
    if (global_scratch) p.smem_scratch = false;
    if (!p.smem_scratch) {
        // the kernel's static shared memory (PmShared, the window barrier: 1920 B as cudaFuncGetAttributes reports it) comes
        // out of the same per-block budget.  Without it a window that left less than that free was neither given fewer
        // angles per batch nor refused here, and failed the occupancy check below with SID_ECUDA instead (measured on a
        // B200: img_size 35, 3 angles, borders 206, 207, 209 and 210; img_size 128, 3 angles, borders 124 and 125)
        cudaFuncAttributes fa;
        CU(cudaFuncGetAttributes(&fa, ktab[kpeaks + legacy_kidx(false)]));
        const size_t smem_max = (size_t)ctx->max_smem_optin - fa.sharedSizeBytes;
        p.smem = base_smem(a.ab);
        while (p.smem > smem_max && a.ab > 1) { --a.ab; p.smem = base_smem(a.ab); }
        if (p.smem > smem_max) {
            if (getenv("SID_DEBUG"))
                fprintf(stderr, "[sid] refuse: legacy smem=%zu limit=%zu static=%zu optin=%d\n", p.smem, smem_max,
                        (size_t)fa.sharedSizeBytes, ctx->max_smem_optin);
            return fail(ctx, SID_EUNSUPPORTED, "search window too large for the fused kernel (border too big)");
        }
    }
    }

    // CTA size: fill the CTA with thread tiles (dp4a) / warp tiles (IMMA) of a typical point
    const int Rt = 2 * typ_border + (Wmax - 2 * max_border) - s + 1;
    p.threads = PM_THREADS;
    if (use_tc) {
        p.threads = TC_THREADS;
    } else if (imma) {
        const int warp_tiles = ((Rt + 15) / 16) * ((Rt + 23) / 24);
        double best_eff = -1.0;
        for (int w = 4; w <= PM_IMMA_THREADS / 32; ++w) {
            const double eff = (double)warp_tiles / (double)((warp_tiles + w - 1) / w * w);
            if (eff >= best_eff - 1e-9) { best_eff = eff; p.threads = 32 * w; }
        }
    } else {
        const int tx = pm_pick_tx(Rt);
        const int ncg = (((Rt + 3) >> 2) + tx - 1) / tx;
        const int nbatch = (n_angles + a.ab - 1) / a.ab;
        const int per = (n_angles + nbatch - 1) / nbatch;
        const long long ntiles = (long long)per * ncg * Rt * 4;
        double best_eff = -1.0;
        for (int bs = 128; bs <= PM_THREADS; bs += 32) {
            const double eff = (double)ntiles / (double)((ntiles + bs - 1) / bs * bs);
            if (eff >= best_eff - 1e-9) { best_eff = eff; p.threads = bs; }
        }
    }

    p.kidx = use_tc ? (p.smem_scratch ? 9 : 8) : legacy_kidx(p.smem_scratch);
    p.kfn = use_tc ? (p.smem_scratch ? (const void *)pm_tc_kernel<true> : (const void *)pm_tc_kernel<false>) : ktab[kpeaks + p.kidx];
    if (int arc = allow_max_smem(ctx, p.kfn)) return arc;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p.occ, p.kfn, p.threads, p.smem));
    if (p.occ < 1) {
        char msg[256];
        snprintf(msg, sizeof msg, "kernel does not fit on an SM (variant %d, %d threads, %zu B dynamic smem, img_size %d, max border %d, "
                 "%d angles/batch, tma %d)", p.kidx, p.threads, p.smem, s, max_border, a.ab, a.tma);
        return fail(ctx, SID_ECUDA, msg);
    }
    p.occ_api = p.occ;
    if (use_tc) {
        // The occupancy API answers 1 for a kernel that executes tcgen05.alloc with a run-time column count (it has to
        // assume all 512 columns); residency is really bounded by registers, shared memory and the columns we ask for.
        cudaFuncAttributes fa;
        CU(cudaFuncGetAttributes(&fa, p.kfn));
        int smem_sm = 0, regs_sm = 0;
        CU(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, ctx->device));
        CU(cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, ctx->device));
        const int by_smem = (int)((size_t)smem_sm / (p.smem + fa.sharedSizeBytes + 1024));
        const int by_regs = regs_sm / std::max(1, fa.numRegs * p.threads);
        p.occ = std::max(1, std::min(std::min(by_smem, by_regs), 512 / tg.tmem_cols));
    }
    a.scratch_per_cta = pm_scratch_bytes(a.max_rr, a.max_hrw, a.ab, smth, split_tail);
    p.kernel = use_tc ? PM_TC : PM_POINTS;
    p.name = use_tc ? "sid::pm_tc_kernel" : imma ? "sid::pm_points_kernel<imma>" : "sid::pm_points_kernel<dp4a>";
    return SID_OK;
}

// What every matching launch of one sid_run / sid_run_pair / sid_run_device / sid_run_maps call shares
struct PmCall {
    const double *c1, *r1, *c2fg, *r2fg, *border;     // device point arrays
    const double *angles, *tab;                        // device angle table
    int rot_order;
    double *out;
    int *status;
    float *maps_out;                 // sid_run_maps only (null otherwise), see PmArgs::maps_out
    const long long *map_off;
    uint8_t *tpl_out;
    long long n;                     // points of the call: the tail hand-off regions are laid out for all of them
    int *cand;                       // set by reserve_call for a masked pass: its candidate rows (n) and their count
    // set by reserve_call
    size_t tail_stride;              // floats per point of the tail hand-off regions
    size_t scratch_slot;             // bytes of global scratch per band stream
    double *peaks = nullptr;         // SID_PEAKS only, see PmArgs::peaks
    double *uncert = nullptr;        // set by reserve_call for an uncertainty pass: n x 3 doubles (uncert_kernel)
};

// The buffers the launches of a call share, reserved once before the first launch, so that none of them is reallocated
// while a launch of the call is in flight.  Launches of different bands run concurrently on two streams: the tail hand-off
// regions of all of them are laid out with ONE stride, and each stream has its own scratch slot and work counter.
int reserve_call(sid_ctx *ctx, PmCall &call, const PmPlan *plans, int nplans) {
    call.tail_stride = 0;
    call.scratch_slot = 0;
    bool masked = false, uncert = false;
    for (int i = 0; i < nplans; ++i) {
        const PmPlan &p = plans[i];
        if (p.kernel == PM_UNCERT) uncert = true;
        // a work item of pm_ws_kernel hands over three integer arrays (PmTailRec::mode 1), the others a float map
        if (p.args.split_tail) call.tail_stride = std::max(call.tail_stride, tail_item_words(p.args.tail_stride, p.kernel == PM_WS));
        if (p.kernel == PM_MASKED) masked = true;
        if (p.kernel != PM_WS && !p.smem_scratch)
            call.scratch_slot = std::max(call.scratch_slot, (size_t)p.args.scratch_per_cta * (size_t)ctx->sm_count * (size_t)p.occ);
#ifdef SID_WS_PROF
        if (p.kernel == PM_WS) call.scratch_slot = std::max(call.scratch_slot, (size_t)ctx->sm_count * 6 * 8 * 8);
#endif
    }
    int rc = reserve(ctx, ctx->counter, 256);
    if (rc) return rc;
    if (call.scratch_slot && (rc = reserve(ctx, ctx->scratch, call.scratch_slot * 2))) return rc;
    if (call.tail_stride) {
        if ((rc = reserve(ctx, ctx->tail_maps, (size_t)call.n * call.tail_stride * sizeof(float)))) return rc;
        if ((rc = reserve(ctx, ctx->tail_recs, (size_t)call.n * sizeof(PmTailRec)))) return rc;
    }
    if (masked || uncert) {
        // the masked and uncertainty passes find their rows by their status: a call without a status array gets the
        // context's
        if (!call.status) {
            if ((rc = reserve(ctx, ctx->status, (size_t)call.n * sizeof(int)))) return rc;
            call.status = (int *)ctx->status.p;
        }
    }
    if (masked) {
        if ((rc = reserve(ctx, ctx->cand, (size_t)call.n * sizeof(int)))) return rc;
        call.cand = (int *)ctx->cand.p;
    }
    if (uncert) {                    // the pass writes every row's record: no fill needed
        if ((rc = reserve(ctx, ctx->uncert, (size_t)call.n * 3 * sizeof(double)))) return rc;
        call.uncert = (double *)ctx->uncert.p;
    }
    return SID_OK;
}

// Enqueue one launch of a plan (and its split tail) on the buffers reserve_call reserved: points order[0 .. n) (null:
// points 0 .. n - 1), their tail hand-off at point offset tail_off of the call's regions; `slot` picks the counter and
// scratch of one of the two band streams.  `continues`: the second class of a two-class call, or the masked pass, so the
// kernel-time events bracket every launch of the call.  The masked pass (PM_MASKED) runs after every other launch of the
// call: it gathers the rows they left with status 0 on the device (masked_candidates_kernel) and takes those.  The
// uncertainty pass (PM_UNCERT) runs after the masked pass, over all n rows of the call.
int enqueue_pm(sid_ctx *ctx, const PmCall &call, const PmPlan &p, long long n, const int *order, cudaStream_t st, int slot,
               long long tail_off, bool continues) {
    PmArgs a = p.args;
    a.img1 = (const uint8_t *)ctx->img1.p; a.rows1 = ctx->rows1; a.cols1 = ctx->cols1; a.pitch1 = ctx->pitch1;
    a.img2 = (const uint8_t *)ctx->img2.p; a.rows2 = ctx->rows2; a.cols2 = ctx->cols2; a.pitch2 = ctx->pitch2;
    a.n = n;
    a.c1 = call.c1; a.r1 = call.r1; a.c2fg = call.c2fg; a.r2fg = call.r2fg; a.border = call.border; a.order = order;
    a.angles = call.angles; a.tab = call.tab; a.rot_order = call.rot_order;
    a.out = call.out; a.status = call.status;
    a.maps_out = call.maps_out; a.map_off = call.map_off; a.tpl_out = call.tpl_out;
    a.peaks = call.peaks;
    a.counter = (unsigned int *)ctx->counter.p + 16 * slot;
    a.scratch = (unsigned char *)ctx->scratch.p + call.scratch_slot * (size_t)slot;      // read by the global-scratch variants only
    if (a.split_tail) {
        a.tail_maps = (float *)ctx->tail_maps.p + (size_t)tail_off * call.tail_stride;
        a.tail_recs = (PmTailRec *)ctx->tail_recs.p + tail_off;
    }
    const long long grid = std::max(1LL, std::min((long long)ctx->sm_count * p.occ, n));
    CU(cudaMemsetAsync(a.counter, 0, sizeof(unsigned int), st));
    unsigned *n_cand = (unsigned *)ctx->counter.p + 32;
    if (p.kernel == PM_MASKED) {
        a.order = call.cand;
        CU(cudaMemsetAsync(n_cand, 0, sizeof(unsigned), st));
        masked_candidates_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(call.status, n, call.cand, n_cand);
        ctx->launches += 1;
        CU(cudaGetLastError());
    }
    const bool debug = getenv("SID_DEBUG") != nullptr;
    const PmWsCfg &wg = p.wg;
    const PmTcCfg &tg = p.tg;
    if (debug && p.kernel == PM_UNCERT)
        fprintf(stderr, "[sid] launch: uncert threads=%d occ=%d grid=%lld\n", p.threads, p.occ, grid);
    else if (debug && p.kernel == PM_MASKED)
        fprintf(stderr, "[sid] launch: masked threads=%d occ=%d scratch=%llu grid=%lld\n", p.threads, p.occ, a.scratch_per_cta, grid);
    else if (debug && p.kernel == PM_WS)
        fprintf(stderr, "[sid] launch: ws smem=%d nstat=%d nab=%d ks=%d npairs=%d nslots=%d slot_bytes=%d npanels=%d wrows=%d n16max=%d grid=%lld\n",
                wg.smem_bytes, wg.nstat, wg.nab, wg.ks, wg.npairs, wg.nslots, wg.slot_bytes, wg.npanels, wg.wrows, wg.n16max, grid);
    else if (debug)
        fprintf(stderr, "[sid] launch: tc=%d kidx=%d threads=%d smem=%zu occ(api)=%d tmem_cols=%d nab=%d ks=%d nacc=%d nb8=%d slotc=%d nslot=%d n16max=%d wrows=%d npanels=%d mma_sums=%d tma=%d nc=%d\n",
                (int)(p.kernel == PM_TC), p.kidx, p.threads, p.smem, p.occ_api, tg.tmem_cols, tg.nab, tg.ks, tg.nacc, tg.nb8, tg.slotc, tg.nslot,
                tg.n16max, tg.wrows, tg.npanels, tg.mma_sums, a.tma, a.nc);
#ifdef SID_WS_PROF
    if (p.kernel == PM_WS) CU(cudaMemsetAsync(a.scratch, 0, (size_t)grid * 6 * 8 * 8, st));
#endif
    void *params_ws[] = {(void *)&a, (void *)&p.wg, (void *)&p.tmap, (void *)&p.tmap1};
    void *params_tc[] = {(void *)&a, (void *)&p.tg, (void *)&p.tmap};
    void *params_points[] = {(void *)&a, (void *)&p.tmap};
    void *params_masked[] = {(void *)&a, (void *)&n_cand};
    void *params_uncert[] = {(void *)&a, (void *)&call.uncert};
    void **params = p.kernel == PM_WS ? params_ws : p.kernel == PM_TC ? params_tc : p.kernel == PM_MASKED ? params_masked
                    : p.kernel == PM_UNCERT ? params_uncert : params_points;
    if (!ctx->k_ev[0]) { CU(cudaEventCreate(&ctx->k_ev[0])); CU(cudaEventCreate(&ctx->k_ev[1])); }
    if (!continues) CU(cudaEventRecord(ctx->k_ev[0], st));
    CU(cudaLaunchKernel(p.kfn, dim3((unsigned)grid), dim3((unsigned)p.threads), params, p.smem, st));
    CU(cudaEventRecord(ctx->k_ev[1], st));
    ctx->k_ev_valid = true;
    // the masked and uncertainty passes keep the name of the correlation kernel of the call
    ctx->k_name = p.kernel == PM_MASKED || p.kernel == PM_UNCERT ? ctx->k_name
                  : p.kernel != PM_WS || !continues ? p.name
                  : strstr(ctx->k_name, "pm_tc_kernel") ? "sid::pm_tc_kernel + sid::pm_ws_kernel"
                  : strstr(ctx->k_name, "pm_points_kernel") ? "sid::pm_points_kernel + sid::pm_ws_kernel" : p.name;
    ctx->launches += 1;
#ifdef SID_WS_PROF
    if (p.kernel == PM_WS) {             // role profile: cycles per bucket and point, averaged over the CTAs
        std::vector<long long> h((size_t)grid * 48);
        CU(cudaStreamSynchronize(st));
        CU(cudaMemcpy(h.data(), a.scratch, h.size() * 8, cudaMemcpyDeviceToHost));
        static const char *names[6] = {"control", "mma0", "gather0", "stats0", "epi0", "epi1"};
        const double per_pt = (double)n / (double)grid;
        for (int r = 0; r < 6; ++r) {
            fprintf(stderr, "[ws prof] %-8s clk/point:", names[r]);
            for (int k = 0; k < 8; ++k) {
                double sum = 0; for (long long c = 0; c < grid; ++c) sum += (double)h[((size_t)c * 6 + r) * 8 + k];
                fprintf(stderr, " %8.0f", sum / (double)grid / per_pt);
            }
            fprintf(stderr, "\n");
        }
    }
#endif
    if (a.split_tail) {
        if (debug) fprintf(stderr, "[sid] launch: tail threads=%d smem=%zu\n", p.tail_threads, p.tail_smem);
        if (a.peaks) pm_tail_kernel<true><<<(unsigned)n, p.tail_threads, p.tail_smem, st>>>(a);
        else pm_tail_kernel<false><<<(unsigned)n, p.tail_threads, p.tail_smem, st>>>(a);
        ctx->launches += 1;
        CU(cudaGetLastError());
    }
    return SID_OK;
}

}  // namespace

extern "C" {

const char *sid_version(void) { return "sea_ice_drift_b200 0.3 (sm_100a, exact-integer u8 tcgen05 MCC, warp-specialised pipeline)"; }

int sid_create(sid_ctx **out, int device) {
    if (!out) return SID_EINVAL;
    *out = nullptr;
    sid_ctx *ctx = new (std::nothrow) sid_ctx();
    if (!ctx) return SID_ENOMEM;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        cudaGetLastError();
        delete ctx;
        return SID_ECUDA;
    }
    ctx->device = device;
    ctx->stream = ctx->own_stream;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    *out = ctx;
    return SID_OK;
}

void sid_destroy(sid_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *bufs[] = {&ctx->img1, &ctx->img2, &ctx->pts, &ctx->order, &ctx->out, &ctx->status,
                      &ctx->angles, &ctx->scratch, &ctx->counter, &ctx->misc, &ctx->tail_maps, &ctx->tail_recs, &ctx->epi, &ctx->fg,
                      &ctx->maps, &ctx->map_off, &ctx->tpl, &ctx->cand, &ctx->peaks, &ctx->filt, &ctx->uncert};
    for (DevBuf *b : bufs) if (b->p && b->owned) cudaFree(b->p);
    if (ctx->pin) cudaFreeHost(ctx->pin);
    if (ctx->stage) cudaFreeHost(ctx->stage);
    delete ctx->pool;
    for (cudaEvent_t e : ctx->stage_event) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->k_ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->slot_event) if (e) cudaEventDestroy(e);
    for (cudaStream_t st : ctx->band_stream) if (st) cudaStreamDestroy(st);
    if (ctx->copy_stream) {
        cudaStreamDestroy(ctx->copy_stream);
        for (cudaEvent_t e : ctx->band_event) if (e) cudaEventDestroy(e);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char *sid_last_error(const sid_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int sid_set_stream(sid_ctx *ctx, void *cuda_stream) {
    if (!ctx) return SID_EINVAL;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return SID_OK;
}

int sid_synchronize(sid_ctx *ctx) {
    if (!ctx) return SID_EINVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

int64_t sid_launch_count(const sid_ctx *ctx) { return ctx ? ctx->launches : 0; }

const char *sid_last_kernel_name(const sid_ctx *ctx) { return ctx ? ctx->k_name : ""; }

double sid_last_kernel_ms(sid_ctx *ctx) {
    if (!ctx || !ctx->k_ev_valid) return -1.0;
    float ms = 0.f;
    if (cudaEventSynchronize(ctx->k_ev[1]) != cudaSuccess || cudaEventElapsedTime(&ms, ctx->k_ev[0], ctx->k_ev[1]) != cudaSuccess) {
        cudaGetLastError();
        return -1.0;
    }
    return (double)ms;
}

static int set_pair_impl(sid_ctx *ctx, const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                         const uint8_t *img2, int rows2, int cols2, int64_t pitch2, cudaMemcpyKind kind) {
    if (!ctx) return SID_EINVAL;
    CU(cudaSetDevice(ctx->device));
    ctx->have_pair = false;
    int rc = upload_image(ctx, ctx->img1, ctx->pitch1, img1, rows1, cols1, pitch1, kind);
    if (rc) return rc;
    rc = upload_image(ctx, ctx->img2, ctx->pitch2, img2, rows2, cols2, pitch2, kind);
    if (rc) return rc;
    ctx->rows1 = rows1; ctx->cols1 = cols1; ctx->rows2 = rows2; ctx->cols2 = cols2;
    ctx->have_pair = true;
    return SID_OK;
}

int sid_set_pair(sid_ctx *ctx, const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                 const uint8_t *img2, int rows2, int cols2, int64_t pitch2) {
    return set_pair_impl(ctx, img1, rows1, cols1, pitch1, img2, rows2, cols2, pitch2, cudaMemcpyHostToDevice);
}
int sid_set_pair_device(sid_ctx *ctx, const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                        const uint8_t *img2, int rows2, int cols2, int64_t pitch2) {
    return set_pair_impl(ctx, img1, rows1, cols1, pitch1, img2, rows2, cols2, pitch2, cudaMemcpyDeviceToDevice);
}

int sid_pair_layout(int rows, int cols, int64_t *pitch, int64_t *bytes) {
    if (rows <= 0 || cols <= 0 || !pitch || !bytes) return SID_EINVAL;
    *pitch = padded_pitch(cols);
    *bytes = *pitch * (int64_t)rows + (int64_t)IMG_TAIL_SLACK;
    return SID_OK;
}

int sid_adopt_pair_device(sid_ctx *ctx, uint8_t *d_img1, int rows1, int cols1, int64_t pitch1, int64_t bytes1,
                          uint8_t *d_img2, int rows2, int cols2, int64_t pitch2, int64_t bytes2) {
    if (!ctx) return SID_EINVAL;
    if (!d_img1 || !d_img2 || rows1 <= 0 || cols1 <= 0 || rows2 <= 0 || cols2 <= 0)
        return fail(ctx, SID_EINVAL, "bad image arguments");
    if (pitch1 < padded_pitch(cols1) || pitch2 < padded_pitch(cols2) || (pitch1 & 15) || (pitch2 & 15) ||
        ((uintptr_t)d_img1 & 255) || ((uintptr_t)d_img2 & 255))
        return fail(ctx, SID_EINVAL, "adopted images need the layout of sid_pair_layout (pitch, 256-byte aligned base)");
    if (bytes1 < pitch1 * (int64_t)rows1 + (int64_t)IMG_TAIL_SLACK || bytes2 < pitch2 * (int64_t)rows2 + (int64_t)IMG_TAIL_SLACK)
        return fail(ctx, SID_EINVAL, "adopted images need the tail slack of sid_pair_layout");
    CU(cudaSetDevice(ctx->device));
    if (ctx->have_pair && !ctx->img1.owned && !ctx->img2.owned && ctx->img1.p == d_img1 && ctx->img2.p == d_img2 &&
        ctx->rows1 == rows1 && ctx->cols1 == cols1 && ctx->pitch1 == pitch1 && ctx->rows2 == rows2 && ctx->cols2 == cols2 &&
        ctx->pitch2 == pitch2)
        return SID_OK;                                          // the same buffers again (refilled in place by the caller)
    CU(cudaStreamSynchronize(ctx->stream));                    // nothing in flight still reads the old pair
    DevBuf *bufs[2] = {&ctx->img1, &ctx->img2};
    for (DevBuf *b : bufs) { if (b->p && b->owned) cudaFree(b->p); b->p = nullptr; b->cap = 0; }
    ctx->img1.p = d_img1; ctx->img1.cap = (size_t)bytes1; ctx->img1.owned = false;
    ctx->img2.p = d_img2; ctx->img2.cap = (size_t)bytes2; ctx->img2.owned = false;
    ctx->rows1 = rows1; ctx->cols1 = cols1; ctx->pitch1 = pitch1;
    ctx->rows2 = rows2; ctx->cols2 = cols2; ctx->pitch2 = pitch2;
    ctx->have_pair = true;
    return SID_OK;
}

int sid_upload_rows(sid_ctx *ctx, uint8_t *d_dst, int64_t dst_pitch, const uint8_t *src, int64_t src_pitch, int cols, int rows) {
    if (!ctx) return SID_EINVAL;
    if (rows == 0) return SID_OK;
    if (!d_dst || !src || cols <= 0 || rows < 0 || dst_pitch < cols || src_pitch < cols) return fail(ctx, SID_EINVAL, "bad arguments");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpy2DAsync(d_dst, (size_t)dst_pitch, src, (size_t)src_pitch, (size_t)cols, (size_t)rows, cudaMemcpyHostToDevice, ctx->stream));
    return SID_OK;
}

int sid_downsample_pair(sid_ctx *ctx, int factor, uint8_t *d_img1, int64_t pitch1, int64_t bytes1,
                        uint8_t *d_img2, int64_t pitch2, int64_t bytes2) {
    if (!ctx) return SID_EINVAL;
    if (!ctx->have_pair) return fail(ctx, SID_ENOPAIR, "no image pair is resident");
    if (factor < 2 || factor > 16) return fail(ctx, SID_EINVAL, "downsampling factor must be in [2, 16]");
    const int r1 = ctx->rows1 / factor, c1 = ctx->cols1 / factor, r2 = ctx->rows2 / factor, c2 = ctx->cols2 / factor;
    if (r1 < 1 || c1 < 1 || r2 < 1 || c2 < 1) return fail(ctx, SID_EINVAL, "downsampled image smaller than 1 x 1");
    if (!d_img1 || !d_img2 || pitch1 < padded_pitch(c1) || pitch2 < padded_pitch(c2) || (pitch1 & 15) || (pitch2 & 15) ||
        bytes1 < pitch1 * (int64_t)r1 + (int64_t)IMG_TAIL_SLACK || bytes2 < pitch2 * (int64_t)r2 + (int64_t)IMG_TAIL_SLACK)
        return fail(ctx, SID_EINVAL, "output buffers need the layout of sid_pair_layout(rows / factor, cols / factor)");
    CU(cudaSetDevice(ctx->device));
    const DsImage im1{(const uint8_t *)ctx->img1.p, ctx->pitch1, d_img1, (long long)pitch1, r1, c1};
    const DsImage im2{(const uint8_t *)ctx->img2.p, ctx->pitch2, d_img2, (long long)pitch2, r2, c2};
    const int tile = ds_tile_out(factor), rows = ds_rows(factor);
    const dim3 grid((unsigned)((std::max(r1, r2) + rows - 1) / rows), (unsigned)((std::max(c1, c2) + tile - 1) / tile), 2);
    if (grid.y > 65535u) return fail(ctx, SID_EINVAL, "image too wide for sid_downsample_pair");
    switch (factor) {       // one instantiation per factor: the loads and the division by 2 k^2 are unrolled / constant
#define SID_DS_CASE(K) case K: downsample_kernel<K><<<grid, DS_THREADS, 0, ctx->stream>>>(im1, im2); break;
        SID_DS_CASE(2) SID_DS_CASE(3) SID_DS_CASE(4) SID_DS_CASE(5) SID_DS_CASE(6) SID_DS_CASE(7) SID_DS_CASE(8)
        SID_DS_CASE(9) SID_DS_CASE(10) SID_DS_CASE(11) SID_DS_CASE(12) SID_DS_CASE(13) SID_DS_CASE(14) SID_DS_CASE(15)
        SID_DS_CASE(16)
#undef SID_DS_CASE
    }
    ctx->launches += 1;
    CU(cudaGetLastError());
    return SID_OK;
}

static int upload_angles(sid_ctx *ctx, int n_angles, const double *angles, const double *angle_tab,
                         const double **d_angles, const double **d_tab, cudaStream_t st = nullptr) {
    const size_t bytes = (size_t)n_angles * 5 * sizeof(double);
    int rc = reserve(ctx, ctx->angles, bytes);
    if (rc) return rc;
    std::vector<double> h((size_t)n_angles * 5);
    for (int k = 0; k < n_angles; ++k) h[k] = angles ? angles[k] : (double)k;
    memcpy(h.data() + n_angles, angle_tab, (size_t)n_angles * 4 * sizeof(double));
    // small pageable copy: the runtime stages it before returning, so `h` may go out of scope
    CU(cudaMemcpyAsync(ctx->angles.p, h.data(), bytes, cudaMemcpyHostToDevice, st ? st : ctx->stream));
    *d_angles = (const double *)ctx->angles.p;
    *d_tab = *d_angles + n_angles;
    return SID_OK;
}

namespace {

// Largest border (<= max_border) for which plan_pm would pick pm_ws_kernel (its geometry, its shared-memory layout and
// the split tail all fit); -1 if none.
int ws_border_limit(sid_ctx *ctx, int s, int n_angles, unsigned flags, int max_border) {
    if (!ws_wanted()) return -1;
    const bool smth = (flags & SID_HES_SMTH) != 0;
    for (int b = std::min(max_border, 40); b >= 1; --b) {
        const int Rmax = 2 * (s / 2) + 2 * b + 1 - s + 1;
        if (Rmax < 2) break;
        if (!split_tail_fits(Rmax * Rmax, smth)) continue;
        PmWsCfg g;
        // the planner pads the angle planes for ITS typical map width (<= 31 words in each of 2 x 3 planes): where that may
        // not fit, try every width, so that a border accepted here is never refused by the launch
        // (the smallest layout: two sets of window statistics)
        bool ok = ws_fits(ctx, s, b, n_angles, 0, 2, g);
        if (ok && !ws_fits(ctx, s, b, n_angles, 0, 2, g, 31 * 4 * 2 * 3))
            for (int rt = 2; rt <= Rmax && ok; ++rt) ok = ws_fits(ctx, s, b, n_angles, rt, 2, g);
        if (ok) return b;
    }
    return -1;
}

// Border classes of a call with borders up to max_border: the points with borders up to the returned limit go to
// pm_ws_kernel in launches of their own, the others to the kernels for larger maps; -1: one class (SID_PM_CLASSES=0, or
// pm_ws_kernel takes all borders or none)
int small_class_limit(sid_ctx *ctx, int s, int n_angles, unsigned flags, int max_border) {
    const char *e = getenv("SID_PM_CLASSES");
    if (e && e[0] == '0') return -1;
    const int limit = ws_border_limit(ctx, s, n_angles, flags, max_border);
    return limit < max_border ? limit : -1;
}

// A point's border in whole pixels (fractional borders: the window can be one pixel wider; not finite, negative or
// >= 4096: 0)
__host__ __device__ inline int border_pixels(double b) {
    return isfinite(b) && b >= 0.0 && b < 4096.0 ? (int)ceil(b) : 0;
}

// Device-resident callers (sid_run_device): split the point indices by border class on the device
__global__ void partition_by_border_kernel(const double *__restrict__ border, int n, int limit, int *__restrict__ order_small,
                                           int *__restrict__ order_big, unsigned *__restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool small = false, valid = i < n;
    if (valid) {
        small = border_pixels(border[i]) <= limit;
    }
    const unsigned m_small = __ballot_sync(0xffffffffu, valid && small), m_big = __ballot_sync(0xffffffffu, valid && !small);
    const int lane = threadIdx.x & 31;
    unsigned base_s = 0, base_b = 0;
    if (lane == 0) {
        if (m_small) base_s = atomicAdd(&counts[0], (unsigned)__popc(m_small));
        if (m_big) base_b = atomicAdd(&counts[1], (unsigned)__popc(m_big));
    }
    base_s = __shfl_sync(0xffffffffu, base_s, 0); base_b = __shfl_sync(0xffffffffu, base_b, 0);
    const unsigned below = (1u << lane) - 1u;
    if (valid && small) order_small[base_s + __popc(m_small & below)] = i;
    if (valid && !small) order_big[base_b + __popc(m_big & below)] = i;
}

// true when `p` is ordinary pageable host memory (cudaMemcpyAsync from it is a slow, synchronous staged copy)
bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

// rows x width bytes from (src, spitch) to (dst, dpitch), split over `nthreads` host threads
// One row: streaming (non-temporal) 16-byte stores when the destination allows -- the staging buffer is written once and
// read by the DMA engine, so allocating its lines in the cache only costs a read-for-ownership per line
inline void copy_row_stream(uint8_t *dst, const uint8_t *src, size_t width) {
    if ((reinterpret_cast<uintptr_t>(dst) & 15u) != 0 || width < 256) { memcpy(dst, src, width); return; }
    const size_t n16 = width / 16;
    const __m128i *s16 = reinterpret_cast<const __m128i *>(src);
    __m128i *d16 = reinterpret_cast<__m128i *>(dst);
    size_t i = 0;
    for (; i + 4 <= n16; i += 4) {
        const __m128i v0 = _mm_loadu_si128(s16 + i), v1 = _mm_loadu_si128(s16 + i + 1);
        const __m128i v2 = _mm_loadu_si128(s16 + i + 2), v3 = _mm_loadu_si128(s16 + i + 3);
        _mm_stream_si128(d16 + i, v0); _mm_stream_si128(d16 + i + 1, v1);
        _mm_stream_si128(d16 + i + 2, v2); _mm_stream_si128(d16 + i + 3, v3);
    }
    for (; i < n16; ++i) _mm_stream_si128(d16 + i, _mm_loadu_si128(s16 + i));
    if (width & 15u) memcpy(dst + n16 * 16, src + n16 * 16, width & 15u);
}

// Rows of up to two images into the pinned staging slot, split over the pool's threads by row count
struct RowCopy { uint8_t *dst; size_t dpitch; const uint8_t *src; size_t spitch, width; int rows; };
void copy_rows_pool(HostPool *pool, const RowCopy *jobs, int njobs) {
    long long total = 0;
    for (int j = 0; j < njobs; ++j) total += std::max(0, jobs[j].rows);
    if (total <= 0) return;
    const int parts = pool ? pool->size() : 1;
    const std::function<void(int)> work = [&](int part) {
        long long lo = total * part / parts, hi = total * (part + 1) / parts, base = 0;
        for (int j = 0; j < njobs; ++j) {
            const RowCopy &c = jobs[j];
            const long long r0 = std::max(lo, base) - base, r1 = std::min(hi, base + c.rows) - base;
            for (long long r = r0; r < r1; ++r) copy_row_stream(c.dst + (size_t)r * c.dpitch, c.src + (size_t)r * c.spitch, c.width);
            base += c.rows;
        }
        _mm_sfence();                    // the streaming stores are globally visible before the DMA is enqueued
    };
    if (pool && parts > 1) pool->run(work); else work(0);
}

struct HostPair {
    const uint8_t *img1, *img2;
    int rows1, cols1, rows2, cols2;
    long long pitch1, pitch2;
};

constexpr int MAX_BANDS = 16;

// Body of sid_run, sid_run_pair and sid_run_maps (maps_out, map_off, tpl_out: see PmArgs).  With `pair` the images are uploaded in row bands on a second
// stream while the fused kernel already works on the points whose windows and templates lie
// entirely inside the bands that have arrived (PCIe copy overlapped with compute).
int run_host(sid_ctx *ctx, const HostPair *pair, int64_t n, const double *c1, const double *r1, const double *c2fg,
             const double *r2fg, const double *border, int img_size, int n_angles, const double *angles,
             const double *angle_tab, int rot_order, unsigned flags, int mtype, double *out, int *status,
             float *maps_out, const long long *map_off, uint8_t *tpl_out) {
    int rc = check_common(ctx, img_size, n_angles, angle_tab, rot_order, mtype);
    if (rc) return rc;
    ctx->peaks_n = -1;
    ctx->peaks_of_table = false;
    ctx->uncert_n = -1;
    if ((rc = check_uncert(ctx, flags))) return rc;
    if (!pair && !ctx->have_pair) return fail(ctx, SID_ENOPAIR, "sid_set_pair has not been called");
    if (n < 0 || (n > 0 && (!c1 || !r1 || !c2fg || !r2fg || !border)) || !angles)
        return fail(ctx, SID_EINVAL, "null point array");
    if (n > 0x7fffffffLL) return fail(ctx, SID_EINVAL, "too many points");
    CU(cudaSetDevice(ctx->device));
    if (pair) {
        if (!pair->img1 || !pair->img2 || pair->rows1 <= 0 || pair->cols1 <= 0 || pair->rows2 <= 0 || pair->cols2 <= 0 ||
            pair->pitch1 < pair->cols1 || pair->pitch2 < pair->cols2)
            return fail(ctx, SID_EINVAL, "bad image arguments");
        if (n == 0) {
            if ((rc = sid_set_pair(ctx, pair->img1, pair->rows1, pair->cols1, pair->pitch1, pair->img2, pair->rows2,
                                   pair->cols2, pair->pitch2)))
                return rc;
            ctx->peaks_n = (flags & SID_PEAKS) ? 0 : -1;
            ctx->uncert_n = (flags & SID_UNCERT) ? 0 : -1;
            return SID_OK;
        }
    }
    if (n == 0) {
        ctx->peaks_n = (flags & SID_PEAKS) ? 0 : -1;
        ctx->uncert_n = (flags & SID_UNCERT) ? 0 : -1;
        return SID_OK;
    }

    // ---- bands (upload granularity); a single band means "everything is already resident".  The bands TAPER: while the
    //      upload runs the kernels of band k hide behind the copy of band k + 1, but the kernels of the LAST band run after
    //      the last byte has arrived -- so the last bands are short (weights below; SID_BAND_PLAN="w0,w1,..." overrides,
    //      SID_BANDS=n gives n equal bands).  Boundaries are multiples of 64 rows.
    const int rows1 = pair ? pair->rows1 : ctx->rows1, rows2 = pair ? pair->rows2 : ctx->rows2;
    const int max_rows = std::max(rows1, rows2);
    int nbands = 1;
    std::vector<double> weights;
    if (pair) {
        if (max_rows >= 8192) weights = {6, 6, 6, 6, 6, 5, 4, 3, 2, 1};
        else weights.assign((size_t)std::max(1, std::min(8, max_rows / 512)), 1.0);
        if (const char *e = getenv("SID_BANDS")) weights.assign((size_t)std::max(1, std::min(MAX_BANDS, atoi(e))), 1.0);
        if (const char *e = getenv("SID_BAND_PLAN")) {
            std::vector<double> w;
            for (const char *q = e; *q && (int)w.size() < MAX_BANDS;) {
                char *end = nullptr;
                const double v = strtod(q, &end);
                if (end == q) break;
                if (v > 0.0) w.push_back(v);
                q = (*end == ',') ? end + 1 : end;
            }
            if (!w.empty()) weights = w;
        }
        nbands = (int)weights.size();
    }
    std::vector<int> band_lo((size_t)nbands + 1, 0);
    {
        double total = 0.0, acc = 0.0;
        for (double w : weights) total += w;
        for (int k = 1; k < nbands; ++k) {
            acc += weights[(size_t)k - 1];
            int y = (int)((double)max_rows * acc / total / 64.0 + 0.5) * 64;
            band_lo[(size_t)k] = std::max(band_lo[(size_t)k - 1], std::min(max_rows, y));
        }
        band_lo[(size_t)nbands] = max_rows;
    }
    int band_rows = 0;                                          // tallest band (sizes the staging slots)
    for (int k = 0; k < nbands; ++k) band_rows = std::max(band_rows, band_lo[(size_t)k + 1] - band_lo[(size_t)k]);
    std::vector<unsigned char> band_of64((size_t)max_rows / 64 + 2, (unsigned char)(nbands - 1));
    for (int k = 0, j = 0; k < nbands; ++k)
        for (; j * 64 < band_lo[(size_t)k + 1] && (size_t)j < band_of64.size(); ++j) band_of64[(size_t)j] = (unsigned char)k;

    // ---- image upload in bands on the copy stream
    if (pair) {
        ctx->have_pair = false;
        if (!ctx->copy_stream) {
            CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
            for (int k = 0; k <= MAX_BANDS; ++k) CU(cudaEventCreateWithFlags(&ctx->band_event[k], cudaEventDisableTiming));
        }
        ctx->pitch1 = padded_pitch(pair->cols1);
        ctx->pitch2 = padded_pitch(pair->cols2);
        const size_t b1 = (size_t)ctx->pitch1 * pair->rows1 + IMG_TAIL_SLACK, b2 = (size_t)ctx->pitch2 * pair->rows2 + IMG_TAIL_SLACK;
        const bool fresh1 = b1 > ctx->img1.cap || !ctx->img1.owned, fresh2 = b2 > ctx->img2.cap || !ctx->img2.owned;
        if ((rc = reserve(ctx, ctx->img1, b1))) return rc;
        if ((rc = reserve(ctx, ctx->img2, b2))) return rc;
        // the copy stream must not overwrite images an earlier launch on the compute stream still reads
        CU(cudaEventRecord(ctx->band_event[MAX_BANDS], ctx->stream));
        CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->band_event[MAX_BANDS], 0));
        if (fresh1) CU(cudaMemsetAsync(ctx->img1.p, 0, ctx->img1.cap, ctx->copy_stream));
        if (fresh2) CU(cudaMemsetAsync(ctx->img2.p, 0, ctx->img2.cap, ctx->copy_stream));
        ctx->rows1 = pair->rows1; ctx->cols1 = pair->cols1; ctx->rows2 = pair->rows2; ctx->cols2 = pair->cols2;
    }

    // Pageable host images (plain NumPy arrays): each band goes through a pinned double buffer, filled by a few host
    // threads while the previous band's DMA and kernels run; band k's kernels are launched right behind its copy.
    bool staged = false;
    int copy_threads = 1;
    if (pair) {
        staged = is_pageable(pair->img1) || is_pageable(pair->img2);
        if (const char *e = getenv("SID_STAGED_UPLOAD")) staged = e[0] != '0';
        copy_threads = (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2));
        if (const char *e = getenv("SID_UPLOAD_THREADS")) copy_threads = std::max(1, std::min(64, atoi(e)));
    }
    const size_t slot_bytes = pair ? ((size_t)band_rows * ((size_t)pair->cols1 + (size_t)pair->cols2) + 255) / 256 * 256 : 0;
    if (staged) {
        if (2 * slot_bytes > ctx->stage_cap) {
            if (ctx->stage) { cudaFreeHost(ctx->stage); ctx->stage = nullptr; ctx->stage_cap = 0; }
            if (cudaMallocHost(&ctx->stage, 2 * slot_bytes) != cudaSuccess) { cudaGetLastError(); return fail(ctx, SID_ENOMEM, "pinned staging allocation failed"); }
            ctx->stage_cap = 2 * slot_bytes;
        }
        for (int k = 0; k < 2; ++k) if (!ctx->stage_event[k]) CU(cudaEventCreateWithFlags(&ctx->stage_event[k], cudaEventDisableTiming));
    }
    auto enqueue_band_copy = [&](int k) -> int {
        const int ya = band_lo[(size_t)k], nrows = band_lo[(size_t)k + 1] - ya;
        const int n1 = std::min(nrows, pair->rows1 - ya), n2 = std::min(nrows, pair->rows2 - ya);
        const uint8_t *s1 = pair->img1 + (size_t)ya * pair->pitch1, *s2 = pair->img2 + (size_t)ya * pair->pitch2;
        size_t sp1 = (size_t)pair->pitch1, sp2 = (size_t)pair->pitch2;
        if (staged) {
            const int slot = k & 1;
            if (k >= 2) CU(cudaEventSynchronize(ctx->stage_event[slot]));      // the DMA of band k-2 has drained this slot
            uint8_t *d1 = (uint8_t *)ctx->stage + (size_t)slot * slot_bytes, *d2 = d1 + (size_t)band_rows * pair->cols1;
            if (copy_threads > 1 && (!ctx->pool || ctx->pool->size() != copy_threads)) {
                delete ctx->pool;
                ctx->pool = new HostPool(copy_threads - 1);
            }
            const RowCopy jobs[2] = {{d1, (size_t)pair->cols1, s1, sp1, (size_t)pair->cols1, std::max(n1, 0)},
                                     {d2, (size_t)pair->cols2, s2, sp2, (size_t)pair->cols2, std::max(n2, 0)}};
            copy_rows_pool(copy_threads > 1 ? ctx->pool : nullptr, jobs, 2);
            s1 = d1; s2 = d2; sp1 = (size_t)pair->cols1; sp2 = (size_t)pair->cols2;
        }
        if (n1 > 0)
            CU(cudaMemcpy2DAsync((char *)ctx->img1.p + (size_t)ya * ctx->pitch1, (size_t)ctx->pitch1, s1, sp1, (size_t)pair->cols1,
                                 (size_t)n1, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (n2 > 0)
            CU(cudaMemcpy2DAsync((char *)ctx->img2.p + (size_t)ya * ctx->pitch2, (size_t)ctx->pitch2, s2, sp2, (size_t)pair->cols2,
                                 (size_t)n2, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (staged) CU(cudaEventRecord(ctx->stage_event[k & 1], ctx->copy_stream));
        CU(cudaEventRecord(ctx->band_event[k], ctx->copy_stream));
        return SID_OK;
    };
    // band 0 goes out before the host-side preparation below (point order, small uploads), which then overlaps its DMA;
    // the small uploads queue behind it on the copy engine (the first kernel needs band 0 anyway), the other bands behind them
    if (pair && !staged && (rc = enqueue_band_copy(0))) return rc;

    // ---- borders: bound, typical value, and the processing order: band of the last image row a point
    //      touches first, then largest window first (counting sort on the combined key)
    int max_border = 0;
    std::vector<int> ib((size_t)n), band((size_t)n, 0);
    const double ext = 0.5 * std::sqrt(2.0) * (img_size + 2) + 3.0;      // template reach around (c1, r1) incl. rounding
    const int hws = img_size / 2;
    for (int64_t i = 0; i < n; ++i) {
        const int v = border_pixels(border[i]);
        ib[(size_t)i] = v;
        max_border = std::max(max_border, v);
        if (nbands > 1) {
            double need = 0.0;
            if (std::isfinite(r1[i]) && std::isfinite(r2fg[i])) need = std::max(r1[i] + ext, r2fg[i] + hws + v + 2.0);
            band[(size_t)i] = need <= 0.0 ? 0 : (int)band_of64[(size_t)std::min((double)(band_of64.size() - 1), need / 64.0)];
        }
    }
    const size_t nkeys = (size_t)nbands * (size_t)(max_border + 1);
    std::vector<int> hist(nkeys + 1, 0);
    auto key_of = [&](int64_t i) { return (size_t)band[(size_t)i] * (size_t)(max_border + 1) + (size_t)(max_border - ib[(size_t)i]); };
    for (int64_t i = 0; i < n; ++i) ++hist[key_of(i) + 1];
    for (size_t k = 1; k < hist.size(); ++k) hist[k] += hist[k - 1];
    std::vector<int> band_start((size_t)nbands + 1, 0);
    for (int k = 0; k <= nbands; ++k) band_start[(size_t)k] = hist[std::min(nkeys, (size_t)k * (size_t)(max_border + 1))];
    std::vector<long long> per_b((size_t)max_border + 1, 0);
    for (int64_t i = 0; i < n; ++i) ++per_b[(size_t)ib[(size_t)i]];
    auto median_border = [&](int b_lo, int b_hi) {          // median of the borders in [b_lo, b_hi] = the typical point of a class
        long long total = 0, acc = 0;
        for (int b = b_lo; b <= b_hi; ++b) total += per_b[(size_t)b];
        for (int b = b_hi; b >= b_lo; --b) { acc += per_b[(size_t)b]; if (2 * acc > total) return b; }
        return b_hi;
    };
    int typ_border = median_border(0, max_border);
    // ---- border classes.  A launch is sized by its largest border, and the fastest kernel (pm_ws_kernel) only takes small
    //      result maps: with the reference's default borders (20 ... 50 by the distance to the nearest keypoint,
    //      pmlib.py:315-322) most points sit at the minimum -- 86 % of BASELINE configs[0]'s grid with a real ORB first
    //      guess -- and a few far from any keypoint would drag the whole call onto the kernels for large maps.  So the points
    //      whose border fits pm_ws_kernel get their own launch per band, behind the larger ones (SID_PM_CLASSES=0: one launch).
    int small_max = -1, typ_small = 0, typ_big = typ_border;
    bool two_class = false;
    const int limit = small_class_limit(ctx, img_size, n_angles, flags, max_border);
    if (limit >= 0) {
        long long n_small = 0;
        for (int b = 0; b <= limit; ++b) if (per_b[(size_t)b]) { n_small += per_b[(size_t)b]; small_max = b; }
        if (n_small >= 256 && small_max >= 1) {
            two_class = true;
            typ_small = median_border(0, small_max);
            typ_big = median_border(limit + 1, max_border);
        }
    }
    std::vector<int> band_mid((size_t)nbands, 0);           // first point of the small class inside each band's range
    for (int k = 0; k < nbands; ++k)
        band_mid[(size_t)k] = two_class ? hist[(size_t)k * (size_t)(max_border + 1) + (size_t)(max_border - small_max)]
                                        : band_start[(size_t)k + 1];

    const size_t pts_bytes = (size_t)n * 5 * sizeof(double);
    const size_t ord_bytes = (size_t)n * sizeof(int);
    const size_t out_bytes = (size_t)n * 5 * sizeof(double);
    const size_t st_bytes = (size_t)n * sizeof(int);
    rc = reserve_pinned(ctx, pts_bytes + ord_bytes + out_bytes + st_bytes + 64);
    if (rc) return rc;
    if ((rc = reserve(ctx, ctx->pts, pts_bytes))) return rc;
    if ((rc = reserve(ctx, ctx->order, ord_bytes))) return rc;
    if ((rc = reserve(ctx, ctx->out, out_bytes))) return rc;
    if ((rc = reserve(ctx, ctx->status, st_bytes))) return rc;
    if ((flags & SID_PEAKS) && (rc = reserve(ctx, ctx->peaks, (size_t)n * SID_N_PEAKS * 4 * sizeof(double)))) return rc;

    double *hp = (double *)ctx->pin;
    memcpy(hp, c1, (size_t)n * 8); memcpy(hp + n, r1, (size_t)n * 8); memcpy(hp + 2 * n, c2fg, (size_t)n * 8);
    memcpy(hp + 3 * n, r2fg, (size_t)n * 8); memcpy(hp + 4 * n, border, (size_t)n * 8);
    int *hord = (int *)((char *)ctx->pin + pts_bytes);
    for (int64_t i = 0; i < n; ++i) hord[hist[key_of(i)]++] = (int)i;

    // ---- small uploads.  With pinned images they go on the COPY stream, between band 0 and band 1: the copy engine serves
    //      one stream's queue in order, but between streams it does not keep the issue order (measured: point arrays enqueued
    //      on the compute stream while band 0 was in flight were served after ALL bands -- 8.3 instead of 5.0 ms per pair).
    //      The staged path enqueues its bands one by one below, so there the small uploads simply go first.
    cudaStream_t up = (pair && !staged) ? ctx->copy_stream : ctx->stream;
    CU(cudaMemcpyAsync(ctx->pts.p, hp, pts_bytes, cudaMemcpyHostToDevice, up));
    CU(cudaMemcpyAsync(ctx->order.p, hord, ord_bytes, cudaMemcpyHostToDevice, up));
    const double *d_angles, *d_tab;
    if ((rc = upload_angles(ctx, n_angles, angles, angle_tab, &d_angles, &d_tab, up))) return rc;
    // rows that end up neither valid nor masked keep NaN (all bits set) peak records
    if (flags & SID_PEAKS) CU(cudaMemsetAsync(ctx->peaks.p, 0xff, (size_t)n * SID_N_PEAKS * 4 * sizeof(double), up));
    if (!ctx->slot_event[0])
        for (int k = 0; k < 3; ++k) CU(cudaEventCreateWithFlags(&ctx->slot_event[k], cudaEventDisableTiming));
    CU(cudaEventRecord(ctx->slot_event[0], up));                       // point / angle uploads are enqueued

    if (pair && !staged)
        for (int k = 1; k < nbands; ++k) if ((rc = enqueue_band_copy(k))) return rc;

    const double *dp = (const double *)ctx->pts.p;
    PmCall call{dp, dp + n, dp + 2 * n, dp + 3 * n, dp + 4 * n, d_angles, d_tab, rot_order, (double *)ctx->out.p,
                (int *)ctx->status.p, maps_out, map_off, tpl_out, n, 0, 0};
    if (flags & SID_PEAKS) call.peaks = (double *)ctx->peaks.p;
    // the larger borders (all points when the call is not split into classes), the class of pm_ws_kernel, the masked pass,
    // the uncertainty pass
    PmPlan plans[4];
    const bool masked = (flags & SID_MASKED) != 0, uncert = (flags & SID_UNCERT) != 0;
    const int nplans = two_class ? 2 : 1, p_unc = nplans + (masked ? 1 : 0);
    if ((rc = plan_pm(ctx, img_size, n_angles, flags, max_border, two_class ? typ_big : typ_border, plans[0]))) return rc;
    if (two_class && (rc = plan_pm(ctx, img_size, n_angles, flags, small_max, typ_small, plans[1]))) return rc;
    if (masked && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, typ_border, plans[nplans], PASS_MASKED))) return rc;
    if (uncert && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, typ_border, plans[p_unc], PASS_UNCERT))) return rc;
    if ((rc = reserve_call(ctx, call, plans, p_unc + (uncert ? 1 : 0)))) return rc;
    const bool two_streams = pair && nbands > 1;
    if (two_streams) {
        if (!ctx->band_stream[0])
            for (int k = 0; k < 2; ++k) CU(cudaStreamCreateWithFlags(&ctx->band_stream[k], cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) CU(cudaStreamWaitEvent(ctx->band_stream[k], ctx->slot_event[0], 0));
    } else if (up != ctx->stream) {
        CU(cudaStreamWaitEvent(ctx->stream, ctx->slot_event[0], 0));
    }
    for (int k = 0; k < nbands; ++k) {
        if (staged && (rc = enqueue_band_copy(k))) return rc;
        // consecutive bands go to alternating streams: the next band's CTAs fill the SMs while this one drains
        cudaStream_t st = two_streams ? ctx->band_stream[k & 1] : ctx->stream;
        if (pair) CU(cudaStreamWaitEvent(st, ctx->band_event[k], 0));
        const int lo = band_start[(size_t)k], hi = band_start[(size_t)k + 1], mid = band_mid[(size_t)k];
        if (hi <= lo) continue;
        const int slot = two_streams ? (k & 1) : 0;
        const int *order = (const int *)ctx->order.p;
        if (mid > lo && (rc = enqueue_pm(ctx, call, plans[0], mid - lo, order + lo, st, slot, lo, false))) return rc;
        if (hi > mid && (rc = enqueue_pm(ctx, call, plans[1], hi - mid, order + mid, st, slot, mid, mid > lo))) return rc;
    }
    if (two_streams) {
        for (int k = 0; k < 2; ++k) {
            CU(cudaEventRecord(ctx->slot_event[1 + k], ctx->band_stream[k]));
            CU(cudaStreamWaitEvent(ctx->stream, ctx->slot_event[1 + k], 0));
        }
    }
    // every band has arrived and every row has its status
    if (masked && (rc = enqueue_pm(ctx, call, plans[nplans], n, nullptr, ctx->stream, 0, 0, true))) return rc;
    // ... and every row has its final table entry and status
    if (uncert && (rc = enqueue_pm(ctx, call, plans[p_unc], n, nullptr, ctx->stream, 0, 0, true))) return rc;
    if (pair) ctx->have_pair = true;
    double *hout = (double *)((char *)ctx->pin + pts_bytes + ord_bytes);
    int *hst = (int *)((char *)hout + out_bytes);
    ctx->table_n = n;                                          // the (n, 5) table stays in ctx->out for sid_pm_epilogue_affine
    if (out) CU(cudaMemcpyAsync(hout, ctx->out.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (status) CU(cudaMemcpyAsync(hst, ctx->status.p, st_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    if (out) memcpy(out, hout, out_bytes);
    if (status) memcpy(status, hst, st_bytes);
    if (flags & SID_PEAKS) { ctx->peaks_n = n; ctx->peaks_of_table = true; }
    if (uncert) ctx->uncert_n = n;
    return SID_OK;
}

}  // namespace

int sid_run(sid_ctx *ctx, int64_t n, const double *c1, const double *r1, const double *c2fg,
            const double *r2fg, const double *border, int img_size, int n_angles, const double *angles,
            const double *angle_tab, int rot_order, unsigned flags, int mtype, double *out, int *status) {
    return run_host(ctx, nullptr, n, c1, r1, c2fg, r2fg, border, img_size, n_angles, angles, angle_tab, rot_order,
                    flags, mtype, out, status, nullptr, nullptr, nullptr);
}

int sid_run_pair(sid_ctx *ctx, const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                 const uint8_t *img2, int rows2, int cols2, int64_t pitch2,
                 int64_t n, const double *c1, const double *r1, const double *c2fg,
                 const double *r2fg, const double *border, int img_size, int n_angles, const double *angles,
                 const double *angle_tab, int rot_order, unsigned flags, int mtype, double *out, int *status) {
    if (!ctx) return SID_EINVAL;
    HostPair hp{img1, img2, rows1, cols1, rows2, cols2, (long long)pitch1, (long long)pitch2};
    return run_host(ctx, &hp, n, c1, r1, c2fg, r2fg, border, img_size, n_angles, angles, angle_tab, rot_order,
                    flags, mtype, out, status, nullptr, nullptr, nullptr);
}

int sid_run_device(sid_ctx *ctx, int64_t n, const double *d_c1, const double *d_r1, const double *d_c2fg,
                   const double *d_r2fg, const double *d_border, int max_border, int img_size, int n_angles,
                   const double *angles, const double *angle_tab, int rot_order, unsigned flags, int mtype,
                   double *d_out, int *d_status) {
    int rc = check_common(ctx, img_size, n_angles, angle_tab, rot_order, mtype);
    if (rc) return rc;
    ctx->peaks_n = -1;
    ctx->peaks_of_table = false;
    ctx->uncert_n = -1;
    if ((rc = check_uncert(ctx, flags))) return rc;
    if (!ctx->have_pair) return fail(ctx, SID_ENOPAIR, "sid_set_pair has not been called");
    if (n < 0 || (n > 0 && (!d_c1 || !d_r1 || !d_c2fg || !d_r2fg || !d_border || !d_out)) || !angles)
        return fail(ctx, SID_EINVAL, "null point array");
    if (n == 0) {
        ctx->peaks_n = (flags & SID_PEAKS) ? 0 : -1;
        ctx->uncert_n = (flags & SID_UNCERT) ? 0 : -1;
        return SID_OK;
    }
    CU(cudaSetDevice(ctx->device));
    if (max_border <= 0) {
        std::vector<double> hb((size_t)n);
        CU(cudaMemcpyAsync(hb.data(), d_border, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        max_border = 1;
        for (double b : hb) max_border = std::max(max_border, border_pixels(b));
    }
    const double *d_angles, *d_tab;
    if ((rc = upload_angles(ctx, n_angles, angles, angle_tab, &d_angles, &d_tab))) return rc;
    PmCall call{d_c1, d_r1, d_c2fg, d_r2fg, d_border, d_angles, d_tab, rot_order, d_out, d_status, nullptr, nullptr, nullptr, n, 0, 0};
    if (flags & SID_PEAKS) {
        const size_t b = (size_t)n * SID_N_PEAKS * 4 * sizeof(double);
        if ((rc = reserve(ctx, ctx->peaks, b))) return rc;
        CU(cudaMemsetAsync(ctx->peaks.p, 0xff, b, ctx->stream));
        call.peaks = (double *)ctx->peaks.p;
    }
    PmPlan plans[4];                 // [0], [1]: the border classes; the masked and uncertainty passes behind them
    const bool masked = (flags & SID_MASKED) != 0, uncert = (flags & SID_UNCERT) != 0;
    // border classes as in sid_run (see run_host): the indices are split on the device, one 8-byte read-back sizes the launches
    const int limit = n < 512 ? -1 : small_class_limit(ctx, img_size, n_angles, flags, max_border);
    if (limit >= 0) {
        if ((rc = reserve(ctx, ctx->order, (size_t)n * 2 * sizeof(int) + 64))) return rc;
        int *d_small = (int *)ctx->order.p, *d_big = d_small + n;
        unsigned *d_counts = (unsigned *)(d_big + n);
        CU(cudaMemsetAsync(d_counts, 0, 8, ctx->stream));
        partition_by_border_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_border, (int)n, limit, d_small, d_big, d_counts);
        ctx->launches += 1;
        unsigned counts[2] = {0, 0};
        CU(cudaMemcpyAsync(counts, d_counts, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(cudaGetLastError());
        const long long n_small = counts[0], n_big = counts[1];
        if (n_small >= 256 && n_big > 0) {
            if ((rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[0]))) return rc;
            if ((rc = plan_pm(ctx, img_size, n_angles, flags, limit, limit, plans[1]))) return rc;
            const int p_unc = masked ? 3 : 2;
            if (masked && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[2], PASS_MASKED))) return rc;
            if (uncert && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[p_unc], PASS_UNCERT))) return rc;
            if ((rc = reserve_call(ctx, call, plans, p_unc + (uncert ? 1 : 0)))) return rc;
            if ((rc = enqueue_pm(ctx, call, plans[0], n_big, d_big, ctx->stream, 0, 0, false))) return rc;
            if ((rc = enqueue_pm(ctx, call, plans[1], n_small, d_small, ctx->stream, 0, n_big, true))) return rc;
            if (masked && (rc = enqueue_pm(ctx, call, plans[2], n, nullptr, ctx->stream, 0, 0, true))) return rc;
            if (uncert && (rc = enqueue_pm(ctx, call, plans[p_unc], n, nullptr, ctx->stream, 0, 0, true))) return rc;
            if (flags & SID_PEAKS) ctx->peaks_n = n;
            if (uncert) ctx->uncert_n = n;
            return SID_OK;
        }
        if (n_big == 0) max_border = limit;              // every point fits the pipeline kernel
    }
    if ((rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[0]))) return rc;
    const int p_unc = masked ? 2 : 1;
    if (masked && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[1], PASS_MASKED))) return rc;
    if (uncert && (rc = plan_pm(ctx, img_size, n_angles, flags, max_border, max_border, plans[p_unc], PASS_UNCERT))) return rc;
    if ((rc = reserve_call(ctx, call, plans, p_unc + (uncert ? 1 : 0)))) return rc;
    if ((rc = enqueue_pm(ctx, call, plans[0], n, nullptr, ctx->stream, 0, 0, false))) return rc;
    if (masked && (rc = enqueue_pm(ctx, call, plans[1], n, nullptr, ctx->stream, 0, 0, true))) return rc;
    if (uncert && (rc = enqueue_pm(ctx, call, plans[p_unc], n, nullptr, ctx->stream, 0, 0, true))) return rc;
    if (flags & SID_PEAKS) ctx->peaks_n = n;
    if (uncert) ctx->uncert_n = n;
    return SID_OK;
}

// ------------------------------------------------------------------ winning maps and templates (sid_run_maps)
namespace {
// Map shapes by the kernels' window rule (window_rect) on the resident pair; `off` (optional) gets the packed offsets
int map_layout(sid_ctx *ctx, int64_t n, const double *c1, const double *r1, const double *c2fg, const double *r2fg,
               const double *border, int img_size, int32_t *shape, std::vector<long long> *off, int64_t *total) {
    if (!ctx) return SID_EINVAL;
    if (!ctx->have_pair) return fail(ctx, SID_ENOPAIR, "sid_set_pair has not been called");
    if (img_size < 2 || img_size > 128) return fail(ctx, SID_EUNSUPPORTED, "img_size must be in [2, 128]");
    if (n < 0 || (n > 0 && (!c1 || !r1 || !c2fg || !r2fg || !border)) || !total) return fail(ctx, SID_EINVAL, "null point array");
    if (off) off->resize((size_t)n);
    const WindowGeom g{img_size, ctx->rows2, ctx->cols2};
    long long acc = 0;
    for (int64_t i = 0; i < n; ++i) {
        long long x0, y0;
        int W, H, RH = 0, RW = 0;
        if (window_rect(g, c1[i], r1[i], c2fg[i], r2fg[i], border[i], x0, y0, W, H)) {
            RH = H - img_size + 1; RW = W - img_size + 1;
        }
        if (shape) { shape[2 * i] = RH; shape[2 * i + 1] = RW; }
        if (off) (*off)[(size_t)i] = acc;
        acc += (long long)RH * RW;
    }
    *total = acc;
    return SID_OK;
}
}  // namespace

int sid_map_layout(sid_ctx *ctx, int64_t n, const double *c1, const double *r1, const double *c2fg, const double *r2fg,
                   const double *border, int img_size, int32_t *map_shape, int64_t *total) {
    return map_layout(ctx, n, c1, r1, c2fg, r2fg, border, img_size, map_shape, nullptr, total);
}

int sid_run_maps(sid_ctx *ctx, int64_t n, const double *c1, const double *r1, const double *c2fg,
                 const double *r2fg, const double *border, int img_size, int n_angles, const double *angles,
                 const double *angle_tab, int rot_order, unsigned flags, int mtype, double *out, int *status,
                 int64_t maps_capacity, float *maps, uint8_t *templates) {
    int rc = check_common(ctx, img_size, n_angles, angle_tab, rot_order, mtype);
    if (rc) return rc;
    ctx->peaks_n = -1;
    ctx->peaks_of_table = false;
    ctx->uncert_n = -1;
    if ((rc = check_uncert(ctx, flags))) return rc;
    if (!angles) return fail(ctx, SID_EINVAL, "null point array");
    if (n > 0x7fffffffLL) return fail(ctx, SID_EINVAL, "too many points");
    std::vector<long long> off;
    int64_t total = 0;
    if ((rc = map_layout(ctx, n, c1, r1, c2fg, r2fg, border, img_size, nullptr, &off, &total))) return rc;
    if (maps_capacity < total) return fail(ctx, SID_EINVAL, "maps_capacity below the total of sid_map_layout");
    if (total > 0 && !maps) return fail(ctx, SID_EINVAL, "null maps buffer");
    if (n == 0) {
        ctx->peaks_n = (flags & SID_PEAKS) ? 0 : -1;
        ctx->uncert_n = (flags & SID_UNCERT) ? 0 : -1;
        return SID_OK;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t tpl_bytes = (size_t)n * img_size * img_size;
    if ((rc = reserve(ctx, ctx->maps, (size_t)std::max<int64_t>(total, 1) * sizeof(float)))) return rc;
    if ((rc = reserve(ctx, ctx->map_off, (size_t)n * sizeof(long long)))) return rc;
    if (templates && (rc = reserve(ctx, ctx->tpl, tpl_bytes))) return rc;
    // segments of rows that end up not valid keep these: NaN (all bits set) maps, zero templates
    CU(cudaMemsetAsync(ctx->maps.p, 0xff, (size_t)total * sizeof(float), ctx->stream));
    if (templates) CU(cudaMemsetAsync(ctx->tpl.p, 0, tpl_bytes, ctx->stream));
    CU(cudaMemcpyAsync(ctx->map_off.p, off.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    rc = run_host(ctx, nullptr, n, c1, r1, c2fg, r2fg, border, img_size, n_angles, angles, angle_tab, rot_order,
                  flags, mtype, out, status, (float *)ctx->maps.p, (const long long *)ctx->map_off.p,
                  templates ? (uint8_t *)ctx->tpl.p : nullptr);
    if (rc) return rc;
    if (total > 0) CU(cudaMemcpy(maps, ctx->maps.p, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost));
    if (templates) CU(cudaMemcpy(templates, ctx->tpl.p, tpl_bytes, cudaMemcpyDeviceToHost));
    return SID_OK;
}

// ------------------------------------------------------------------ post-processing epilogue (SURVEY 8f rank 2)
namespace {
__device__ __forceinline__ double affine_eval(const double *m, double c, double r) {      // (m0*c + m1*r) + m2, NumPy's order, no FMA
    return __dadd_rn(__dadd_rn(__dmul_rn(m[0], c), __dmul_rn(m[1], r)), m[2]);
}
__global__ void pm_epilogue_fill_kernel(double *out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = nan("");
}
struct EpiArgs { double xy[6]; double ll[6]; };
// reference pmlib.py:462-497: sub-pixel remainder, pixel -> x/y and lon/lat, u = x2 - x1, v = y2 - y1, _fill_gpi scatter
__global__ void pm_epilogue_kernel(long long n_valid, const int *gidx, const double *res, const double *c2pm1, const double *r2pm1,
                                   const EpiArgs e, long long n_grid, double *out) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_valid) return;
    const long long g = gidx[k];
    const double c = c2pm1[g], r = r2pm1[g];
    const double c2 = __dadd_rn(res[5 * k], __dsub_rn(c, rint(c)));          // results[:, 0] + (c2pm1 - round(c2pm1))[gpi]
    const double r2 = __dadd_rn(res[5 * k + 1], __dsub_rn(r, rint(r)));
    out[g] = __dsub_rn(affine_eval(e.xy, c2, r2), affine_eval(e.xy, c, r));
    out[n_grid + g] = __dsub_rn(affine_eval(e.xy + 3, c2, r2), affine_eval(e.xy + 3, c, r));
    out[2 * n_grid + g] = res[5 * k + 2];
    out[3 * n_grid + g] = res[5 * k + 3];
    out[4 * n_grid + g] = res[5 * k + 4];
    out[5 * n_grid + g] = affine_eval(e.ll, c2, r2);
    out[6 * n_grid + g] = affine_eval(e.ll + 3, c2, r2);
}
}  // namespace

int sid_pm_epilogue_affine(sid_ctx *ctx, int64_t n_valid, const int32_t *grid_index, int64_t n_grid, const double *c2pm1,
                           const double *r2pm1, const double *results, const double *xy, const double *ll, double *out) {
    if (!ctx) return SID_EINVAL;
    if (n_valid < 0 || n_grid <= 0 || n_valid > n_grid || (n_valid > 0 && !grid_index) || !c2pm1 || !r2pm1 || !xy || !ll || !out)
        return fail(ctx, SID_EINVAL, "bad epilogue arguments");
    if (!results && ctx->table_n != n_valid)
        return fail(ctx, SID_EINVAL, "no device result table of that length (run sid_run / sid_run_pair first, or pass results)");
    CU(cudaSetDevice(ctx->device));
    const size_t b_idx = ((size_t)n_valid * 4 + 255) & ~(size_t)255, b_grid = ((size_t)n_grid * 8 + 255) & ~(size_t)255;
    const size_t b_res = results ? (((size_t)n_valid * 40 + 255) & ~(size_t)255) : 0, b_out = (size_t)n_grid * 56;
    int rc = reserve(ctx, ctx->epi, b_idx + 2 * b_grid + b_res + b_out);
    if (rc) return rc;
    char *base = (char *)ctx->epi.p;
    int *d_idx = (int *)base;
    double *d_c = (double *)(base + b_idx), *d_r = (double *)(base + b_idx + b_grid);
    double *d_res = results ? (double *)(base + b_idx + 2 * b_grid) : (double *)ctx->out.p;
    double *d_out = (double *)(base + b_idx + 2 * b_grid + b_res);
    if (n_valid) CU(cudaMemcpyAsync(d_idx, grid_index, (size_t)n_valid * 4, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_c, c2pm1, (size_t)n_grid * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_r, r2pm1, (size_t)n_grid * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (results && n_valid) CU(cudaMemcpyAsync(d_res, results, (size_t)n_valid * 40, cudaMemcpyHostToDevice, ctx->stream));
    EpiArgs e;
    memcpy(e.xy, xy, sizeof e.xy);
    memcpy(e.ll, ll, sizeof e.ll);
    pm_epilogue_fill_kernel<<<(unsigned)((7 * n_grid + 255) / 256), 256, 0, ctx->stream>>>(d_out, 7 * n_grid);
    if (n_valid) pm_epilogue_kernel<<<(unsigned)((n_valid + 255) / 256), 256, 0, ctx->stream>>>(n_valid, d_idx, d_res, d_c, d_r, e, n_grid, d_out);
    ctx->launches += n_valid ? 2 : 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, d_out, b_out, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

int sid_get_uncertainty(sid_ctx *ctx, int64_t n, double *out) {
    if (!ctx) return SID_EINVAL;
    if (n < 0 || ctx->uncert_n != n) return fail(ctx, SID_EINVAL, "the previous sid_run* call did not set SID_UNCERT for n points");
    if (n > 0 && !out) return fail(ctx, SID_EINVAL, "null output pointer");
    if (n == 0) return SID_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(out, ctx->uncert.p, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

int sid_get_peaks(sid_ctx *ctx, int64_t n, double *out) {
    if (!ctx) return SID_EINVAL;
    if (n < 0 || ctx->peaks_n != n) return fail(ctx, SID_EINVAL, "the previous sid_run* call did not set SID_PEAKS for n points");
    if (n > 0 && !out) return fail(ctx, SID_EINVAL, "null output pointer");
    if (n == 0) return SID_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(out, ctx->peaks.p, (size_t)n * SID_N_PEAKS * 4 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

// ------------------------------------------------------------------ outlier filter (normalised median test)
namespace {
__global__ void outlier_index_kernel(long long n_valid, const int *gidx, int *inv) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_valid) inv[gidx[k]] = (int)k;
}
// median of v[0 .. k) (k <= 8), sorted in place; np.median's (a + b) * 0.5 of the middle two for even k
__device__ __forceinline__ double median_small(double (&v)[8], int k) {
    for (int i = 1; i < k; ++i) {
        const double x = v[i];
        int j = i - 1;
        while (j >= 0 && v[j] > x) { v[j + 1] = v[j]; --j; }
        v[j + 1] = x;
    }
    return (k & 1) ? v[k / 2] : __dmul_rn(__dadd_rn(v[k / 2 - 1], v[k / 2]), 0.5);
}
// e_x^2 + e_y^2 > threshold^2 against the neighbours' medians m and median residuals rm
__device__ __forceinline__ bool outlier_test(double dx, double dy, const double (&m)[2], const double (&rm)[2], double eps,
                                             double thr2) {
    const double ex = __ddiv_rn(fabs(__dsub_rn(dx, m[0])), __dadd_rn(rm[0], eps));
    const double ey = __ddiv_rn(fabs(__dsub_rn(dy, m[1])), __dadd_rn(rm[1], eps));
    return __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)) > thr2;
}
// One thread per table row: the rule of sid_filter_outliers (include/sid_b200.h).  Reads res / peaks, writes out / flag.
__global__ void outlier_filter_kernel(long long n_valid, int grid_rows, int grid_cols, const int *gidx, const int *inv,
                                      const double *c2pm1, const double *r2pm1, const double *res, const double *peaks,
                                      double eps, double thr2, double *out, int *flag) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_valid) return;
    const double *row = res + 5 * k;
    double *o = out + 5 * k;
    for (int c = 0; c < 5; ++c) o[c] = row[c];
    if (!isfinite(row[0])) { flag[k] = -3; return; }
    const int g = gidx[k], gr = g / grid_cols, gc = g - gr * grid_cols;
    const double cg = rint(c2pm1[g]), rg = rint(r2pm1[g]);
    double dx[8], dy[8];
    int nn = 0;
    for (int di = -1; di <= 1; ++di) {
        for (int dj = -1; dj <= 1; ++dj) {
            const int y = gr + di, x = gc + dj;
            if ((di == 0 && dj == 0) || y < 0 || y >= grid_rows || x < 0 || x >= grid_cols) continue;
            const int q = inv[y * grid_cols + x];
            if (q < 0 || !isfinite(res[5 * (long long)q])) continue;
            const int gq = y * grid_cols + x;
            dx[nn] = __dsub_rn(res[5 * (long long)q], rint(c2pm1[gq]));
            dy[nn] = __dsub_rn(res[5 * (long long)q + 1], rint(r2pm1[gq]));
            ++nn;
        }
    }
    if (nn < 3) { flag[k] = -2; return; }
    double m[2], rm[2];
    m[0] = median_small(dx, nn);
    m[1] = median_small(dy, nn);
    for (int i = 0; i < nn; ++i) { dx[i] = fabs(__dsub_rn(dx[i], m[0])); dy[i] = fabs(__dsub_rn(dy[i], m[1])); }
    rm[0] = median_small(dx, nn);
    rm[1] = median_small(dy, nn);
    if (!outlier_test(__dsub_rn(row[0], cg), __dsub_rn(row[1], rg), m, rm, eps, thr2)) { flag[k] = 0; return; }
    for (int r = 0; r < SID_N_PEAKS; ++r) {
        const double *pk = peaks + (12 * k + 4 * r);
        if (!isfinite(pk[0])) continue;
        if (outlier_test(__dsub_rn(pk[0], cg), __dsub_rn(pk[1], rg), m, rm, eps, thr2)) continue;
        o[0] = pk[0]; o[1] = pk[1]; o[3] = pk[2]; o[4] = pk[3];
        flag[k] = r + 1;
        return;
    }
    for (int c = 0; c < 5; ++c) o[c] = nan("");
    flag[k] = -1;
}
}  // namespace

int sid_filter_outliers(sid_ctx *ctx, int grid_rows, int grid_cols, int64_t n_valid, const int32_t *grid_index,
                        const double *c2pm1, const double *r2pm1, const double *results, const double *peaks,
                        double eps, double threshold, double *out, int32_t *flag) {
    if (!ctx) return SID_EINVAL;
    const long long n_grid = (long long)grid_rows * (long long)grid_cols;
    if (grid_rows <= 0 || grid_cols <= 0 || n_grid > 0x7fffffffLL || n_valid < 0 || n_valid > n_grid ||
        (n_valid > 0 && !grid_index) || !c2pm1 || !r2pm1)
        return fail(ctx, SID_EINVAL, "bad outlier filter arguments");
    if (!(eps >= 0.0) || !(threshold >= 0.0) || !std::isfinite(eps) || !std::isfinite(threshold))
        return fail(ctx, SID_EINVAL, "eps and threshold must be finite and >= 0");
    const bool resident = !results && !peaks;
    if (!resident && (!results || !peaks)) return fail(ctx, SID_EINVAL, "pass both results and peaks, or neither");
    if (resident && (ctx->table_n != n_valid || ctx->peaks_n != n_valid || !ctx->peaks_of_table))
        return fail(ctx, SID_EINVAL, "no device table with SID_PEAKS of that length (run sid_run / sid_run_pair with SID_PEAKS first)");
    if (!out && !resident) return fail(ctx, SID_EINVAL, "out may be NULL only with the device-resident inputs");
    {   // every grid position once, inside the grid: the scatter below must not race or write out of bounds
        std::vector<unsigned char> seen((size_t)n_grid, 0);
        for (int64_t k = 0; k < n_valid; ++k) {
            const int32_t g = grid_index[k];
            if (g < 0 || g >= n_grid || seen[(size_t)g]) return fail(ctx, SID_EINVAL, "grid_index out of range or repeated");
            seen[(size_t)g] = 1;
        }
    }
    CU(cudaSetDevice(ctx->device));
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_inv = al((size_t)n_grid * 4), b_idx = al((size_t)n_valid * 4), b_grid = al((size_t)n_grid * 8);
    const size_t b_res = resident ? 0 : al((size_t)n_valid * 40), b_pk = resident ? 0 : al((size_t)n_valid * 96);
    const size_t b_out = al((size_t)n_valid * 40), b_flag = al((size_t)n_valid * 4);
    int rc = reserve(ctx, ctx->filt, b_inv + b_idx + 2 * b_grid + b_res + b_pk + b_out + b_flag);
    if (rc) return rc;
    char *base = (char *)ctx->filt.p;
    int *d_inv = (int *)base;
    int *d_idx = (int *)(base + b_inv);
    double *d_c = (double *)(base + b_inv + b_idx), *d_r = (double *)(base + b_inv + b_idx + b_grid);
    char *p = base + b_inv + b_idx + 2 * b_grid;
    double *d_res = resident ? (double *)ctx->out.p : (double *)p;
    double *d_pk = resident ? (double *)ctx->peaks.p : (double *)(p + b_res);
    double *d_out = (double *)(p + b_res + b_pk);
    int *d_flag = (int *)(p + b_res + b_pk + b_out);
    CU(cudaMemsetAsync(d_inv, 0xff, (size_t)n_grid * 4, ctx->stream));                // -1: no table row
    if (n_valid) CU(cudaMemcpyAsync(d_idx, grid_index, (size_t)n_valid * 4, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_c, c2pm1, (size_t)n_grid * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_r, r2pm1, (size_t)n_grid * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (!resident && n_valid) {
        CU(cudaMemcpyAsync(d_res, results, (size_t)n_valid * 40, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(d_pk, peaks, (size_t)n_valid * 96, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (n_valid) {
        const unsigned blocks = (unsigned)((n_valid + 255) / 256);
        outlier_index_kernel<<<blocks, 256, 0, ctx->stream>>>(n_valid, d_idx, d_inv);
        outlier_filter_kernel<<<blocks, 256, 0, ctx->stream>>>(n_valid, grid_rows, grid_cols, d_idx, d_inv, d_c, d_r, d_res,
                                                               d_pk, eps, threshold * threshold, d_out, d_flag);
        ctx->launches += 2;
        CU(cudaGetLastError());
        // decisions read the unfiltered table only: the filtered one is written to a second buffer and copied back
        if (out) CU(cudaMemcpyAsync(out, d_out, (size_t)n_valid * 40, cudaMemcpyDeviceToHost, ctx->stream));
        else CU(cudaMemcpyAsync(ctx->out.p, d_out, (size_t)n_valid * 40, cudaMemcpyDeviceToDevice, ctx->stream));
        if (flag) CU(cudaMemcpyAsync(flag, d_flag, (size_t)n_valid * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

// ------------------------------------------------------------------ first guess (SURVEY 8f rank 1)
namespace {
struct HostGrid {
    std::vector<double> x, y;
    std::vector<int> start, index;
    double x0 = 0, y0 = 0, cell = 1;
    int nx = 1, ny = 1;
};
// uniform hash grid, ~2 points per cell, points sorted by cell (counting sort)
void build_grid(const double *px, const double *py, int n, HostGrid &g) {
    double xmin = 1e300, xmax = -1e300, ymin = 1e300, ymax = -1e300;
    for (int i = 0; i < n; ++i) { xmin = std::min(xmin, px[i]); xmax = std::max(xmax, px[i]); ymin = std::min(ymin, py[i]); ymax = std::max(ymax, py[i]); }
    if (n == 0) { xmin = ymin = 0; xmax = ymax = 1; }
    const double w = std::max(xmax - xmin, 1.0), h = std::max(ymax - ymin, 1.0);
    g.cell = std::max(std::sqrt(w * h * 2.0 / std::max(n, 1)), 1.0);
    g.nx = std::min(2048, std::max(1, (int)std::ceil(w / g.cell) + 1));
    g.ny = std::min(2048, std::max(1, (int)std::ceil(h / g.cell) + 1));
    g.cell = std::max(g.cell, std::max(w / (g.nx - 0.5), h / (g.ny - 0.5)));
    g.x0 = xmin; g.y0 = ymin;
    const double inv = 1.0 / g.cell;
    auto cell_of = [&](double v, double v0, int m) { int c = (int)std::floor((v - v0) * inv); return c < 0 ? 0 : (c >= m ? m - 1 : c); };
    std::vector<int> cid((size_t)n);
    g.start.assign((size_t)g.nx * g.ny + 1, 0);
    for (int i = 0; i < n; ++i) { cid[(size_t)i] = cell_of(py[i], g.y0, g.ny) * g.nx + cell_of(px[i], g.x0, g.nx); ++g.start[(size_t)cid[(size_t)i] + 1]; }
    for (size_t c = 0; c + 1 < g.start.size(); ++c) g.start[c + 1] += g.start[c];
    std::vector<int> fill(g.start.begin(), g.start.end() - 1);
    g.x.resize((size_t)n); g.y.resize((size_t)n); g.index.resize((size_t)n);
    for (int i = 0; i < n; ++i) { const int k = fill[(size_t)cid[(size_t)i]]++; g.x[(size_t)k] = px[i]; g.y[(size_t)k] = py[i]; g.index[(size_t)k] = i; }
}
// convex hull (Andrew's monotone chain), counter-clockwise, collinear points dropped
void convex_hull(const double *px, const double *py, int n, std::vector<int> &hull) {
    std::vector<int> idx((size_t)n);
    for (int i = 0; i < n; ++i) idx[(size_t)i] = i;
    std::sort(idx.begin(), idx.end(), [&](int a, int b) { return px[a] < px[b] || (px[a] == px[b] && py[a] < py[b]); });
    auto cross = [&](int o, int a, int b) { return (px[a] - px[o]) * (py[b] - py[o]) - (py[a] - py[o]) * (px[b] - px[o]); };
    hull.assign((size_t)2 * n + 2, 0);
    int k = 0;
    for (int i = 0; i < n; ++i) { while (k >= 2 && cross(hull[(size_t)k - 2], hull[(size_t)k - 1], idx[(size_t)i]) <= 0) --k; hull[(size_t)k++] = idx[(size_t)i]; }
    for (int i = n - 2, t = k + 1; i >= 0; --i) { while (k >= t && cross(hull[(size_t)k - 2], hull[(size_t)k - 1], idx[(size_t)i]) <= 0) --k; hull[(size_t)k++] = idx[(size_t)i]; }
    hull.resize((size_t)std::max(0, k - 1));
}
}  // namespace

int sid_first_guess(sid_ctx *ctx, int n_src, const double *sx, const double *sy, const double *vx, const double *vy,
                    int n_seed, const double *kx, const double *ky, int64_t n_q, const double *qx, const double *qy,
                    double *out_vx, double *out_vy, double *out_dist, int32_t *out_flag) {
    if (!ctx) return SID_EINVAL;
    if (n_src < 0 || n_seed < 0 || n_q < 0 || (n_src > 0 && (!sx || !sy || !vx || !vy)) || (n_seed > 0 && (!kx || !ky)) ||
        (n_q > 0 && (!qx || !qy || !out_vx || !out_vy || !out_dist || !out_flag)))
        return fail(ctx, SID_EINVAL, "bad first-guess arguments");
    if (n_q == 0) return SID_OK;
    CU(cudaSetDevice(ctx->device));
    HostGrid gs, gk;
    build_grid(sx, sy, n_src, gs);
    build_grid(kx, ky, n_seed, gk);
    std::vector<int> hull;
    if (n_src >= 3) convex_hull(sx, sy, n_src, hull);
    const int nh = (int)hull.size();
    std::vector<double> hx((size_t)nh), hy((size_t)nh);
    double bx0 = 1e300, bx1 = -1e300, by0 = 1e300, by1 = -1e300;      // the hull's bounding box is the sources'
    for (int i = 0; i < nh; ++i) {
        hx[(size_t)i] = sx[hull[(size_t)i]]; hy[(size_t)i] = sy[hull[(size_t)i]];
        bx0 = std::min(bx0, hx[(size_t)i]); bx1 = std::max(bx1, hx[(size_t)i]); by0 = std::min(by0, hy[(size_t)i]); by1 = std::max(by1, hy[(size_t)i]);
    }
    std::vector<double> hband((size_t)nh);                             // SciPy's band around every hull edge (sid_fg_kernel.cuh)
    for (int i = 0; i < nh; ++i) {
        const int j = i + 1 == nh ? 0 : i + 1;
        hband[(size_t)i] = FG_HULL_BAND_EPS * std::hypot(bx1 - bx0, by1 - by0) * std::hypot(hx[(size_t)j] - hx[(size_t)i], hy[(size_t)j] - hy[(size_t)i]);
    }
    // one staging block: everything the kernel reads, 256-byte aligned pieces
    struct Piece { const void *src; size_t bytes; size_t off; };
    std::vector<Piece> pieces;
    size_t total = 0;
    auto add = [&](const void *p, size_t bytes) { pieces.push_back({p, bytes, total}); total += (bytes + 255) & ~(size_t)255; return pieces.size() - 1; };
    const size_t i_sx = add(gs.x.data(), (size_t)n_src * 8), i_sy = add(gs.y.data(), (size_t)n_src * 8);
    const size_t i_ss = add(gs.start.data(), gs.start.size() * 4), i_si = add(gs.index.data(), (size_t)n_src * 4);
    const size_t i_vx = add(vx, (size_t)n_src * 8), i_vy = add(vy, (size_t)n_src * 8);
    const size_t i_hx = add(hx.data(), (size_t)nh * 8), i_hy = add(hy.data(), (size_t)nh * 8), i_hi = add(hull.data(), (size_t)nh * 4);
    const size_t i_hb = add(hband.data(), (size_t)nh * 8);
    const size_t i_kx = add(gk.x.data(), (size_t)n_seed * 8), i_ky = add(gk.y.data(), (size_t)n_seed * 8);
    const size_t i_ks = add(gk.start.data(), gk.start.size() * 4), i_ki = add(gk.index.data(), (size_t)n_seed * 4);
    const size_t i_qx = add(qx, (size_t)n_q * 8), i_qy = add(qy, (size_t)n_q * 8);
    const size_t o_vx = total; total += ((size_t)n_q * 8 + 255) & ~(size_t)255;
    const size_t o_vy = total; total += ((size_t)n_q * 8 + 255) & ~(size_t)255;
    const size_t o_d = total; total += ((size_t)n_q * 8 + 255) & ~(size_t)255;
    const size_t o_f = total; total += ((size_t)n_q * 4 + 255) & ~(size_t)255;
    int rc = reserve(ctx, ctx->fg, total);
    if (rc) return rc;
    char *base = (char *)ctx->fg.p;
    for (const Piece &pc : pieces)
        if (pc.bytes) CU(cudaMemcpyAsync(base + pc.off, pc.src, pc.bytes, cudaMemcpyHostToDevice, ctx->stream));
    FgArgs a;
    memset(&a, 0, sizeof a);
    auto at = [&](size_t i) { return base + pieces[i].off; };
    a.src.x = (const double *)at(i_sx); a.src.y = (const double *)at(i_sy); a.src.start = (const int *)at(i_ss); a.src.index = (const int *)at(i_si);
    a.src.x0 = gs.x0; a.src.y0 = gs.y0; a.src.cell = gs.cell; a.src.inv_cell = 1.0 / gs.cell; a.src.nx = gs.nx; a.src.ny = gs.ny; a.src.n = n_src;
    a.vx = (const double *)at(i_vx); a.vy = (const double *)at(i_vy);
    a.hx = (const double *)at(i_hx); a.hy = (const double *)at(i_hy); a.hidx = (const int *)at(i_hi); a.nh = nh;
    a.hband = (const double *)at(i_hb);
    a.seed.x = (const double *)at(i_kx); a.seed.y = (const double *)at(i_ky); a.seed.start = (const int *)at(i_ks); a.seed.index = (const int *)at(i_ki);
    a.seed.x0 = gk.x0; a.seed.y0 = gk.y0; a.seed.cell = gk.cell; a.seed.inv_cell = 1.0 / gk.cell; a.seed.nx = gk.nx; a.seed.ny = gk.ny; a.seed.n = n_seed;
    a.nq = n_q; a.qx = (const double *)at(i_qx); a.qy = (const double *)at(i_qy);
    a.out_vx = (double *)(base + o_vx); a.out_vy = (double *)(base + o_vy); a.out_dist = (double *)(base + o_d); a.out_flag = (int *)(base + o_f);
    first_guess_kernel<<<(unsigned)((n_q + 127) / 128), 128, 0, ctx->stream>>>(a);
    ctx->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_vx, base + o_vx, (size_t)n_q * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(out_vy, base + o_vy, (size_t)n_q * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(out_dist, base + o_d, (size_t)n_q * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(out_flag, base + o_f, (size_t)n_q * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

// ------------------------------------------------------------------ single-call entry points

int sid_get_template(sid_ctx *ctx, const uint8_t *img, int rows, int cols, int64_t pitch, double c, double r,
                     const double *angle_tab, int s, int rot_order, uint8_t *out) {
    if (!ctx) return SID_EINVAL;
    if (!img || !out || !angle_tab || s <= 0 || s > 4096) return fail(ctx, SID_EINVAL, "bad get_template arguments");
    if (rot_order != 0 && rot_order != 1) return fail(ctx, SID_EUNSUPPORTED, "rot_order must be 0 or 1");
    CU(cudaSetDevice(ctx->device));
    long long dp;
    int rc = upload_image(ctx, ctx->img1, dp, img, rows, cols, pitch, cudaMemcpyHostToDevice);
    ctx->have_pair = false;
    if (rc) return rc;
    const size_t tb = (size_t)s * s;
    if ((rc = reserve(ctx, ctx->misc, tb + 64 + 4 * 8 + 16))) return rc;
    uint8_t *d_t = (uint8_t *)ctx->misc.p;
    const size_t off_tab = (tb + 63) / 64 * 64;
    double *d_tab = (double *)(d_t + off_tab);
    uint32_t *d_stats = (uint32_t *)(d_tab + 4);
    CU(cudaMemcpyAsync(d_tab, angle_tab, 32, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(d_stats, 0, 12, ctx->stream));
    templates_kernel<<<1, 256, 0, ctx->stream>>>((const uint8_t *)ctx->img1.p, rows, cols, dp, c, r, d_tab, s, rot_order, d_t, d_stats);
    ctx->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, d_t, tb, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return SID_OK;
}

// NCC map of a device image/template pair into d_out; isum/isq/tstats are device scratch.
static int match_on_device(sid_ctx *ctx, const uint8_t *d_img, int H, int W, long long pitch, const uint8_t *d_tpl,
                           int th, int tw, long long tp, uint32_t *d_isum, uint32_t *d_isq, bool integrals_ready,
                           uint32_t *d_tstats, float *d_out) {
    const int RH = H - th + 1, RW = W - tw + 1;
    if (!integrals_ready) {
        integral_rows_kernel<<<(H + 1 + 127) / 128, 128, 0, ctx->stream>>>(d_img, H, W, pitch, d_isum, d_isq);
        integral_cols_kernel<<<(W + 1 + 127) / 128, 128, 0, ctx->stream>>>(H, W, d_isum, d_isq);
        ctx->launches += 2;
    }
    CU(cudaMemsetAsync(d_tstats, 0, 8, ctx->stream));
    template_sums_kernel<<<std::min(64, (th * tw + 255) / 256), 256, 0, ctx->stream>>>(d_tpl, th, tw, tp, d_tstats);
    MtArgs a;
    a.img = d_img; a.H = H; a.W = W; a.pitch = pitch;
    a.tpl = d_tpl; a.th = th; a.tw = tw; a.tp = tp;
    a.isum = d_isum; a.isq = d_isq; a.tstats = d_tstats;
    const double area = (double)th * (double)tw;
    a.inv_area = 1.0 / area; a.sqrt_inv_area = std::sqrt(a.inv_area);
    a.out = d_out;
    a.tpw = (tw + 15) / 16 * 4;
    int n16 = (MT_COLS + tw + 3 + 15) / 16 + 1;
    if ((n16 & 1) == 0) ++n16;
    a.wpw = n16 * 4;
    const size_t smem = ((size_t)(MT_ROWS + th - 1) * a.wpw + PM_WIN_SLACK + (size_t)th * a.tpw) * 4;
    if (smem > (size_t)ctx->max_smem_optin) return fail(ctx, SID_EUNSUPPORTED, "template too large for match_template");
    if (int arc = allow_max_smem(ctx, (const void *)match_template_kernel)) return arc;
    dim3 grid((RW + MT_COLS - 1) / MT_COLS, (RH + MT_ROWS - 1) / MT_ROWS);
    match_template_kernel<<<grid, 256, smem, ctx->stream>>>(a);
    ctx->launches += 2;
    CU(cudaGetLastError());
    return SID_OK;
}

int sid_match_template(sid_ctx *ctx, const uint8_t *img, int H, int W, int64_t pitch, const uint8_t *tpl,
                       int th, int tw, int64_t tpitch, int method, float *out) {
    if (!ctx) return SID_EINVAL;
    if (method != SID_TM_CCOEFF_NORMED) return fail(ctx, SID_EUNSUPPORTED, "only TM_CCOEFF_NORMED (5) is implemented");
    if (!img || !tpl || !out || th <= 0 || tw <= 0 || H < th || W < tw || pitch < W || tpitch < tw)
        return fail(ctx, SID_EINVAL, "bad match_template arguments (image must not be smaller than the template)");
    if ((long long)th * tw > 32768) return fail(ctx, SID_EUNSUPPORTED, "template area above 32768 pixels");
    CU(cudaSetDevice(ctx->device));
    long long dp;
    int rc = upload_image(ctx, ctx->img2, dp, img, H, W, pitch, cudaMemcpyHostToDevice);
    ctx->have_pair = false;
    if (rc) return rc;
    const int RH = H - th + 1, RW = W - tw + 1;
    const size_t int_bytes = (size_t)(H + 1) * (W + 1) * 4;
    const size_t tpl_bytes = ((size_t)th * tw + 255) / 256 * 256;
    const size_t out_bytes = (size_t)RH * RW * 4;
    if ((rc = reserve(ctx, ctx->misc, 2 * int_bytes + tpl_bytes + out_bytes + 1024))) return rc;
    unsigned char *base = (unsigned char *)ctx->misc.p;
    uint32_t *d_isum = (uint32_t *)base, *d_isq = (uint32_t *)(base + int_bytes);
    uint8_t *d_tpl = base + 2 * int_bytes;
    float *d_out = (float *)(base + 2 * int_bytes + tpl_bytes);
    uint32_t *d_ts = (uint32_t *)(base + 2 * int_bytes + tpl_bytes + out_bytes);
    d_ts = (uint32_t *)(((uintptr_t)d_ts + 15) & ~(uintptr_t)15);
    CU(cudaMemcpy2DAsync(d_tpl, (size_t)tw, tpl, (size_t)tpitch, (size_t)tw, (size_t)th, cudaMemcpyHostToDevice, ctx->stream));
    rc = match_on_device(ctx, (const uint8_t *)ctx->img2.p, H, W, dp, d_tpl, th, tw, tw, d_isum, d_isq, false, d_ts, d_out);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    return SID_OK;
}

int sid_knn_hamming2(sid_ctx *ctx, const uint8_t *d1, int n1, const uint8_t *d2, int n2, int desc_bytes,
                     int32_t *idx, int32_t *dist) {
    if (!ctx) return SID_EINVAL;
    if (desc_bytes != 32) return fail(ctx, SID_EUNSUPPORTED, "only 32-byte (ORB) descriptors are implemented");
    if (n1 < 0 || n2 < 0 || (n1 > 0 && (!d1 || !idx || !dist)) || (n2 > 0 && !d2)) return fail(ctx, SID_EINVAL, "bad knn arguments");
    if (n1 == 0) return SID_OK;
    if (n2 == 0) { for (int k = 0; k < 2 * n1; ++k) { idx[k] = -1; dist[k] = -1; } return SID_OK; }
    CU(cudaSetDevice(ctx->device));
    const int qblocks = (n1 + KNN_THREADS - 1) / KNN_THREADS;
    int nseg = (ctx->sm_count * 8 + qblocks - 1) / qblocks;               // >= 8 CTAs per SM in flight
    nseg = std::max(1, std::min(nseg, std::min(64, (n2 + KNN_TILE - 1) / KNN_TILE)));
    int seg_len = ((n2 + nseg - 1) / nseg + KNN_TILE - 1) / KNN_TILE * KNN_TILE;
    nseg = (n2 + seg_len - 1) / seg_len;
    const size_t b1 = (size_t)n1 * 32, b2 = (size_t)n2 * 32, bp = (size_t)nseg * n1 * sizeof(Top2), bo = (size_t)n1 * 2 * 4;
    const size_t o2 = (b1 + 255) / 256 * 256, op = o2 + (b2 + 255) / 256 * 256, oi = op + (bp + 255) / 256 * 256, od = oi + (bo + 255) / 256 * 256;
    int rc = reserve(ctx, ctx->misc, od + bo + 256);
    if (rc) return rc;
    unsigned char *base = (unsigned char *)ctx->misc.p;
    CU(cudaMemcpyAsync(base, d1, b1, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(base + o2, d2, b2, cudaMemcpyHostToDevice, ctx->stream));
    knn_hamming2_kernel<<<dim3((unsigned)qblocks, (unsigned)nseg), KNN_THREADS, 0, ctx->stream>>>(
        (const uint4 *)base, n1, (const uint4 *)(base + o2), n2, seg_len, (Top2 *)(base + op));
    knn_merge_kernel<<<(n1 + 255) / 256, 256, 0, ctx->stream>>>((const Top2 *)(base + op), n1, nseg, (int *)(base + oi), (int *)(base + od));
    ctx->launches += 2;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(idx, base + oi, bo, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(dist, base + od, bo, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    return SID_OK;
}

int sid_deformation(sid_ctx *ctx, int n, const double *x, const double *y, const double *u, const double *v,
                    int m, const int32_t *tri, const double *area_in,
                    double *e1, double *e2, double *e3, double *area, double *perim) {
    if (!ctx) return SID_EINVAL;
    if (n < 0 || m < 0 || (n > 0 && (!x || !y || !u || !v)) || (m > 0 && (!tri || !e1 || !e2 || !e3 || !area || !perim)))
        return fail(ctx, SID_EINVAL, "bad deformation arguments");
    if (m == 0) return SID_OK;
    CU(cudaSetDevice(ctx->device));
    const size_t bn = ((size_t)n * 8 + 255) / 256 * 256, bm = ((size_t)m * 8 + 255) / 256 * 256;
    const size_t bt = ((size_t)m * 12 + 255) / 256 * 256;
    int rc = reserve(ctx, ctx->misc, 4 * bn + bt + 6 * bm + 256);
    if (rc) return rc;
    unsigned char *base = (unsigned char *)ctx->misc.p;
    DeforArgs a;
    const double *src[4] = {x, y, u, v};
    double *dn[4];
    for (int k = 0; k < 4; ++k) {
        dn[k] = (double *)(base + k * bn);
        if (n > 0) CU(cudaMemcpyAsync(dn[k], src[k], (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    a.x = dn[0]; a.y = dn[1]; a.u = dn[2]; a.v = dn[3];
    int32_t *dt = (int32_t *)(base + 4 * bn);
    CU(cudaMemcpyAsync(dt, tri, (size_t)m * 12, cudaMemcpyHostToDevice, ctx->stream));
    a.tri = dt;
    double *dm = (double *)(base + 4 * bn + bt);
    a.e1 = dm; a.e2 = (double *)((char *)dm + bm); a.e3 = (double *)((char *)dm + 2 * bm);
    a.area = (double *)((char *)dm + 3 * bm); a.perim = (double *)((char *)dm + 4 * bm);
    double *dain = (double *)((char *)dm + 5 * bm);
    a.area_in = nullptr;
    if (area_in) {
        CU(cudaMemcpyAsync(dain, area_in, (size_t)m * 8, cudaMemcpyHostToDevice, ctx->stream));
        a.area_in = dain;
    }
    a.n = n; a.m = m;
    deformation_kernel<<<(m + 255) / 256, 256, 0, ctx->stream>>>(a);
    ctx->launches += 1;
    CU(cudaGetLastError());
    double *dst[5] = {e1, e2, e3, area, perim};
    for (int k = 0; k < 5; ++k)
        CU(cudaMemcpyAsync(dst[k], (char *)dm + k * bm, (size_t)m * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    return SID_OK;
}

int sid_get_hessian(sid_ctx *ctx, const float *ccm, int rows, int cols, unsigned flags, float *out) {
    if (!ctx) return SID_EINVAL;
    if (!ccm || !out || rows < 2 || cols < 2) return fail(ctx, SID_EINVAL, "get_hessian needs a map of at least 2 x 2");
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)rows * cols, b = n * 4;
    int rc = reserve(ctx, ctx->misc, 4 * b + 64);
    if (rc) return rc;
    float *d = (float *)ctx->misc.p;
    CU(cudaMemcpyAsync(d, ccm, b, cudaMemcpyHostToDevice, ctx->stream));
    HesArgs a;
    a.ccm = d; a.rows = rows; a.cols = cols; a.flags = flags; gaussian_weights(a.gw);
    a.tmp_a = d + n; a.tmp_b = d + 2 * n; a.out = d + 3 * n;
    hessian_map_kernel<<<1, 1024, 0, ctx->stream>>>(a);
    ctx->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, a.out, b, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    return SID_OK;
}

int sid_rotate_and_match(sid_ctx *ctx, const uint8_t *img1, int rows1, int cols1, int64_t pitch1, double c1,
                         double r1, int img_size, const uint8_t *image2, int H, int W, int64_t pitch2,
                         int n_angles, const double *angle_tab, int rot_order, unsigned flags, int mtype,
                         int *valid, double *dc, double *dr, int *best_angle_idx, float *best_r, float *best_h,
                         float *best_result, uint8_t *best_template) {
    int rc = check_common(ctx, img_size, n_angles, angle_tab, rot_order, mtype);
    if (rc) return rc;
    if (!valid || !dc || !dr || !best_angle_idx || !best_r || !best_h) return fail(ctx, SID_EINVAL, "null output pointer");
    if (flags & SID_PEAKS) return fail(ctx, SID_EUNSUPPORTED, "SID_PEAKS is for the batched sid_run* calls");
    if (flags & SID_UNCERT) return fail(ctx, SID_EUNSUPPORTED, "SID_UNCERT is for the batched sid_run* calls");
    const int s = img_size;
    if (!img1 || !image2 || H < s + 1 || W < s + 1)
        return fail(ctx, SID_EINVAL, "search window must exceed the template by at least one pixel in each axis");
    CU(cudaSetDevice(ctx->device));
    long long dp1, dp2;
    ctx->have_pair = false;
    if ((rc = upload_image(ctx, ctx->img1, dp1, img1, rows1, cols1, pitch1, cudaMemcpyHostToDevice))) return rc;
    if ((rc = upload_image(ctx, ctx->img2, dp2, image2, H, W, pitch2, cudaMemcpyHostToDevice))) return rc;
    const int RH = H - s + 1, RW = W - s + 1;
    const size_t rr = (size_t)RH * RW;
    const size_t int_bytes = ((size_t)(H + 1) * (W + 1) * 4 + 255) / 256 * 256;
    const size_t tpl_bytes = ((size_t)n_angles * s * s + 255) / 256 * 256;
    const size_t map_bytes = (rr * 4 + 255) / 256 * 256;
    const size_t small = 4096 + (size_t)n_angles * 64;
    if ((rc = reserve(ctx, ctx->misc, 2 * int_bytes + tpl_bytes + ((size_t)n_angles + 3) * map_bytes + small))) return rc;
    unsigned char *base = (unsigned char *)ctx->misc.p;
    uint32_t *d_isum = (uint32_t *)base, *d_isq = (uint32_t *)(base + int_bytes);
    uint8_t *d_tpl = base + 2 * int_bytes;
    float *d_maps = (float *)(base + 2 * int_bytes + tpl_bytes);     // one map per angle, then tmp_a, tmp_b, hes
    unsigned char *sm = base + 2 * int_bytes + tpl_bytes + ((size_t)n_angles + 3) * map_bytes;
    double *d_tab = (double *)sm;                                     // n_angles * 4 doubles
    uint32_t *d_stats = (uint32_t *)(sm + (size_t)n_angles * 32);     // n_angles * 3
    uint32_t *d_ts = d_stats + (size_t)n_angles * 3 + 4;              // 2
    unsigned long long *d_key = (unsigned long long *)(((uintptr_t)(d_ts + 4) + 15) & ~(uintptr_t)15);   // one per angle
    float *d_peak = (float *)(d_key + n_angles + 1);
    double *d_offsets = (double *)(d_peak + 2);                       // 2, with SID_SUBPIXEL
    const size_t mstride = map_bytes / 4;

    CU(cudaMemcpyAsync(d_tab, angle_tab, (size_t)n_angles * 32, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(d_stats, 0, (size_t)n_angles * 12, ctx->stream));
    templates_kernel<<<n_angles, 256, 0, ctx->stream>>>((const uint8_t *)ctx->img1.p, rows1, cols1, dp1, c1, r1, d_tab, s,
                                                       rot_order, d_tpl, d_stats);
    ctx->launches += 1;
    std::vector<uint32_t> hstats((size_t)n_angles * 3);
    CU(cudaMemcpyAsync(hstats.data(), d_stats, (size_t)n_angles * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    *valid = 1;
    for (int a = 0; a < n_angles; ++a) if (hstats[(size_t)a * 3 + 2]) *valid = 0;
    // SID_MASKED: a template holds a 0 pixel; the masked rule takes the point when every template qualifies
    std::vector<long long> mstat;                                     // n, St, Stt per angle
    if (!*valid && (flags & SID_MASKED)) {
        std::vector<uint8_t> htpl((size_t)n_angles * s * s);
        CU(cudaMemcpy(htpl.data(), d_tpl, htpl.size(), cudaMemcpyDeviceToHost));
        mstat.resize((size_t)n_angles * 3);
        bool ok = true;
        for (int a = 0; a < n_angles; ++a) {
            long long cnt = 0;
            for (int k = 0; k < s * s; ++k) cnt += htpl[(size_t)a * s * s + k] != 0;
            long long *m = &mstat[(size_t)a * 3];
            m[0] = cnt; m[1] = hstats[(size_t)a * 3]; m[2] = hstats[(size_t)a * 3 + 1];
            ok = ok && masked_template_ok(s, m[0], m[1], m[2]);
        }
        if (ok) *valid = 2;
        else mstat.clear();
    }
    if (!*valid) {
        *dc = NAN; *dr = NAN; *best_angle_idx = -1; *best_r = NAN; *best_h = NAN;
        return SID_OK;
    }
    // every angle's map and arg-max are enqueued back to back; ONE read-back of the keys decides the winner (strict '>' in
    // angle order, like the reference loop pmlib.py:155-166)
    for (int a = 0; a < n_angles; ++a) {
        float *d_map = d_maps + (size_t)a * mstride;
        if (!mstat.empty()) {
            const long long *m = &mstat[(size_t)a * 3];
            const unsigned grid = (unsigned)std::min<size_t>((rr + 255) / 256, (size_t)ctx->sm_count * 8);
            masked_map_kernel<<<grid, 256, 0, ctx->stream>>>((const uint8_t *)ctx->img2.p, H, W, dp2, d_tpl + (size_t)a * s * s, s,
                                                           m[0], m[1], m[2], d_map);
            ctx->launches += 1;
            CU(cudaGetLastError());
        } else {
            rc = match_on_device(ctx, (const uint8_t *)ctx->img2.p, H, W, dp2, d_tpl + (size_t)a * s * s, s, s, s,
                                 d_isum, d_isq, a > 0, d_ts, d_map);
            if (rc) return rc;
        }
        argmax_kernel<<<1, 1024, 0, ctx->stream>>>(d_map, (int)rr, d_key + a);
        ctx->launches += 1;
    }
    std::vector<unsigned long long> keys((size_t)n_angles, 0ull);
    CU(cudaMemcpyAsync(keys.data(), d_key, (size_t)n_angles * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    float br = -INFINITY; int ba = -1; uint32_t bidx = 0;
    for (int a = 0; a < n_angles; ++a) {
        const unsigned long long key = keys[(size_t)a];
        const uint32_t hi = (uint32_t)(key >> 32);
        const uint32_t ubits = (hi & 0x80000000u) ? (hi & 0x7fffffffu) : ~hi;
        float v; memcpy(&v, &ubits, 4);
        if (v > br) { br = v; ba = a; bidx = 0xffffffffu - (uint32_t)(key & 0xffffffffull); }
    }
    if (ba < 0) {
        *valid = 0; *dc = NAN; *dr = NAN; *best_angle_idx = -1; *best_r = NAN; *best_h = NAN;
        return SID_OK;
    }
    PeakArgs pa;
    pa.best = d_maps + (size_t)ba * mstride; pa.rows = RH; pa.cols = RW; pa.idx = (int)bidx; pa.r = br; pa.flags = flags;
    gaussian_weights(pa.gw);
    pa.tmp_a = d_maps + (size_t)n_angles * mstride; pa.tmp_b = pa.tmp_a + mstride; pa.hes = pa.tmp_b + mstride; pa.out = d_peak;
    pa.offsets = d_offsets;
    peak_stats_kernel<<<1, 1024, 0, ctx->stream>>>(pa);
    ctx->launches += 1;
    float hp[2];
    double offsets[2] = {0.0, 0.0};
    CU(cudaMemcpyAsync(hp, d_peak, 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (flags & SID_SUBPIXEL) CU(cudaMemcpyAsync(offsets, d_offsets, 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (best_result) CU(cudaMemcpyAsync(best_result, pa.best, rr * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (best_template) CU(cudaMemcpyAsync(best_template, d_tpl + (size_t)ba * s * s, (size_t)s * s, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaGetLastError());
    const int bi = (int)(bidx / (uint32_t)RW), bj = (int)(bidx % (uint32_t)RW);
    *dr = (double)bi - (double)(H - s) / 2.0;
    *dc = (double)bj - (double)(W - s) / 2.0;
    if (flags & SID_SUBPIXEL) {         // the batched kernels' order: (unrefined) + offset
        *dr = *dr + offsets[1];
        *dc = *dc + offsets[0];
    }
    *best_angle_idx = ba;
    *best_r = hp[0];
    *best_h = hp[1];
    return SID_OK;
}

}  // extern "C"
