/*
 * mcc_oracle.c -- TEST INFRASTRUCTURE ONLY (not part of the product).
 *
 * Plain-C, single-file CPU restatement of the pattern-matching (MCC) hot path of
 * nansencenter/sea_ice_drift v0.7.1, written from the behaviour of the reference,
 * not from its text.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline leg may load this library; the product path never does.
 *
 * Parity status: PINNED against the reference executed live in the build
 * container (oracle/ref_import.py + oracle/make_golden.py -> tests/golden/),
 * because the reference's own tests hold no numeric golden values for this
 * path (reference sea_ice_drift/tests.py:296-346 assert shapes only).
 *
 * What each function follows (paths under /root/reference/):
 *   sido_get_template      sea_ice_drift/pmlib.py:89-115  (+ scipy 1.18.1
 *                          ndimage.affine_transform, order 0/1, mode=constant,
 *                          cval=0, uint8 output; arithmetic pinned empirically)
 *   sido_match_template    sea_ice_drift/pmlib.py:156 -> cv2.matchTemplate(
 *                          TM_CCOEFF_NORMED), OpenCV 4.13 imgproc/templmatch.cpp
 *                          (third-party, un-vendored); the correlation numerator is
 *                          computed EXACTLY in integers here, whereas OpenCV's
 *                          DFT/IPP float32 path carries ~1e-6 noise.
 *   sido_hessian           sea_ice_drift/pmlib.py:36-59   (np.gradient x3, hypot,
 *                          median, std; optional gaussian_filter sigma=1)
 *   sido_rotate_and_match  sea_ice_drift/pmlib.py:117-174
 *   sido_use_mcc_batch     sea_ice_drift/pmlib.py:176-247, 436-448 (the Pool map)
 *
 * The per-angle table `tab` (4 doubles per angle: cos, sin, tcdot0, tcdot1) is
 * computed by the caller with NumPy exactly as pmlib.py:105-110 does, so that
 * libm differences never enter:   a = radians(angle - alpha0)
 *   T = [[cos a, -sin a], [sin a, cos a]];  tcdot = [tc, tc] . T, tc = int(s/2.)+1
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

#define SIDO_OK 0
#define SIDO_EINVAL -1
#define SIDO_ENOMEM -2

/* ------------------------------------------------------------------ template */

/* pmlib.py:105-113.  Output pixel (i,j) samples img1 at
 *   row = off0 + i*cos + j*sin,  col = off1 + i*(-sin) + j*cos   (left to right, no FMA)
 * with off = [r, c] - tcdot.  Outside [0, dim-1] -> 0.
 * order 0: nearest = floor(x + 0.5).  order 1: bilinear in double, then
 * floor(v + 0.5) clipped to [0,255]. */
int sido_get_template(const uint8_t *img, int rows, int cols, int64_t pitch,
                      double c, double r, const double *tab, int s, int order,
                      uint8_t *out)
{
    if (!img || !out || !tab || s <= 0 || rows <= 0 || cols <= 0) return SIDO_EINVAL;
    if (order != 0 && order != 1) return SIDO_EINVAL;
    const double cs = tab[0], sn = tab[1];
    const double off0 = r - tab[2], off1 = c - tab[3];
    const double m00 = cs, m01 = sn, m10 = -sn, m11 = cs;
    for (int i = 0; i < s; ++i) {
        for (int j = 0; j < s; ++j) {
            volatile double t0 = (double)i * m00, t1 = (double)j * m01;
            volatile double t2 = (double)i * m10, t3 = (double)j * m11;
            double row = off0 + t0; row = row + t1;
            double col = off1 + t2; col = col + t3;
            uint8_t v = 0;
            if (row >= 0.0 && row <= (double)(rows - 1) && col >= 0.0 && col <= (double)(cols - 1)) {   /* NaN: outside */
                if (order == 0) {
                    int64_t ri = (int64_t)floor(row + 0.5), ci = (int64_t)floor(col + 0.5);
                    if (ri > rows - 1) ri = rows - 1;
                    if (ci > cols - 1) ci = cols - 1;
                    v = img[ri * pitch + ci];
                } else {
                    double fr = floor(row), fc = floor(col);
                    int64_t r0 = (int64_t)fr, c0 = (int64_t)fc;
                    double fy = row - fr, fx = col - fc;
                    double wy0 = 1.0 - fy, wy1 = fy, wx0 = 1.0 - fx, wx1 = fx;
                    int64_t r1 = r0 + 1 > rows - 1 ? rows - 1 : r0 + 1;
                    int64_t c1 = c0 + 1 > cols - 1 ? cols - 1 : c0 + 1;
                    volatile double p;
                    double t = 0.0;
                    p = (double)img[r0 * pitch + c0] * wy0; p = p * wx0; t = t + p;
                    p = (double)img[r0 * pitch + c1] * wy0; p = p * wx1; t = t + p;
                    p = (double)img[r1 * pitch + c0] * wy1; p = p * wx0; t = t + p;
                    p = (double)img[r1 * pitch + c1] * wy1; p = p * wx1; t = t + p;
                    t = t > 0.0 ? t + 0.5 : 0.0;
                    if (t > 255.0) t = 255.0;
                    v = (uint8_t)t;
                }
            }
            out[i * s + j] = v;
        }
    }
    return SIDO_OK;
}

/* ------------------------------------------------------------------ NCC */

/* TM_CCOEFF_NORMED as OpenCV's common_matchTemplate evaluates it, with an exact
 * integer correlation numerator:
 *   num  = corr - winSum * mean(T)
 *   t    = sqrt(max(winSqSum - winSum^2/N, 0)) * ||T - mean(T)||
 *   out  = num/t if |num| < t;  +-1 if |num| < 1.125 t;  else 0     (float32)
 * and the whole map = 1 when var(T) < DBL_EPSILON. */
int sido_match_template(const uint8_t *img, int H, int W, int64_t pitch,
                        const uint8_t *tpl, int th, int tw, int64_t tpitch,
                        float *out)
{
    if (!img || !tpl || !out || th <= 0 || tw <= 0 || H < th || W < tw) return SIDO_EINVAL;
    const int RH = H - th + 1, RW = W - tw + 1;
    /* template statistics (cv::meanStdDev) */
    int64_t tsum = 0, tsq = 0;
    for (int i = 0; i < th; ++i)
        for (int j = 0; j < tw; ++j) {
            int64_t v = tpl[i * tpitch + j];
            tsum += v; tsq += v * v;
        }
    const double area = (double)th * (double)tw;
    const double invArea = 1.0 / area;
    const double scale = 1.0 / area;
    const double tmean = (double)tsum * scale;
    double tvar = (double)tsq * scale - tmean * tmean;
    if (tvar < 0.0) tvar = 0.0;
    const double tsdv = sqrt(tvar);
    double templNorm = tsdv * tsdv;
    if (templNorm < DBL_EPSILON) {
        for (int k = 0; k < RH * RW; ++k) out[k] = 1.0f;
        return SIDO_OK;
    }
    templNorm = sqrt(templNorm);
    templNorm /= sqrt(invArea);

    /* integral images of the search window (exact) */
    const int IW = W + 1;
    int64_t *isum = (int64_t *)calloc((size_t)(H + 1) * IW, sizeof(int64_t));
    int64_t *isq = (int64_t *)calloc((size_t)(H + 1) * IW, sizeof(int64_t));
    if (!isum || !isq) { free(isum); free(isq); return SIDO_ENOMEM; }
    for (int y = 0; y < H; ++y) {
        int64_t rs = 0, rq = 0;
        for (int x = 0; x < W; ++x) {
            int64_t v = img[y * pitch + x];
            rs += v; rq += v * v;
            isum[(y + 1) * IW + x + 1] = isum[y * IW + x + 1] + rs;
            isq[(y + 1) * IW + x + 1] = isq[y * IW + x + 1] + rq;
        }
    }
    for (int y = 0; y < RH; ++y) {
        for (int x = 0; x < RW; ++x) {
            int64_t corr = 0;
            for (int i = 0; i < th; ++i) {
                const uint8_t *ip = img + (int64_t)(y + i) * pitch + x;
                const uint8_t *tp = tpl + (int64_t)i * tpitch;
                int32_t rowacc = 0;
                for (int j = 0; j < tw; ++j) rowacc += (int32_t)ip[j] * (int32_t)tp[j];
                corr += rowacc;
            }
            int64_t ws = isum[y * IW + x] - isum[y * IW + x + tw] - isum[(y + th) * IW + x] + isum[(y + th) * IW + x + tw];
            int64_t wq = isq[y * IW + x] - isq[y * IW + x + tw] - isq[(y + th) * IW + x] + isq[(y + th) * IW + x + tw];
            double t = (double)ws;
            volatile double tt = t * t;
            double wndMean2 = tt * invArea;
            volatile double tm = t * tmean;
            double num = (double)corr - tm;
            double wndSum2 = (double)wq;
            double diff2 = wndSum2 - wndMean2;
            if (diff2 < 0.0) diff2 = 0.0;
            double thr = 10.0 * (double)FLT_EPSILON * wndSum2;
            if (thr > 0.5) thr = 0.5;
            if (diff2 <= thr) t = 0.0;
            else t = sqrt(diff2) * templNorm;
            if (fabs(num) < t) num /= t;
            else if (fabs(num) < t * 1.125) num = num > 0 ? 1.0 : -1.0;
            else num = 0.0;
            out[y * RW + x] = (float)num;
        }
    }
    free(isum); free(isq);
    return SIDO_OK;
}

/* ------------------------------------------------------------------ Hessian */

static void gradient_axis(const float *f, int rows, int cols, int axis, float *g)
{
    /* np.gradient, unit spacing, edge_order=1, float32 arithmetic */
    if (axis == 0) {
        for (int x = 0; x < cols; ++x) {
            g[x] = f[cols + x] - f[x];
            g[(rows - 1) * cols + x] = f[(rows - 1) * cols + x] - f[(rows - 2) * cols + x];
        }
        for (int y = 1; y < rows - 1; ++y)
            for (int x = 0; x < cols; ++x)
                g[y * cols + x] = (f[(y + 1) * cols + x] - f[(y - 1) * cols + x]) / 2.0f;
    } else {
        for (int y = 0; y < rows; ++y) {
            const float *fr = f + y * cols; float *gr = g + y * cols;
            gr[0] = fr[1] - fr[0];
            gr[cols - 1] = fr[cols - 1] - fr[cols - 2];
            for (int x = 1; x < cols - 1; ++x) gr[x] = (fr[x + 1] - fr[x - 1]) / 2.0f;
        }
    }
}

static int cmp_float(const void *a, const void *b)
{
    float x = *(const float *)a, y = *(const float *)b;
    return (x > y) - (x < y);
}

/* np.median (float32): middle element, or float32 mean of the two middle ones */
static float median_f32(const float *v, int n, float *scratch)
{
    for (int i = 0; i < n; ++i) if (isnan(v[i])) return NAN;
    memcpy(scratch, v, (size_t)n * sizeof(float));
    qsort(scratch, (size_t)n, sizeof(float), cmp_float);
    if (n & 1) return scratch[n / 2];
    volatile float s2 = scratch[n / 2 - 1] + scratch[n / 2];
    return s2 / 2.0f;
}

/* np.std (float32, ddof=0): float32 mean, float32 deviations and squares,
 * sums carried in double (NumPy's float32 pairwise sums differ by <= a few ulp). */
static float std_f32(const float *v, int n)
{
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += (double)v[i];
    float mean = (float)(s / (double)n);
    double q = 0.0;
    for (int i = 0; i < n; ++i) {
        volatile float d = v[i] - mean;
        volatile float d2 = d * d;
        q += (double)d2;
    }
    float var = (float)(q / (double)n);
    return sqrtf(var);
}

/* scipy.ndimage.gaussian_filter(ccm, 1): 9 taps, reflect, axis 0 then axis 1,
 * float32 between the passes, double accumulation. */
static void gaussian_sigma1(const float *in, int rows, int cols, float *out, float *tmp)
{
    double w[9], sum = 0.0;
    for (int k = -4; k <= 4; ++k) { w[k + 4] = exp(-0.5 * (double)(k * k)); sum += w[k + 4]; }
    for (int k = 0; k < 9; ++k) w[k] /= sum;
    /* axis 0 */
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) {
            double acc = w[4] * (double)in[y * cols + x];
            for (int k = 1; k <= 4; ++k) {
                int ya = y - k, yb = y + k;
                /* reflect: (d c b a | a b c d | d c b a) */
                while (ya < 0 || ya >= rows) { if (ya < 0) ya = -ya - 1; if (ya >= rows) ya = 2 * rows - 1 - ya; }
                while (yb < 0 || yb >= rows) { if (yb < 0) yb = -yb - 1; if (yb >= rows) yb = 2 * rows - 1 - yb; }
                acc += w[4 + k] * ((double)in[ya * cols + x] + (double)in[yb * cols + x]);
            }
            tmp[y * cols + x] = (float)acc;
        }
    /* axis 1 */
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) {
            double acc = w[4] * (double)tmp[y * cols + x];
            for (int k = 1; k <= 4; ++k) {
                int xa = x - k, xb = x + k;
                while (xa < 0 || xa >= cols) { if (xa < 0) xa = -xa - 1; if (xa >= cols) xa = 2 * cols - 1 - xa; }
                while (xb < 0 || xb >= cols) { if (xb < 0) xb = -xb - 1; if (xb >= cols) xb = 2 * cols - 1 - xb; }
                acc += w[4 + k] * ((double)tmp[y * cols + xa] + (double)tmp[y * cols + xb]);
            }
            out[y * cols + x] = (float)acc;
        }
}

/* pmlib.py:36-59 */
int sido_hessian(const float *ccm, int rows, int cols, int hes_norm, int hes_smth, float *out)
{
    if (!ccm || !out || rows < 2 || cols < 2) return SIDO_EINVAL;
    const int n = rows * cols;
    float *buf = (float *)malloc((size_t)n * 5 * sizeof(float));
    if (!buf) return SIDO_ENOMEM;
    float *sm = buf, *gy = buf + n, *gx = buf + 2 * n, *d2 = buf + 3 * n, *tmp = buf + 4 * n;
    const float *src = ccm;
    if (hes_smth) { gaussian_sigma1(ccm, rows, cols, sm, tmp); src = sm; }
    gradient_axis(src, rows, cols, 0, gy);      /* dcc_dy */
    gradient_axis(src, rows, cols, 1, gx);      /* dcc_dx */
    gradient_axis(gx, rows, cols, 1, d2);       /* d2cc_dx2 */
    gradient_axis(gy, rows, cols, 0, tmp);      /* d2cc_dy2 */
    for (int k = 0; k < n; ++k) {
        double a = (double)d2[k], b = (double)tmp[k];
        volatile double aa = a * a, bb = b * b;
        out[k] = (float)sqrt(aa + bb);
    }
    if (hes_norm) {
        float med = median_f32(out, n, gy);
        float sd = std_f32(out, n);
        for (int k = 0; k < n; ++k) { volatile float d = out[k] - med; out[k] = d / sd; }
    }
    free(buf);
    return SIDO_OK;
}

/* ------------------------------------------------------------------ rotate_and_match */

/* pmlib.py:117-174.  Returns SIDO_OK; *valid = 0 reproduces the reference's
 * "return 7 x NaN" at the first angle whose template contains a 0 pixel. */
int sido_rotate_and_match(const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                          double c1, double r1, int s,
                          const uint8_t *image2, int H, int W, int64_t pitch2,
                          int n_angles, const double *tab, int order,
                          int hes_norm, int hes_smth, int mcc_norm,
                          int *valid, double *dc, double *dr, int *best_angle_idx,
                          float *best_r, float *best_h,
                          float *best_result /* RH*RW or NULL */,
                          uint8_t *best_template /* s*s or NULL */)
{
    if (s <= 0 || H < s || W < s || n_angles <= 0) return SIDO_EINVAL;
    const int RH = H - s + 1, RW = W - s + 1;
    if (RH < 2 || RW < 2) return SIDO_EINVAL;
    uint8_t *tpl = (uint8_t *)malloc((size_t)s * s * 2);
    float *res = (float *)malloc((size_t)RH * RW * 3 * sizeof(float));
    if (!tpl || !res) { free(tpl); free(res); return SIDO_ENOMEM; }
    uint8_t *btpl = tpl + s * s;
    float *bres = res + RH * RW, *hes = res + 2 * RH * RW;
    float br = -INFINITY; int bi = 0, bj = 0, ba = -1;
    *valid = 1;
    for (int a = 0; a < n_angles; ++a) {
        int rc = sido_get_template(img1, rows1, cols1, pitch1, c1, r1, tab + 4 * a, s, order, tpl);
        if (rc) { free(tpl); free(res); return rc; }
        int has_zero = 0;
        for (int k = 0; k < s * s; ++k) if (tpl[k] == 0) { has_zero = 1; break; }
        if (has_zero) { *valid = 0; break; }
        rc = sido_match_template(image2, H, W, pitch2, tpl, s, s, s, res);
        if (rc) { free(tpl); free(res); return rc; }
        /* np.argmax: first maximum in row-major order */
        float mx = res[0]; int mk = 0;
        for (int k = 1; k < RH * RW; ++k) if (res[k] > mx) { mx = res[k]; mk = k; }
        if (mx > br) {
            br = mx; ba = a; bi = mk / RW; bj = mk % RW;
            memcpy(bres, res, (size_t)RH * RW * sizeof(float));
            memcpy(btpl, tpl, (size_t)s * s);
        }
    }
    if (*valid && ba < 0) *valid = 0;      /* all-NaN style degenerate case */
    if (!*valid) {
        *dc = NAN; *dr = NAN; *best_angle_idx = -1; *best_r = NAN; *best_h = NAN;
        free(tpl); free(res);
        return SIDO_OK;
    }
    int rc = sido_hessian(bres, RH, RW, hes_norm, hes_smth, hes);
    if (rc) { free(tpl); free(res); return rc; }
    *best_h = hes[bi * RW + bj];
    *dr = (double)bi - (double)(H - s) / 2.0;
    *dc = (double)bj - (double)(W - s) / 2.0;
    *best_angle_idx = ba;
    if (mcc_norm) {
        float med = median_f32(bres, RH * RW, hes);
        float sd = std_f32(bres, RH * RW);
        volatile float d = br - med;
        br = d / sd;
    }
    *best_r = br;
    if (best_result) memcpy(best_result, bres, (size_t)RH * RW * sizeof(float));
    if (best_template) memcpy(best_template, btpl, (size_t)s * s);
    free(tpl); free(res);
    return SIDO_OK;
}

/* ------------------------------------------------------------------ use_mcc over a batch */

/* pmlib.py:176-212 for every point i (the body of the Pool map, pmlib.py:436-448).
 * out: n x 5 doubles (c2, r2, angle, r, h), NaN rows where the reference returns NaN.
 * status[i] (optional): 1 valid, 0 NaN (zero pixel), -1 window outside img2 (rejected). */
int sido_use_mcc_batch(int64_t n, const double *c1, const double *r1,
                       const double *c2fg, const double *r2fg, const double *border,
                       const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                       const uint8_t *img2, int rows2, int cols2, int64_t pitch2,
                       int s, int n_angles, const double *angles, const double *tab,
                       int order, int hes_norm, int hes_smth, int mcc_norm,
                       double *out, int *status)
{
    if (n < 0 || !out) return SIDO_EINVAL;
    const int hws = (int)((double)s / 2.0);
    int err = 0;
    for (int64_t i = 0; i < n; ++i) {
        double *o = out + 5 * i;
        o[0] = o[1] = o[2] = o[3] = o[4] = NAN;
        /* a non-finite input has no window and no template (the reference fails on it; the kernels reject it, as
         * here): never sample image 1 at a NaN coordinate */
        if (!isfinite(c1[i]) || !isfinite(r1[i]) || !isfinite(c2fg[i]) || !isfinite(r2fg[i]) || !isfinite(border[i]) ||
            fabs(c2fg[i]) >= 1e9 || fabs(r2fg[i]) >= 1e9 || fabs(border[i]) >= 1e9) {
            if (status) status[i] = -1;
            continue;
        }
        /* python int() truncates toward zero */
        int64_t y0 = (int64_t)(r2fg[i] - hws - border[i]);
        int64_t y1 = (int64_t)(r2fg[i] + hws + border[i] + 1);
        int64_t x0 = (int64_t)(c2fg[i] - hws - border[i]);
        int64_t x1 = (int64_t)(c2fg[i] + hws + border[i] + 1);
        /* numpy slicing clips the far end silently; a negative start would wrap
         * (reference then fails inside cv2) -> rejected here */
        if (y1 > rows2) y1 = rows2;
        if (x1 > cols2) x1 = cols2;
        if (y0 < 0 || x0 < 0 || y1 - y0 < s + 1 || x1 - x0 < s + 1) {
            if (status) status[i] = -1;
            continue;
        }
        int valid = 0, ba = -1; double dc, dr; float br, bh;
        int rc = sido_rotate_and_match(img1, rows1, cols1, pitch1, c1[i], r1[i], s,
                                       img2 + y0 * pitch2 + x0, (int)(y1 - y0), (int)(x1 - x0), pitch2,
                                       n_angles, tab, order, hes_norm, hes_smth, mcc_norm,
                                       &valid, &dc, &dr, &ba, &br, &bh, NULL, NULL);
        if (rc) {
            err = rc;
            continue;
        }
        if (status) status[i] = valid;
        if (valid) {
            o[0] = c2fg[i] + dc; o[1] = r2fg[i] + dr; o[2] = angles[ba];
            o[3] = (double)br; o[4] = (double)bh;
        }
    }
    return err;
}

const char *sido_version(void) { return "sido-1 (restates sea_ice_drift 0.7.1 pmlib hot path)"; }

/* ------------------------------------------------------------------ feature-tracking matcher (SURVEY 8f) */

/* cv2.BFMatcher(NORM_HAMMING).knnMatch(d1, d2, k=2) at the reference's call site ftlib.py:95-96: the two
 * train descriptors with the smallest Hamming distance, equal distances ordered by train index (pinned
 * against OpenCV 4.13, tests/test_ftlib.py).  idx/dist: n1 x 2 ints, -1 where there is no such neighbour. */
int sido_knn_hamming2(const uint8_t *d1, int n1, const uint8_t *d2, int n2, int nbytes, int32_t *idx, int32_t *dist)
{
    if (n1 < 0 || n2 < 0 || nbytes <= 0) return SIDO_EINVAL;
    for (int q = 0; q < n1; ++q) {
        int b0 = 0x7fffffff, b1 = 0x7fffffff, i0 = -1, i1 = -1;
        for (int t = 0; t < n2; ++t) {
            int d = 0;
            for (int k = 0; k < nbytes; ++k) d += __builtin_popcount((unsigned)(d1[(size_t)q * nbytes + k] ^ d2[(size_t)t * nbytes + k]));
            if (d < b0) { b1 = b0; i1 = i0; b0 = d; i0 = t; }
            else if (d < b1) { b1 = d; i1 = t; }
        }
        idx[2 * q] = i0; idx[2 * q + 1] = i1;
        dist[2 * q] = i0 >= 0 ? b0 : -1; dist[2 * q + 1] = i1 >= 0 ? b1 : -1;
    }
    return SIDO_OK;
}
