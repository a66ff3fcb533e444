/*
 * masked_oracle.c -- TEST INFRASTRUCTURE ONLY: the exact CPU oracle of the masked correlation (SID_MASKED,
 * include/sid_b200.h) that the GPU tables, maps and templates are compared with bit for bit.
 *
 * It extends the plain-C oracle of the reference's hot path (oracle/mcc_oracle.c, included unchanged, so template
 * sampling, the unmasked NCC, the Hessian and the statistics are exactly that oracle's) with:
 *   sido_match_template_masked   the masked rule on one window: the Pearson correlation over the template's valid
 *                                pixels from exact integer sums (cv2.matchTemplate(..., TM_CCOEFF_NORMED, mask=(T > 0)))
 *   sido_rotate_and_match_ex     sido_rotate_and_match with the row selection of SID_MASKED (*valid = 2 for a masked row)
 *   sido_use_mcc_batch_ex        sido_use_mcc_batch with the same selection (status 2)
 * Built by tests/masked_oracle.py.
 */
#include "../oracle/mcc_oracle.c"

/* ------------------------------------------------------------------ masked NCC */

/* ------------------------------------------------------------------ masked NCC (extension, SID_MASKED) */

/* Template statistics of the masked rule: n = number of valid (> 0) pixels, St = sum T, Stt = sum T^2 (over all
 * pixels: T is 0 where the mask is 0). */
void sido_masked_stats(const uint8_t *tpl, int s, int64_t *n, int64_t *st, int64_t *stt)
{
    int64_t a = 0, b = 0, c = 0;
    for (int k = 0; k < s * s; ++k) { int64_t v = tpl[k]; a += v > 0; b += v; c += v * v; }
    *n = a; *st = b; *stt = c;
}

/* Pearson correlation of the template's valid pixels (M = T > 0) with the window patch W at every position, what
 * cv2.matchTemplate(image, templ, TM_CCOEFF_NORMED, mask=(templ > 0)) computes, from exact integer sums:
 *   C = sum T W, Sw = sum M W, Sww = sum M W^2;  num = n C - St Sw, vt = n Stt - St^2, vw = n Sww - Sw^2
 *   r = (double)num / (sqrt((double)vt) * sqrt((double)vw)), clamped to [-1, 1], rounded to float32;  vw = 0 -> 0.
 * Window zeros are data.  The caller guarantees vt > 0. */
int sido_match_template_masked(const uint8_t *img, int H, int W, int64_t pitch, const uint8_t *tpl, int s, float *out)
{
    if (!img || !tpl || !out || s <= 0 || H < s || W < s) return SIDO_EINVAL;
    const int RH = H - s + 1, RW = W - s + 1;
    int64_t n, st, stt;
    sido_masked_stats(tpl, s, &n, &st, &stt);
    const double sqrt_vt = sqrt((double)(n * stt - st * st));
    for (int y = 0; y < RH; ++y) {
        for (int x = 0; x < RW; ++x) {
            int64_t c = 0, sw = 0, sww = 0;
            for (int i = 0; i < s; ++i) {
                const uint8_t *ip = img + (int64_t)(y + i) * pitch + x;
                const uint8_t *tp = tpl + (int64_t)i * s;
                for (int j = 0; j < s; ++j) {
                    const int64_t v = ip[j];
                    c += v * tp[j];
                    if (tp[j]) { sw += v; sww += v * v; }
                }
            }
            const int64_t num = n * c - st * sw, vw = n * sww - sw * sw;
            double r = 0.0;
            if (vw != 0) {
                const double den = sqrt_vt * sqrt((double)vw);
                r = (double)num / den;
                if (r > 1.0) r = 1.0;
                if (r < -1.0) r = -1.0;
            }
            out[y * RW + x] = (float)r;
        }
    }
    return SIDO_OK;
}

/* ------------------------------------------------------------------ rotate_and_match with the masked rule */

/* Whether a row the reference returns as NaN (some template holds a 0 pixel) is matched by the masked rule instead:
 * every angle's template has at least ceil(s^2 / 2) valid pixels and vt = n Stt - St^2 > 0.  *any_zero: some template
 * holds a 0 pixel. */
static int masked_row(const uint8_t *img1, int rows1, int cols1, int64_t pitch1, double c1, double r1, int s,
                      int n_angles, const double *tab, int order, uint8_t *tpl, int *any_zero, int *eligible)
{
    *any_zero = 0; *eligible = 1;
    for (int a = 0; a < n_angles; ++a) {
        int rc = sido_get_template(img1, rows1, cols1, pitch1, c1, r1, tab + 4 * a, s, order, tpl);
        if (rc) return rc;
        int64_t n, st, stt;
        sido_masked_stats(tpl, s, &n, &st, &stt);
        if (n < (int64_t)s * s) *any_zero = 1;
        if (2 * n < (int64_t)s * s || n * stt - st * st <= 0) *eligible = 0;
    }
    return SIDO_OK;
}

/* pmlib.py:117-174.  Returns SIDO_OK; *valid = 0 reproduces the reference's
 * "return 7 x NaN" at the first angle whose template contains a 0 pixel.
 * masked != 0 (SID_MASKED): such a row is matched by the masked rule (sido_match_template_masked, every angle) when
 * masked_row accepts it, and *valid = 2. */
int sido_rotate_and_match_ex(const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                             double c1, double r1, int s,
                             const uint8_t *image2, int H, int W, int64_t pitch2,
                             int n_angles, const double *tab, int order,
                             int hes_norm, int hes_smth, int mcc_norm,
                             int *valid, double *dc, double *dr, int *best_angle_idx,
                             float *best_r, float *best_h,
                             float *best_result /* RH*RW or NULL */,
                             uint8_t *best_template /* s*s or NULL */,
                             int masked)
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
    int use_mask = 0;
    if (masked) {
        int any_zero, eligible;
        int rc = masked_row(img1, rows1, cols1, pitch1, c1, r1, s, n_angles, tab, order, tpl, &any_zero, &eligible);
        if (rc) { free(tpl); free(res); return rc; }
        use_mask = any_zero && eligible;
    }
    *valid = use_mask ? 2 : 1;
    for (int a = 0; a < n_angles; ++a) {
        int rc = sido_get_template(img1, rows1, cols1, pitch1, c1, r1, tab + 4 * a, s, order, tpl);
        if (rc) { free(tpl); free(res); return rc; }
        int has_zero = 0;
        for (int k = 0; k < s * s; ++k) if (tpl[k] == 0) { has_zero = 1; break; }
        if (has_zero && !use_mask) { *valid = 0; break; }
        if (use_mask) rc = sido_match_template_masked(image2, H, W, pitch2, tpl, s, res);
        else rc = sido_match_template(image2, H, W, pitch2, tpl, s, s, s, res);
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
 * status[i] (optional): 1 valid, 0 NaN (zero pixel), -1 window outside img2 (rejected), 2 matched by the masked rule
 * (masked != 0, see sido_rotate_and_match_ex). */
int sido_use_mcc_batch_ex(int64_t n, const double *c1, const double *r1,
                          const double *c2fg, const double *r2fg, const double *border,
                          const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                          const uint8_t *img2, int rows2, int cols2, int64_t pitch2,
                          int s, int n_angles, const double *angles, const double *tab,
                          int order, int hes_norm, int hes_smth, int mcc_norm,
                          double *out, int *status, int masked)
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
        int rc = sido_rotate_and_match_ex(img1, rows1, cols1, pitch1, c1[i], r1[i], s,
                                          img2 + y0 * pitch2 + x0, (int)(y1 - y0), (int)(x1 - x0), pitch2,
                                          n_angles, tab, order, hes_norm, hes_smth, mcc_norm,
                                          &valid, &dc, &dr, &ba, &br, &bh, NULL, NULL, masked);
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

