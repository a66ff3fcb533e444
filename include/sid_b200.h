/*
 * sid_b200.h -- C ABI of the B200-native pattern-matching (MCC) hot path.
 *
 * Drop-in boundary for nansencenter/sea_ice_drift v0.7.1 (paths below are under
 * the reference tree, sea_ice_drift/):
 *
 *   sid_run / sid_run_pair / sid_run_device
 *                              replace the per-point loop of pattern_matching,
 *                              pmlib.py:430-448 (_init_pool + Pool.map(use_mcc_mp)),
 *                              i.e. use_mcc (pmlib.py:176-212) for every grid point.
 *                              Argument order mirrors _init_pool's tuple (pmlib.py:438).
 *   sid_run_maps               sid_run that also returns every point's winning NCC map and
 *                              template (rotate_and_match's best_result / best_template).
 *   sid_rotate_and_match       replaces rotate_and_match, pmlib.py:117-174.
 *   sid_get_template           replaces get_template, pmlib.py:89-115.
 *   sid_match_template         replaces the template_matcher plug-in call
 *                              cv2.matchTemplate(image, templ, TM_CCOEFF_NORMED),
 *                              pmlib.py:120 (default) / pmlib.py:156 (call site).
 *   sid_get_hessian            replaces get_hessian, pmlib.py:36-59.
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns 0 or a negative
 *     SID_E* code and never throws/aborts; sid_last_error() gives the message.
 *   - images are uint8, row-major, `pitch` bytes between rows; pixel value 0 means
 *     "invalid" exactly as in the reference (lib.py:52-57).
 *   - `angle_tab` holds 4 doubles per angle: cos a, sin a, tcdot0, tcdot1 with
 *     a = radians(angle - alpha0), tc = int(img_size/2.)+1 and
 *     tcdot = [tc,tc] . [[cos a,-sin a],[sin a,cos a]]  (pmlib.py:105-110); the
 *     caller evaluates it with NumPy so results do not depend on a device libm.
 *   - a context is bound to one device and one stream; it is not re-entrant.
 *   - invalid POINTS are not errors: they yield NaN rows, exactly where the
 *     reference returns NaN (a 0 pixel in any angle's template, pmlib.py:152-154).
 *     Points whose search window starts outside image 2 (the reference would wrap
 *     or fail inside cv2) also yield NaN rows and status -1.
 */
#ifndef SID_B200_H
#define SID_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sid_ctx sid_ctx;

#define SID_OK 0
#define SID_EINVAL (-1)      /* bad argument                                  */
#define SID_ECUDA (-2)       /* CUDA runtime error (see sid_last_error)       */
#define SID_ENOMEM (-3)      /* host or device allocation failed              */
#define SID_EUNSUPPORTED (-4)/* e.g. mtype != TM_CCOEFF_NORMED, rot_order > 1 */
#define SID_ENOPAIR (-5)     /* sid_set_pair has not been called              */

#define SID_TM_CCOEFF_NORMED 5 /* == cv2.TM_CCOEFF_NORMED */

/* flags for sid_run* / sid_rotate_and_match */
#define SID_HES_NORM 1u      /* get_hessian(hes_norm=True)  -- reference default */
#define SID_HES_SMTH 2u      /* get_hessian(hes_smth=True)                       */
#define SID_MCC_NORM 4u      /* rotate_and_match(mcc_norm=True)                  */
/* SID_SUBPIXEL (extension, not in the reference): refine c2 / r2 (dc / dr) to sub-pixel precision by the vertex of the
 * parabola through the peak of the winning angle's RAW float32 NCC map and its two neighbours, per axis:
 *   a, b, c = m[bi][bj-1], m[bi][bj], m[bi][bj+1] widened to double;  p = b - a, q = b - c;
 *   dx = (p - q) / (2 (p + q));  c2 = (c2fg + dc) + dx     (IEEE double, round to nearest, no fused operations)
 * and the same down the column for dy and r2.  |dx|, |dy| <= 0.5; a peak on the first or last column (row) leaves c2
 * (r2) exactly as without the flag.  Angle, r, h, the NaN rows and status are bit-identical to the call without it. */
#define SID_SUBPIXEL 8u
/* SID_MASKED (extension, not in the reference): match the rows the reference returns as NaN because some angle's template
 * holds a 0 pixel (land, no-data, samples outside image 1) by the Pearson correlation over the template's valid pixels.
 * For one angle's template T (s x s): M = (T > 0), n = sum M, St = sum T, Stt = sum T^2; at map position p over the
 * window patch W (window pixels are data, zeros included; only the template is masked):
 *   C = sum T W, Sw = sum M W, Sww = sum M W^2;  num = n C - St Sw, vt = n Stt - St^2, vw = n Sww - Sw^2   (exact int64)
 *   r = (double)num / (sqrt((double)vt) * sqrt((double)vw)) in IEEE double without contraction, clamped to [-1, 1],
 *   rounded to float32;  r = 0 where vw = 0
 * (cv2.matchTemplate(image, T, TM_CCOEFF_NORMED, mask=(T > 0))).  A row is re-matched this way, every angle masked, when
 * the call without the flag gives it SID_PT_NAN, every angle's template has at least ceil(s^2 / 2) valid pixels and
 * vt > 0 for every angle; its status is SID_PT_MASKED.  Winner, h, mcc_norm, hes_smth and SID_SUBPIXEL follow the usual
 * rules on the masked float maps.  Every other row is bit-identical to the call without the flag. */
#define SID_MASKED 16u
/* SID_PEAKS (extension, not in the reference): also record, for every row, the SID_N_PEAKS next-best peaks of its winning
 * map, for the outlier filter (sid_filter_outliers).  m is the row's RAW float32 winning-angle map, RH x RW (the map
 * sid_run_maps returns), flat index f(i, j) = i RW + j.  p is a PEAK when every in-map 8-neighbour q has m[q] < m[p] if
 * f(q) < f(p) and m[q] <= m[p] if f(q) > f(p): a plateau counts once, at its first index (np.argmax's rule; the primary
 * peak is always one).  The SECONDARY peaks are all peaks but the primary, by m descending, ties by f ascending; the first
 * SID_N_PEAKS are kept, each as four doubles c2, r2, r, h computed exactly as the row computes its own:
 *   c2 = c2fg + (j - (W - s) / 2), r2 = r2fg + (i - (H - s) / 2), plus peak_offsets at (i, j) with SID_SUBPIXEL;
 *   r = m[p], or (m[p] - median m) / std m under mcc_norm, in float32 as the row's r;
 *   h = get_hessian(m, hes_norm, hes_smth)[p], normalised with the median and std that normalised the row's h.
 * Missing peaks (fewer than SID_N_PEAKS; a flat template's all-1.0 map has none) and rows that are neither SID_PT_VALID nor
 * SID_PT_MASKED get NaN records.  Every sid_run* honours it; the table, status and maps are bit-identical to the call
 * without it; sid_get_peaks copies the records out, and sid_filter_outliers reads them on the device.
 * sid_rotate_and_match refuses it (SID_EUNSUPPORTED). */
#define SID_PEAKS 32u
#define SID_N_PEAKS 3
/* SID_UNCERT (extension, not in the reference): also record, for every row, the covariance of the sub-pixel offsets
 * (dx, dy) that SID_SUBPIXEL added to c2 and r2 -- three doubles var_c, var_r, cov_cr in image-2 pixels^2 -- by correlation
 * statistics (Wieneke 2015, Meas. Sci. Technol. 26, 074002).  Valid only with SID_SUBPIXEL: without it every sid_run*
 * returns SID_EINVAL before any launch.  For a SID_PT_VALID or SID_PT_MASKED row: T the winning angle's template (s x s,
 * the bytes sid_run_maps returns), W_P the window patch at map position P (the kernels' window rule), m the RAW float32
 * winning map (RH x RW) and (bi, bj) its primary integer peak.  M_k = 1 (VALID) or (T_k > 0) (MASKED), and
 *   n = sum M_k, St = sum M_k T_k, t_k = M_k (n T_k - St), Vt = sum t_k^2                                 (exact int64)
 *   Sw(P) = sum M_k W_P,k, w_k(P) = M_k (n W_P,k - Sw(P)), A(P) = sum t_k w_k(P), V(P) = sum w_k(P)^2     (exact int64:
 *   |t|, |w| < 2^22 for s <= 128), S(P, Q) = sum t_k^2 w_k(P) w_k(Q)  (exact 128-bit: |S| < 2^102 at s = 128)
 *   K(P, Q) = D(n S(P, Q) - A(P) A(Q)) / (((D(n) D(Vt)) sqrt(D(V(P)))) sqrt(D(V(Q))))
 * with D the correctly rounded (ties to even) integer -> double conversion of the exact numerator (|.| < 2^117) and every
 * operation IEEE double, round to nearest, without contraction.  The per-pixel contributions
 * x_k(P) = t_k w_k(P) / (sqrt(Vt) sqrt(V(P))) sum to the Pearson correlation at P; K is n times their population
 * covariance over the n pixels, i.e. the covariance of the correlation values at P and Q when pixels are independent.
 * Positions, in this order: P0 = (bi, bj), X- / X+ = (bi, bj -+ 1), Y- / Y+ = (bi -+ 1, bj); K is evaluated
 * once per unordered pair, P the earlier of the two in that order.  With a, b, c = m at X-, P0, X+ widened to double,
 * p = b - a, q = b - c, w = (p + q) (p + q) and g = (-q / w, (q - p) / w, p / w) (the gradient of the vertex
 * d = (p - q) / (2 (p + q)) in (a, b, c)); g' the same down the column (Y-, P0, Y+):
 *   var_c = (g0 h0 + g1 h1) + g2 h2,  h_u = (K(u, X-) g0 + K(u, P0) g1) + K(u, X+) g2,  u = X-, P0, X+
 *   var_r the same with g' over Y-, P0, Y+;  cov_cr with g on the left over (X-, P0, X+), g' on the right over (Y-, P0, Y+).
 * NaN: a peak on the first or last map column makes var_c and cov_cr NaN (that axis is not refined), one on the first or
 * last row var_r and cov_cr; V(P) = 0 at a position an axis uses makes that axis' variance and cov_cr NaN; rows that are
 * neither VALID nor MASKED get three NaN.  mcc_norm and hes_smth do not enter.  The pass is one extra launch behind every
 * other launch of the call; the table, status, maps, templates and peaks are bit-identical to the call without the flag.
 * sid_get_uncertainty copies the records out; sid_rotate_and_match refuses the flag (SID_EUNSUPPORTED). */
#define SID_UNCERT 64u

/* point status written by sid_run* (optional output) */
#define SID_PT_VALID 1
#define SID_PT_NAN 0         /* zero pixel in a template -> NaN row              */
#define SID_PT_REJECTED (-1) /* window not inside image 2 / too small            */
#define SID_PT_MASKED 2      /* SID_MASKED: matched by the masked rule          */

const char *sid_version(void);

/* Create / destroy a context on CUDA device `device`. */
int sid_create(sid_ctx **out, int device);
void sid_destroy(sid_ctx *ctx);
const char *sid_last_error(const sid_ctx *ctx);

/* Run all work of this context on `cuda_stream` (a cudaStream_t passed as void*;
 * NULL = the context's own stream, (void*)1 = cudaStreamLegacy, the default stream). */
int sid_set_stream(sid_ctx *ctx, void *cuda_stream);
int sid_synchronize(sid_ctx *ctx);

/* Upload the image pair (host pointers); it stays resident on the device until
 * the next call (time-series reuse).  Replaces the images in _init_pool's tuple. */
int sid_set_pair(sid_ctx *ctx,
                 const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                 const uint8_t *img2, int rows2, int cols2, int64_t pitch2);
/* Same, but the sources are DEVICE pointers (device-to-device copy into the
 * context's padded layout), e.g. a peer-broadcast image. */
int sid_set_pair_device(sid_ctx *ctx,
                        const uint8_t *d_img1, int rows1, int cols1, int64_t pitch1,
                        const uint8_t *d_img2, int rows2, int cols2, int64_t pitch2);

/* Layout the library uses for a resident image: row pitch (a legal TMA stride: multiple of 16, >= cols + 16) and the
 * total allocation (pitch * rows + tail slack).  For callers that fill the pair themselves (sid_adopt_pair_device). */
int sid_pair_layout(int rows, int cols, int64_t *pitch, int64_t *bytes);
/* Use CALLER-OWNED device buffers as the resident pair, without a copy: the multi-GPU path, where every rank
 * uploads one row slab of each image and an in-place NCCL all-gather over NVLink completes the buffers (replaces
 * the fork/copy-on-write replication of the reference's Pool, pmlib.py:430-448).  The buffers must follow
 * sid_pair_layout (256-byte aligned base, pitch, bytes) and outlive their use; the library never frees them. */
int sid_adopt_pair_device(sid_ctx *ctx,
                          uint8_t *d_img1, int rows1, int cols1, int64_t pitch1, int64_t bytes1,
                          uint8_t *d_img2, int rows2, int cols2, int64_t pitch2, int64_t bytes2);

/* First guess of pattern_matching on the device (reference pmlib.py:249-324 prepare_first_guess, pmlib.py:61-77
 * get_distance_to_nearest_keypoint; lib.py:179-201 interpolation_near): for every query point q
 *   out_vx/out_vy  the Delaunay-linear interpolant of (vx, vy) given at the sources (sx, sy) -- what
 *                  scipy.interpolate.griddata(method='linear') returns -- NaN outside the sources' convex hull;
 *   out_dist       the distance to the nearest (kx, ky) point (the reference samples a full-image distance transform);
 *   out_flag       0 ok, 1 outside the hull, 2 not resolved numerically (caller falls back to its host path).
 * No triangulation is built: each point finds its own Delaunay triangle by pivoting (csrc/sid_fg_kernel.cuh). */
int sid_first_guess(sid_ctx *ctx, int n_src, const double *sx, const double *sy, const double *vx, const double *vy,
                    int n_seed, const double *kx, const double *ky,
                    int64_t n_q, const double *qx, const double *qy,
                    double *out_vx, double *out_vy, double *out_dist, int32_t *out_flag);

/* Post-processing of pattern_matching for AFFINE geolocation (reference pmlib.py:462-497 and lib.py:408-412), on the
 * device: sub-pixel remainder c2 += c2pm1 - round(c2pm1), pixel -> destination x/y and lon/lat, u = x2 - x1,
 * v = y2 - y1, and the _fill_gpi scatter into NaN-filled grids.
 *   n_valid, grid_index  the valid grid points (gpi) in table order and their flat grid positions
 *   c2pm1, r2pm1         n_grid image-2 pixel coordinates of the grid (host)
 *   results              host (n_valid, 5) table, or NULL: use the table the previous sid_run / sid_run_pair left on
 *                        the device (those accept out == NULL, so the table never visits the host)
 *   xy, ll               2 x 3 row-major affine maps pixel -> destination x/y and pixel -> lon/lat: m0*c + m1*r + m2
 *   out                  host, 7 x n_grid doubles: u, v, a, r, h, lon2, lat2                                         */
int sid_pm_epilogue_affine(sid_ctx *ctx, int64_t n_valid, const int32_t *grid_index, int64_t n_grid,
                           const double *c2pm1, const double *r2pm1, const double *results,
                           const double *xy, const double *ll, double *out);

/* SID_PEAKS records of the previous sid_run* call: out = n x SID_N_PEAKS x 4 doubles (c2, r2, r, h per peak, rank order,
 * NaN where missing), host pointer, synchronous.  SID_EINVAL (context stays usable) when that call did not set SID_PEAKS
 * or had a different n. */
int sid_get_peaks(sid_ctx *ctx, int64_t n, double *out);

/* SID_UNCERT records of the previous sid_run* call: out = n x 3 doubles (var_c, var_r, cov_cr), host pointer,
 * synchronous.  SID_EINVAL (context stays usable) when that call did not set SID_UNCERT or had a different n. */
int sid_get_uncertainty(sid_ctx *ctx, int64_t n, double *out);

/* Normalised median test (Westerweel & Scarano 2005, "universal outlier detection") over the grid of a result table, with
 * replacement by a secondary peak (SID_PEAKS), on the device.  Every operation is an IEEE double op without contraction.
 *   grid_rows x grid_cols  the grid; n_valid, grid_index, c2pm1, r2pm1 as for sid_pm_epilogue_affine (n_grid = rows x cols)
 *   results, peaks         host (n_valid, 5) table and (n_valid, SID_N_PEAKS, 4) records, or both NULL: what the previous
 *                          sid_run / sid_run_pair / sid_run_maps left on the device (it must have set SID_PEAKS)
 *   out                    host (n_valid, 5) filtered table; NULL (device-resident inputs only) updates the device table
 *                          in place, so that sid_pm_epilogue_affine(results = NULL) reads the filtered table
 *   flag                   optional host n_valid ints (below)
 * Rule, decided on the unfiltered table in one pass.  Displacement of a row at grid position g:
 * d = (c2 - rint(c2pm1[g]), r2 - rint(r2pm1[g])) (rint: ties to even).  Neighbours: the in-grid 8-neighbours of g whose row
 * has a finite c2.  With k < 3 neighbours the row is kept, flag -2.  Per axis: m = median of the neighbours' d ((a + b) *
 * 0.5 of the middle two for even k), r_m = median of |d_i - m|, e = |d0 - m| / (r_m + eps).  The row is an outlier iff
 * e_x^2 + e_y^2 > threshold^2; it then takes the first finite secondary peak, in rank order, that passes the same test
 * against the same m and r_m (its c2, r2, r, h; angle unchanged; flag = its rank 1 ... SID_N_PEAKS), else it becomes a NaN
 * row, flag -1.  Kept rows: flag 0; NaN rows: flag -3.  Suggested eps 1.0 px, threshold 2.0. */
int sid_filter_outliers(sid_ctx *ctx, int grid_rows, int grid_cols, int64_t n_valid, const int32_t *grid_index,
                        const double *c2pm1, const double *r2pm1,
                        const double *results, const double *peaks,
                        double eps, double threshold, double *out, int32_t *flag);

/* Asynchronous 2-D host -> device copy of `rows` image rows on the context's stream (a rank's row slab of the
 * pair, before the all-gather that completes the adopted buffers). */
int sid_upload_rows(sid_ctx *ctx, uint8_t *d_dst, int64_t dst_pitch, const uint8_t *src, int64_t src_pitch, int cols, int rows);

/* k x k box downsampling of the RESIDENT pair (k = factor in [2, 16]) into caller-owned device buffers laid out by
 * sid_pair_layout(rows / k, cols / k) of each image (floor: trailing rows and columns are dropped).  Output pixel
 * (i, j) is 0 if any of the k * k source pixels (rows k*i ... k*i+k-1, columns k*j ... k*j+k-1) is 0 (invalid, as
 * everywhere in this library), else floor(mean + 0.5) computed exactly in integers, (2 * sum + k*k) / (2 * k*k).  Only
 * the rows * cols bytes of each image are written, never the pitch padding.  The buffers can then be adopted as the
 * pair of another context (sid_adopt_pair_device) to match on the coarse pair (pmlib.coarse_tracking).  Checked on the
 * host before any launch: SID_ENOPAIR without a resident pair; SID_EINVAL for a factor outside [2, 16], a downsampled
 * image smaller than 1 x 1, or a buffer whose pitch or size is below sid_pair_layout's (or a pitch not a multiple of
 * 16); the context stays usable.  One launch (sid::downsample_kernel), asynchronous on the context's stream. */
int sid_downsample_pair(sid_ctx *ctx, int factor,
                        uint8_t *d_img1, int64_t pitch1, int64_t bytes1,
                        uint8_t *d_img2, int64_t pitch2, int64_t bytes2);

/* use_mcc for n grid points (host arrays in, host array out, synchronous).  All sid_run* honour SID_MASKED, SID_PEAKS and SID_UNCERT.
 *   c1, r1        float pixel coordinates on image 1
 *   c2fg, r2fg    integer-valued first guess on image 2
 *   border        integer-valued search radius per point
 *   out           n x 5 row-major doubles: c2, r2, angle, r, h  (NaN rows = invalid); with SID_SUBPIXEL in `flags`
 *                 c2 / r2 are refined to sub-pixel precision, the other columns do not change
 *   status        optional (may be NULL), n ints, SID_PT_*                          */
int sid_run(sid_ctx *ctx, int64_t n,
            const double *c1, const double *r1,
            const double *c2fg, const double *r2fg, const double *border,
            int img_size, int n_angles, const double *angles, const double *angle_tab,
            int rot_order, unsigned flags, int mtype,
            double *out, int *status);

/* sid_set_pair + sid_run in ONE call, with the host-to-device copy of the image pair overlapped
 * with the computation: the pair is uploaded in row bands on a second stream and the points are
 * processed band by band as soon as every image row they touch has arrived.  Results are
 * identical to sid_set_pair followed by sid_run; the pair stays resident afterwards.  Page-locked host
 * images are copied by DMA directly; pageable ones (plain malloc / NumPy memory) go band by band through
 * a pinned double buffer that a few host threads fill while the previous band is in flight (EW-sized
 * pair, B200: 6.1 ms per call pinned, 9.7 ms pageable, against 26 ms for a plain pageable cudaMemcpy).
 * SID_SUBPIXEL refines c2 / r2 as in sid_run. */
int sid_run_pair(sid_ctx *ctx,
                 const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                 const uint8_t *img2, int rows2, int cols2, int64_t pitch2,
                 int64_t n,
                 const double *c1, const double *r1,
                 const double *c2fg, const double *r2fg, const double *border,
                 int img_size, int n_angles, const double *angles, const double *angle_tab,
                 int rot_order, unsigned flags, int mtype,
                 double *out, int *status);

/* Same with DEVICE pointers for the point arrays and outputs; asynchronous on
 * the context's stream (no host synchronisation).  `max_border` must bound
 * border[] (it sizes shared memory / scratch); pass <= 0 to have the library
 * read the borders back (synchronises).  SID_SUBPIXEL refines c2 / r2 as in sid_run. */
int sid_run_device(sid_ctx *ctx, int64_t n,
                   const double *d_c1, const double *d_r1,
                   const double *d_c2fg, const double *d_r2fg, const double *d_border,
                   int max_border,
                   int img_size, int n_angles, const double *angles, const double *angle_tab,
                   int rot_order, unsigned flags, int mtype,
                   double *d_out, int *d_status);

/* Shapes of the correlation maps sid_run_maps returns for these points on the RESIDENT pair: map i is
 * map_shape[2i] x map_shape[2i+1] = (H - img_size + 1) x (W - img_size + 1), where H x W is the point's search
 * window as use_mcc slices it (pmlib.py:200-208: truncation of r2fg +- hws +- border, NumPy's clipping of the far
 * edge), so fractional first guesses or borders and windows at the far edge give non-square maps.  Points the
 * window rule rejects (their status is SID_PT_REJECTED) get 0 x 0; NaN rows (SID_PT_NAN) keep their shape.
 * *total = sum of the map sizes (floats).  map_shape may be NULL. */
int sid_map_layout(sid_ctx *ctx, int64_t n,
                   const double *c1, const double *r1,
                   const double *c2fg, const double *r2fg, const double *border,
                   int img_size, int32_t *map_shape, int64_t *total);

/* sid_run plus, for every point, what rotate_and_match returns as best_result and best_template
 * (pmlib.py:117-174, [5] and [6]); host pointers, resident pair, synchronous.  out / status are those of sid_run,
 * bit for bit.  With SID_SUBPIXEL the table is refined as in sid_run and the maps are unchanged (the offsets are
 * computed from them).
 *   maps        maps_capacity floats: the maps of sid_map_layout packed in point order.  For a valid row, the raw
 *               float32 NCC map of the winning angle (the first of equal peaks; hes_smth and mcc_norm do not touch
 *               it; a flat template gives all 1.0); for a SID_PT_MASKED row its masked map.  Segments of rows that
 *               are neither are NaN.
 *   templates   optional (may be NULL), n x img_size x img_size bytes: the winning angle's template (zeros
 *               included for a SID_PT_MASKED row); 0 for rows that are neither valid nor masked.
 * maps_capacity below sid_map_layout's total -> SID_EINVAL before anything is launched. */
int sid_run_maps(sid_ctx *ctx, int64_t n,
                 const double *c1, const double *r1,
                 const double *c2fg, const double *r2fg, const double *border,
                 int img_size, int n_angles, const double *angles, const double *angle_tab,
                 int rot_order, unsigned flags, int mtype,
                 double *out, int *status,
                 int64_t maps_capacity, float *maps, uint8_t *templates);

/* Number of kernel launches issued by this context so far (bench accounting). */
int64_t sid_launch_count(const sid_ctx *ctx);
/* Device time (ms, CUDA events on the launching stream) of the most recent launch of the fused
 * point kernel; waits for it to finish.  -1 if nothing was launched yet. */
double sid_last_kernel_ms(sid_ctx *ctx);
/* Name of the point kernel the most recent launch used ("sid::pm_ws_kernel", "sid::pm_tc_kernel",
 * "sid::pm_points_kernel<imma>", "sid::pm_points_kernel<dp4a>"); "" before the first launch.  The paths
 * are interchangeable (bit-identical tables); the dispatch picks by search radius (DESIGN.md section 4). */
const char *sid_last_kernel_name(const sid_ctx *ctx);

/* rotate_and_match for one point against an explicit search window `image2`
 * (host pointers).  Outputs: *valid (0 -> the reference returns 7 x NaN),
 * dc, dr, best_angle_idx (index into the angle list), best_r, best_h, and
 * optionally the best NCC map ((H-s+1) x (W-s+1) floats) and template (s x s).
 * SID_SUBPIXEL adds the sub-pixel offsets of sid_run to *dc / *dr; best_result is the unrefined map.
 * SID_MASKED applies the masked rule to any window size; *valid = 2 (SID_PT_MASKED) for a point it matched. */
int sid_rotate_and_match(sid_ctx *ctx,
                         const uint8_t *img1, int rows1, int cols1, int64_t pitch1,
                         double c1, double r1, int img_size,
                         const uint8_t *image2, int H, int W, int64_t pitch2,
                         int n_angles, const double *angle_tab,
                         int rot_order, unsigned flags, int mtype,
                         int *valid, double *dc, double *dr, int *best_angle_idx,
                         float *best_r, float *best_h,
                         float *best_result, uint8_t *best_template);

/* get_template: s x s rotated/shifted uint8 patch (angle_tab: 4 doubles). */
int sid_get_template(sid_ctx *ctx,
                     const uint8_t *img, int rows, int cols, int64_t pitch,
                     double c, double r, const double *angle_tab, int s, int rot_order,
                     uint8_t *out);

/* template_matcher plug-in: zero-mean normalised cross-correlation map,
 * (H-th+1) x (W-tw+1) float32, method must be SID_TM_CCOEFF_NORMED. */
int sid_match_template(sid_ctx *ctx,
                       const uint8_t *img, int H, int W, int64_t pitch,
                       const uint8_t *tpl, int th, int tw, int64_t tpitch,
                       int method, float *out);

/* Feature-tracking matcher (SURVEY 8f, the caller side of the hot path): the two nearest train descriptors
 * in Hamming distance for every query descriptor, i.e. what
 * cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch(d1, d2, k=2) returns at the reference's call site
 * ftlib.py:92-99 (the `matcher` plug-in kwarg of get_match_coords).  Host pointers, descriptors are rows of
 * desc_bytes bytes (32 = ORB).  idx / dist: n1 x 2 ints, best first; equal distances go to the lower train
 * index (OpenCV's order); -1 where fewer than two train descriptors exist. */
int sid_knn_hamming2(sid_ctx *ctx, const uint8_t *d1, int n1, const uint8_t *d2, int n2, int desc_bytes,
                     int32_t *idx, int32_t *dist);

/* Deformation of triangular elements (SURVEY 8f, the consumer side of the hot path): what
 * get_deformation_on_triangulation (libdefor.py:50-99) and get_deformation_elems (libdefor.py:4-48) return.
 * Host pointers.  x, y, u, v: n node values; tri: m x 3 node indices, row-major; area_in: optional m element
 * areas (NULL = Heron's formula from the side lengths, as get_deformation_on_triangulation does).
 * Outputs, m doubles each: e1 divergence, e2 shear, e3 vorticity, area, perimeter; NaN for an element with a
 * node index outside [0, n). */
int sid_deformation(sid_ctx *ctx, int n, const double *x, const double *y, const double *u, const double *v,
                    int m, const int32_t *tri, const double *area_in,
                    double *e1, double *e2, double *e3, double *area, double *perim);

/* get_hessian of a float32 map (rows x cols) -> float32 map of the same shape. */
int sid_get_hessian(sid_ctx *ctx, const float *ccm, int rows, int cols,
                    unsigned flags, float *out);

#ifdef __cplusplus
}
#endif
#endif /* SID_B200_H */
