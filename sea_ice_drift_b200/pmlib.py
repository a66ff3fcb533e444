"""Drop-in replacement for the pattern-matching part of ``sea_ice_drift.pmlib``.

Same function names, argument meaning, defaults, return shapes and NaN behaviour
as the reference (``/root/reference/sea_ice_drift/pmlib.py``); the per-point MCC
loop (reference pmlib.py:430-448 and everything it calls) runs as ONE batched
launch of hand-written sm_100a kernels through the C ABI in
``include/sid_b200.h``.  There is no CPU implementation behind these functions:
without the CUDA library / a CUDA device they raise.

Kept on the host, as in the reference: the lon/lat <-> pixel transforms done by
the Nansat objects, the first-guess interpolation and the final re-gridding.
"""
from __future__ import absolute_import, print_function

import os
import time

import numpy as np
from scipy import ndimage
from scipy.spatial import cKDTree

from . import _lib
from ._lib import SID_TM_CCOEFF_NORMED, flags_from_kwargs, flags_from_options
from .lib import interpolation_poly, interpolation_near, _fill_gpi

TM_CCOEFF_NORMED = SID_TM_CCOEFF_NORMED          # == cv2.TM_CCOEFF_NORMED
DEFAULT_SRS = '+proj=latlong +datum=WGS84 +ellps=WGS84 +no_defs'

# module-level state with the reference's names (reference pmlib.py:33-34), so code that
# drives use_mcc_mp by hand keeps working
shared_args = None
shared_kwargs = None

def _ctx(kwargs=None):
    device = None if not kwargs else kwargs.get('device')
    return _lib.default_context(device)


def _is_builtin_matcher(fn):
    if fn is None or fn is match_template:
        return True
    return getattr(fn, '__name__', '') == 'matchTemplate' and 'cv2' in (getattr(fn, '__module__', '') or 'cv2')


def match_template(image, templ, method=TM_CCOEFF_NORMED, **kwargs):
    """GPU ``template_matcher``: same call shape as ``cv2.matchTemplate(image, templ,
    cv2.TM_CCOEFF_NORMED)`` (reference pmlib.py:120, 156); float32 map of shape
    (H-th+1, W-tw+1)."""
    return _ctx(kwargs).match_template(image, templ, method)


def get_hessian(ccm, hes_norm=True, hes_smth=False, **kwargs):
    """Peak-sharpness map of a cross-correlation matrix (reference pmlib.py:36-59)."""
    return _ctx(kwargs).get_hessian(ccm, flags_from_kwargs(hes_norm, hes_smth, False))


def get_template(img, c, r, a, s, rot_order=0, **kwargs):
    """Rotated/shifted s x s uint8 template around (c, r) (reference pmlib.py:89-115)."""
    return _ctx(kwargs).get_template(img, c, r, a, s, rot_order)


try:                                        # the reference's default (pmlib.py:120); recognised and run on the GPU
    import cv2 as _cv2
    _DEFAULT_MATCHER = _cv2.matchTemplate
except ImportError:                         # no OpenCV installed: same behaviour, our own callable as the default
    _DEFAULT_MATCHER = match_template


def rotate_and_match(img1, c1, r1, img_size, image2, alpha0,
                     angles=[-3, 0, 3],
                     mtype=TM_CCOEFF_NORMED,
                     template_matcher=_DEFAULT_MATCHER,
                     mcc_norm=False,
                     **kwargs):
    """Best match of the rotated templates of one point inside ``image2``
    (reference pmlib.py:117-174).  Returns ``(dc, dr, best_a, best_r, best_h,
    best_result, best_template)`` or seven NaNs when a template holds a 0 pixel.

    ``template_matcher`` left at None, set to :func:`match_template` or to
    ``cv2.matchTemplate`` selects the GPU matcher; any other callable is honoured
    as the reference's plug-in and called once per angle.

    ``subpixel=True`` (extension): ``dc`` / ``dr`` refined to sub-pixel precision by a parabola through the peak of
    ``best_result`` and its two neighbours per axis (``SID_SUBPIXEL``, include/sid_b200.h); needs the built-in
    matcher.

    ``masked=True`` (extension): where a template holds a 0 pixel, match by the Pearson correlation over the
    templates' valid pixels instead of returning NaNs, when every angle's template has at least half its pixels valid
    and is not flat (``SID_MASKED``, include/sid_b200.h); needs the built-in matcher."""
    rot_order = kwargs.get('rot_order', 0)
    for option in ('subpixel', 'masked'):
        if kwargs.get(option) and not _is_builtin_matcher(template_matcher):
            raise ValueError("%s=True needs the built-in matcher (template_matcher None, match_template or "
                             "cv2.matchTemplate)" % option)
    flags = flags_from_options(dict(kwargs, mcc_norm=mcc_norm))
    ctx = _ctx(kwargs)
    if _is_builtin_matcher(template_matcher):
        res = ctx.rotate_and_match(img1, c1, r1, img_size, image2, list(angles), alpha0, rot_order, flags, mtype)
        if res is None:
            return (np.nan,) * 7
        dc, dr, ia, r, h, ccm, tpl = res
        return dc, dr, angles[ia], r, h, ccm, tpl
    # user-supplied matcher: templates and Hessian still come from the GPU
    best = None
    for angle in angles:
        tpl = ctx.get_template(img1, c1, r1, angle - alpha0, img_size, rot_order)
        if tpl.min() == 0:
            return (np.nan,) * 7
        ccm = template_matcher(image2, tpl, mtype)
        if best is None or ccm.max() > best[0]:
            best = (ccm.max(), angle, ccm, tpl, np.unravel_index(np.argmax(ccm), ccm.shape))
    peak, angle, ccm, tpl, ij = best
    h = ctx.get_hessian(ccm, flags & 3)[ij]
    dr = ij[0] - (image2.shape[0] - tpl.shape[0]) / 2.
    dc = ij[1] - (image2.shape[1] - tpl.shape[1]) / 2.
    if mcc_norm:
        peak = (peak - np.median(ccm)) / np.std(ccm)
    return dc, dr, angle, peak, h, ccm, tpl


def use_mcc_batch(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, **kwargs):
    """``use_mcc`` for every point at once: the body of the reference's Pool map
    (pmlib.py:436-448) as one fused kernel launch.  Returns an (N, 5) float64 table
    ``c2, r2, angle, r, h`` with NaN rows where the reference returns NaN.

    ``resident=True`` (extension): reuse the image pair uploaded by this context's previous call instead of
    uploading ``img1`` / ``img2`` again -- an explicit contract, for callers that run several grids or kwargs
    sets over one pair; raises nothing and uploads anyway when no pair is resident.

    ``return_maps=True`` (extension): return ``(table, maps, templates)`` where ``maps[i]`` is what
    ``rotate_and_match(...)[5]`` gives for point i's window -- the float32 NCC map of the winning angle -- or None
    where the row is NaN, and ``templates[i]`` (an (N, img_size, img_size) uint8 array) is ``[6]``, the winning
    angle's template (zeros where the row is NaN).

    ``subpixel=True`` (extension): ``c2`` / ``r2`` refined to sub-pixel precision on the device by a parabola through
    the peak of the winning map and its two neighbours per axis (``SID_SUBPIXEL``, include/sid_b200.h); the other
    columns, the NaN rows and the maps of ``return_maps`` are unchanged.  Needs the built-in matcher.

    ``masked=True`` (extension): rows that are NaN because a template holds a 0 pixel (land, no-data) are matched by
    the Pearson correlation over the templates' valid pixels where every angle's template has at least
    ``ceil(img_size**2 / 2)`` valid pixels and is not flat (``SID_MASKED``, include/sid_b200.h); ``return_maps`` then
    gives their masked maps and templates.  Every other row is unchanged.  Needs the built-in matcher.

    ``peaks=True`` (extension): also return the three next-best peaks of every row's winning map (``SID_PEAKS``,
    include/sid_b200.h) as an (N, 3, 4) float64 array of c2, r2, r, h per peak, NaN where missing, appended to what the
    call returns: ``(table, peaks)`` or ``(table, maps, templates, peaks)``.  The table is unchanged.  Needs the
    built-in matcher.

    ``uncertainty=True`` (extension, needs ``subpixel=True``): also return the covariance of every row's sub-pixel
    offsets by correlation statistics (``SID_UNCERT``, include/sid_b200.h) as an (N, 3) float64 array of var_c, var_r,
    cov_cr in image-2 pixels^2, NaN where undefined, appended last (after the peaks when both are asked for).  The
    table is unchanged.  Needs the built-in matcher."""
    matcher = kwargs.get('template_matcher')
    return_maps = kwargs.get('return_maps', False)
    want_peaks = kwargs.get('peaks', False)
    want_unc = kwargs.get('uncertainty', False)
    for option in ('return_maps', 'subpixel', 'masked', 'peaks', 'uncertainty'):
        if kwargs.get(option) and not _is_builtin_matcher(matcher):
            raise ValueError("%s=True needs the built-in matcher (template_matcher None, match_template or "
                             "cv2.matchTemplate)" % option)
    if not _is_builtin_matcher(matcher):
        rows = [use_mcc(a, b, c, d, e, img1, img2, img_size, alpha0, **kwargs)
                for a, b, c, d, e in zip(c1, r1, c2fg, r2fg, border)]
        return np.array(rows, dtype=np.float64).reshape(-1, 5)
    flags = flags_from_options(kwargs) | (_lib.SID_PEAKS if want_peaks else 0)
    ctx = _ctx(kwargs)
    args = (c1, r1, c2fg, r2fg, border, img_size, list(kwargs.get('angles', [-3, 0, 3])), alpha0,
            kwargs.get('rot_order', 0), flags, kwargs.get('mtype', TM_CCOEFF_NORMED))
    # The pair is uploaded on EVERY call (overlapped with the matching, so it costs ~1.5 ms per EW pair) unless
    # the caller states explicitly that the pair of its previous call is still the one to match: the library
    # never infers identity from pointers or sampled checksums (an in-place edit such as masking land, or a new
    # array at a recycled address, would silently match against the old pair).
    if return_maps:
        if not (kwargs.get('resident') and ctx._pair_key is not None):
            ctx.set_pair(img1, img2)
            ctx._pair_key = (np.shape(img1), np.shape(img2))
        out = ctx.run_maps(*args)
    elif kwargs.get('resident') and ctx._pair_key is not None:
        out = ctx.run(*args)
    else:
        out = ctx.run_pair(img1, img2, *args)
        ctx._pair_key = (np.shape(img1), np.shape(img2))
    if not (want_peaks or want_unc):
        return out
    extra = ()
    n = len(out[0]) if return_maps else len(out)
    if want_peaks:
        extra += (ctx.peaks(n),)
    if want_unc:
        extra += (ctx.uncertainty(n),)
    return (out if return_maps else (out,)) + extra


def use_mcc(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, **kwargs):
    """MCC for one point (reference pmlib.py:176-212): ``(c2, r2, a, r, h)``."""
    matcher = kwargs.get('template_matcher')
    if not _is_builtin_matcher(matcher):
        hws = int(img_size / 2.)
        image = img2[int(r2fg - hws - border):int(r2fg + hws + border + 1),
                     int(c2fg - hws - border):int(c2fg + hws + border + 1)]
        dc, dr, a, r, h = rotate_and_match(img1, c1, r1, img_size, image, alpha0, **kwargs)[:5]
        return c2fg + dc, r2fg + dr, a, r, h
    row = use_mcc_batch([c1], [r1], [c2fg], [r2fg], [border], img1, img2, img_size, alpha0, **kwargs)[0]
    if np.isnan(row[0]):
        return np.nan, np.nan, np.nan, np.nan, np.nan
    angles = list(kwargs.get('angles', [-3, 0, 3]))
    angle = angles[int(np.argmin(np.abs(np.asarray(angles, dtype=np.float64) - row[2])))]
    return row[0], row[1], angle, np.float32(row[3]), np.float32(row[4])


def use_mcc_mp(i):
    """``use_mcc`` on point ``i`` of the module-level ``shared_args`` /
    ``shared_kwargs`` (reference pmlib.py:214-247)."""
    sa = shared_args
    return use_mcc(sa[0][i], sa[1][i], sa[2][i], sa[3][i], sa[4][i], sa[5], sa[6], sa[7], sa[8], **shared_kwargs)


def get_distance_to_nearest_keypoint(x1, y1, shape):
    """Full-resolution image of the distance (px) to the nearest keypoint
    (reference pmlib.py:61-77)."""
    seed = np.zeros(shape, dtype=bool)
    seed[np.uint16(y1), np.uint16(x1)] = True
    return ndimage.distance_transform_edt(~seed, return_distances=True, return_indices=False)


def _distance_at(x1, y1, cols, rows):
    """Same values as ``get_distance_to_nearest_keypoint(...)[rows, cols]`` without the
    full-image transform: exact nearest-seed distance between integer pixels."""
    seeds = np.column_stack([np.uint16(y1).astype(np.float64), np.uint16(x1).astype(np.float64)])
    dist, _ = cKDTree(seeds).query(np.column_stack([rows.astype(np.float64), cols.astype(np.float64)]))
    return dist


def get_initial_rotation(n1, n2):
    """Angle (degrees) between the two scenes' pixel grids (reference pmlib.py:79-87)."""
    lons, lats = n2.get_corners()
    x0, y0 = n1.transform_points([lons[0]], [lats[0]], 1)
    x1, y1 = n1.transform_points([lons[1]], [lats[1]], 1)
    return np.degrees(np.arctan2(x1 - x0, y1 - y0)[0])


def _device_present():
    """True when a CUDA device (and the library) can be used for the first guess."""
    try:
        _lib.default_context()
        return True
    except Exception:
        return False


def _near_device(ctx, sx, sy, vx, vy, qx, qy, seeds=None):
    """interpolation_near(method='linear') (and optionally the nearest-seed distance) through sid_first_guess.
    Returns (vx_q, vy_q, dist, resolved, unique): ``resolved`` False when some point could not be decided numerically,
    ``unique`` False when some grid point lies in a cell of cocircular keypoints (triangulation not unique)."""
    kx, ky = seeds if seeds is not None else (np.zeros(0), np.zeros(0))
    ovx, ovy, dist, flag = ctx.first_guess(sx, sy, vx, vy, kx, ky, qx, qy)
    shape = np.shape(qx)
    return ovx.reshape(shape), ovy.reshape(shape), dist.reshape(shape), not np.any(flag == 2), not np.any(flag == 3)


def prepare_first_guess(c2pm1, r2pm1, n1, c1, r1, n2, c2, r2, img_size,
                        min_fg_pts=5, min_border=20, max_border=50, old_border=True, **kwargs):
    """First-guess position on image 2 and search radius for every grid point
    (reference pmlib.py:249-324): Delaunay-linear interpolation of the feature
    tracking vectors with a polynomial fallback outside their hull; the radius is
    the distance to the nearest keypoint clamped to [min_border, max_border].

    ``first_guess='auto'`` (the default where a CUDA device is present) evaluates the Delaunay-linear interpolant and
    the nearest-keypoint distances on the GPU without building a triangulation (``sid_first_guess``: every grid point
    finds its own Delaunay triangle by pivoting) and returns that when the result is unique -- then it equals the SciPy /
    reference values.  Where four keypoints are cocircular (integer pixel coordinates, e.g. ORB keypoints under an
    identity geolocation) the Delaunay triangulation is not unique and Qhull's arbitrary choice may differ: ``'auto'``
    then takes the SciPy path so that the result is always the reference's; ``first_guess='device'`` keeps the (equally
    valid) device result.  ``first_guess='host'`` is the SciPy path (one Qhull triangulation shared by both value sets,
    KD-tree distances), also taken for ``method != 'linear'``."""
    n2_shape = n2.shape()
    lon1, lat1 = n1.transform_points(c1, r1)
    c1n2, r1n2 = n2.transform_points(lon1, lat1, 1)
    c2p2, r2p2 = np.round(interpolation_poly(c1n2, r1n2, c2, r2, c2pm1, r2pm1, **kwargs))
    mode = kwargs.get('first_guess')
    if mode is None:
        mode = 'auto' if (kwargs.get('method', 'linear') == 'linear' and len(np.atleast_1d(c1)) >= 3
                          and _device_present()) else 'host'
    done = False
    if mode in ('device', 'auto'):
        ctx = _ctx(kwargs)
        c2pm1 = np.asarray(c2pm1, dtype=np.float64)
        r2pm1 = np.asarray(r2pm1, dtype=np.float64)
        inside = ((c2pm1 >= 0) * (c2pm1 < n2_shape[1]) * (r2pm1 >= 0) * (r2pm1 < n2_shape[0]))
        seeds = (np.uint16(c2).astype(np.float64), np.uint16(r2).astype(np.float64))
        integer_grid = np.array_equal(np.round(c2pm1), c2pm1) and np.array_equal(np.round(r2pm1), r2pm1)
        if old_border:
            vx, vy, dist, ok, unique = _near_device(ctx, c1n2, r1n2, c2, r2, c2pm1, r2pm1, seeds if integer_grid else None)
            ok = ok and (unique or mode == 'device')
            if ok and not integer_grid:      # the reference samples the distance image at the ROUNDED grid positions
                dist = _near_device(ctx, np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0),
                                    np.round(c2pm1).astype(np.int16).astype(np.float64),
                                    np.round(r2pm1).astype(np.int16).astype(np.float64), seeds)[2]
            if ok:
                c2fg, r2fg = np.round(vx), np.round(vy)
                border = np.zeros(c2pm1.size) + max_border
                border[inside.ravel()] = dist.ravel()[inside.ravel()]
                done = True
        else:
            c2tst, r2tst = interpolation_poly(c1n2, r1n2, c2, r2, c1n2, r1n2, **kwargs)
            vx, vy, _, ok, unique = _near_device(ctx, c1n2, r1n2, c2, r2, c2pm1, r2pm1)
            dx, dy, _, ok2, _ = _near_device(ctx, c1n2, r1n2, c2 - c2tst, r2 - r2tst, c2pm1, r2pm1)
            if ok and ok2 and (unique or mode == 'device'):
                c2fg, r2fg = np.round(vx), np.round(vy)
                border = np.hypot(dx, dy)
                done = True
    if not done:
        c2fg, r2fg = np.round(interpolation_near(c1n2, r1n2, c2, r2, c2pm1, r2pm1, **kwargs))
        if old_border:
            border = np.zeros(c2pm1.size) + max_border
            inside = ((c2pm1 >= 0) * (c2pm1 < n2_shape[1]) * (r2pm1 >= 0) * (r2pm1 < n2_shape[0]))
            border[inside] = _distance_at(c2, r2,
                                          np.round(c2pm1[inside]).astype(np.int16),
                                          np.round(r2pm1[inside]).astype(np.int16))
        else:
            c2tst, r2tst = interpolation_poly(c1n2, r1n2, c2, r2, c1n2, r1n2, **kwargs)
            c2dif, r2dif = interpolation_near(c1n2, r1n2, c2 - c2tst, r2 - r2tst, c2pm1, r2pm1, **kwargs)
            border = np.hypot(c2dif, r2dif)
    border[border < min_border] = min_border
    border[border > max_border] = max_border
    outside_hull = np.isnan(c2fg)
    border[outside_hull] = max_border
    border = np.floor(border)
    c2fg[outside_hull] = c2p2[outside_hull]
    r2fg[np.isnan(r2fg)] = r2p2[np.isnan(r2fg)]
    return c2fg, r2fg, border


COARSE_DEFAULTS = dict(factor=4, step=32, img_size=35, max_drift=100.0, min_quality=4.0, angles=[-3, 0, 3], seed=0)


def _incircle_zero(ax, ay, bx, by, cx, cy, dx, dy):
    """True where d lies exactly on the circle through a, b, c (int64 coordinates, exact)."""
    ax, ay, bx, by, cx, cy = ax - dx, ay - dy, bx - dx, by - dy, cx - dx, cy - dy
    a2, b2, c2 = ax * ax + ay * ay, bx * bx + by * by, cx * cx + cy * cy
    return ax * (by * c2 - b2 * cy) - ay * (bx * c2 - b2 * cx) + a2 * (bx * cy - by * cx) == 0


def coarse_lattice(shape1, step, seed):
    """Integer lattice ``step`` apart on a coarse image of ``shape1`` (rows, cols), every point moved by a seeded integer
    jitter of at most ``step // 4`` per axis.  Returns int64 (c1, r1) in row-major lattice order.

    On an exact lattice every Delaunay cell of the points is cocircular, so the triangulation that
    :func:`prepare_first_guess` interpolates over is not unique and its ``'auto'`` mode takes the Qhull path.  With the
    jitter, a cell can still be cocircular by chance (about one cell in 600 at ``step`` 16); the jitter of such a cell's
    first corner is drawn again until no lattice cell is.  That is all the redraw guarantees: four points of different
    cells (a sliver along the hull, a diamond across three rows) can still be cocircular -- none at ``step`` 16 and 32,
    a few at ``step`` 8 in DESIGN.md section 8 -- and ``'auto'`` then takes the Qhull path, with the same result."""
    if step < 4:
        raise ValueError("step must be at least 4 coarse pixels")
    rng = np.random.default_rng(seed)
    amp = step // 4
    xs = np.arange(step // 2, shape1[1], step, dtype=np.int64)
    ys = np.arange(step // 2, shape1[0], step, dtype=np.int64)
    gx, gy = np.meshgrid(xs, ys)
    jx = rng.integers(-amp, amp + 1, gx.shape)
    jy = rng.integers(-amp, amp + 1, gx.shape)
    for _ in range(64):
        c, r = gx + jx, gy + jy
        bad = _incircle_zero(c[:-1, :-1], r[:-1, :-1], c[:-1, 1:], r[:-1, 1:], c[1:, 1:], r[1:, 1:], c[1:, :-1], r[1:, :-1])
        if not bad.any():
            break
        iy, ix = np.nonzero(bad)
        jx[iy, ix] = rng.integers(-amp, amp + 1, iy.size)
        jy[iy, ix] = rng.integers(-amp, amp + 1, iy.size)
    return (gx + jx).ravel(), (gy + jy).ravel()


def coarse_inputs(n1, n2, shape1, shape2, factor, step, img_size, max_drift, seed=0):
    """The coarse matching problem of :func:`coarse_tracking` on coarse images of ``shape1`` / ``shape2``: the lattice
    points that pattern_matching's window rule keeps (in coarse pixels), their zero-drift first guess on coarse image 2
    from the geolocation of ``n1`` / ``n2``, the coarse border and the initial rotation.  Returns
    ``(c1, r1, c2fg, r2fg, border, alpha0)``; c1 ... border are float64 arrays, the border is
    ``ceil(max_drift / factor) + 2`` everywhere."""
    k = int(factor)
    c1, r1 = coarse_lattice(shape1, step, seed)
    c1, r1 = c1.astype(np.float64), r1.astype(np.float64)
    off = (k - 1) / 2.
    lon, lat = n1.transform_points(k * c1 + off, k * r1 + off)
    x2, y2 = n2.transform_points(lon, lat, 1)
    c2fg, r2fg = np.round((np.asarray(x2) - off) / k), np.round((np.asarray(y2) - off) / k)
    border = float(np.ceil(max_drift / k) + 2)
    hws = round(img_size / 2) + 1
    hws_hypot = np.hypot(hws, hws)
    with np.errstate(invalid='ignore'):
        gpi = ((c2fg - border - hws > 0) & (r2fg - border - hws > 0) &
               (c2fg + border + hws < shape2[1]) & (r2fg + border + hws < shape2[0]) &
               (c1 - hws_hypot > 0) & (r1 - hws_hypot > 0) & (c1 + hws_hypot < shape1[1]) & (r1 + hws_hypot < shape1[0]))
    return c1[gpi], r1[gpi], c2fg[gpi], r2fg[gpi], np.full(int(gpi.sum()), border), get_initial_rotation(n1, n2)


def coarse_matches(table, status, c1, r1, factor, img_size, min_quality):
    """Full-resolution matches ``(x1, y1, x2, y2)`` from the coarse table: rows with status valid, finite values and
    ``r * h > min_quality``.  Template pixel ``int(s / 2) + 1`` samples coarse image 1 at (c1, r1) and lies at
    ``c2 + 1`` in coarse image 2 for odd ``img_size`` s and at ``c2 + 1.5`` for even s; a coarse pixel j covers the
    full-resolution pixels ``k * j ... k * j + k - 1``, centred on ``k * j + (k - 1) / 2``."""
    k = int(factor)
    table = np.asarray(table, dtype=np.float64).reshape(-1, 5)
    with np.errstate(invalid='ignore'):
        keep = (np.asarray(status) == _lib.SID_PT_VALID) & np.isfinite(table).all(axis=1) & \
            (table[:, 3] * table[:, 4] > min_quality)
    off = (k - 1) / 2.
    delta = 1.0 if int(img_size) % 2 else 1.5
    return (k * c1[keep] + off, k * r1[keep] + off,
            k * (table[keep, 0] + delta) + off, k * (table[keep, 1] + delta) + off)


_coarse_buffers = {}


def _coarse_buffer(device, which, layout, nbytes):
    """Device buffer of coarse image ``which`` (torch uint8, 256-byte aligned by the allocator): one per device and image,
    grown when a call needs more bytes, so a process that sees many scene sizes keeps only the largest.  Zeroed when
    ``layout`` (the coarse shape and factor) differs from its previous use, so the pitch padding is 0 as after an
    upload.  The fill is queued on torch's current stream: the caller orders it before the context's work."""
    import torch
    buf, last = _coarse_buffers.get((device, which), (None, None))
    if buf is None or buf.numel() < nbytes:
        buf = torch.zeros(nbytes, dtype=torch.uint8, device=torch.device('cuda', device))
    elif last != layout:
        buf.zero_()
    _coarse_buffers[(device, which)] = (buf, layout)
    return buf


_coarse_contexts = {}


def coarse_tracking(n1, n2, **kwargs):
    """Feature-tracking matches without feature tracking: ``(x1, y1, x2, y2)``, full-resolution pixel coordinates on
    image 1 and image 2, what the reference's ``ftlib.feature_tracking`` returns, so they can go wherever its matches
    go (``prepare_first_guess``, ``pattern_matching``, ``SeaIceDrift.get_drift_PM``).

    The pair is made resident on the device and box-downsampled there by ``factor`` (``sid_downsample_pair``); a
    private context adopts the coarse pair and matches a jittered lattice ``step`` coarse pixels apart
    (:func:`coarse_lattice`) from the zero-drift first guess of the geolocation, border ``ceil(max_drift / factor) +
    2``, templates of ``img_size`` coarse pixels, ``angles`` around the initial rotation, default flags.  Matches with
    ``r * h > min_quality`` are mapped back to full resolution (:func:`coarse_matches`), in lattice order; their error
    is about ``factor / 2`` px.  No image leaves the device.  Keywords and defaults: ``factor`` 4 (2 ... 16), ``step``
    32 (the fastest whole drift call of steps 8 ... 32 on an EW-sized pair, DESIGN.md section 8), ``img_size`` 35, ``max_drift`` 100 (full-resolution px), ``min_quality`` 4.0, ``angles`` [-3, 0, 3], ``seed``
    0 (the lattice jitter), ``device``."""
    opts = dict(COARSE_DEFAULTS)
    opts.update((key, kwargs[key]) for key in COARSE_DEFAULTS if key in kwargs)
    k, s = int(opts['factor']), int(opts['img_size'])
    if not 2 <= k <= 16 or k != opts['factor']:
        raise ValueError("factor must be an integer in [2, 16]")
    if not 2 <= s <= 128:
        raise ValueError("img_size must be in [2, 128]")
    img1, img2 = _lib.as_u8_image(n1[1]), _lib.as_u8_image(n2[1])
    shape1 = (img1.shape[0] // k, img1.shape[1] // k)
    shape2 = (img2.shape[0] // k, img2.shape[1] // k)
    if min(shape1 + shape2) < s:
        raise ValueError("a %d x downsampled image (%s, %s) is smaller than one %d x %d template"
                         % (k, shape1, shape2, s, s))
    c1, r1, c2fg, r2fg, border, alpha0 = coarse_inputs(n1, n2, shape1, shape2, k, int(opts['step']), s,
                                                       float(opts['max_drift']), opts['seed'])
    if c1.size == 0:
        return tuple(np.zeros(0) for _ in range(4))
    import torch
    ctx = _ctx(kwargs)
    ctx.set_pair(img1, img2)
    bufs = []
    for which, shape in enumerate((shape1, shape2)):
        pitch, nbytes = _lib.pair_layout(*shape)
        buf = _coarse_buffer(ctx.device, which, (shape, k), nbytes)
        bufs.append((buf.data_ptr(), pitch, buf.numel()))
    # the buffers' zero fill runs on torch's current stream, the downsampling on the context's own (non-blocking) stream
    torch.cuda.current_stream(ctx.device).synchronize()
    ctx.downsample_pair(k, bufs[0], bufs[1])
    ctx.synchronize()                        # the private context's stream reads what the default one wrote
    key = (os.getpid(), ctx.device)
    coarse = _coarse_contexts.get(key)
    if coarse is None:
        coarse = _coarse_contexts[key] = _lib.Context(ctx.device)
    (p1, pitch1, b1), (p2, pitch2, b2) = bufs
    coarse.adopt_pair_device(p1, shape1, pitch1, b1, p2, shape2, pitch2, b2)
    table, status = coarse.run(c1, r1, c2fg, r2fg, border, s, list(opts['angles']), alpha0, 0, _lib.SID_HES_NORM,
                               want_status=True)
    return coarse_matches(table, status, c1, r1, k, s, float(opts['min_quality']))


OUTLIER_EPS, OUTLIER_THRESHOLD = 1.0, 2.0


def _grid_shape(shape):
    """(rows, cols) of a grid of ``shape``: a 1-D grid is one row."""
    shape = tuple(int(v) for v in shape)
    if len(shape) == 1:
        return 1, shape[0]
    if len(shape) != 2:
        raise ValueError("the grid must be 1-D or 2-D")
    return shape


def filter_outliers(table, peaks, gpi, c2pm1, r2pm1, eps=OUTLIER_EPS, threshold=OUTLIER_THRESHOLD, **kwargs):
    """Normalised median test (Westerweel & Scarano 2005) with replacement by secondary peaks, on the device
    (``sid_filter_outliers``, include/sid_b200.h), for callers with their own grid.  ``table``: the (N, 5) table of
    :func:`use_mcc_batch` for the True positions of the grid-shaped boolean ``gpi`` in row-major order; ``peaks``: its
    (N, 3, 4) ``peaks=True`` records; ``c2pm1`` / ``r2pm1``: the grid's image-2 pixel coordinates.  Every row is
    compared with its 8 grid neighbours' displacements ``(c2, r2) - round(c2pm1, r2pm1)``; an outlier takes its first
    secondary peak that passes the test, else becomes NaN.  Returns ``(table, flags)``: flags 0 kept, 1 ... 3 replaced
    by that peak, -1 rejected, -2 fewer than 3 neighbours (kept), -3 NaN row."""
    gpi = np.asarray(gpi, dtype=bool)
    return _ctx(kwargs).filter_outliers(_grid_shape(gpi.shape), gpi, c2pm1, r2pm1, table, peaks, eps, threshold)


def _nsr(srs):
    try:
        from nansat import NSR
        return NSR(srs)
    except ImportError:
        return srs


def pattern_matching(lon_pm1, lat_pm1, n1, c1, r1, n2, c2, r2,
                     margin=0, img_size=35, threads=5, srs=DEFAULT_SRS, **kwargs):
    """Pattern matching between two scenes (reference pmlib.py:326-497).

    Returns ``(u, v, a, r, h, lon2_dst, lat2_dst)``, each shaped like ``lon_pm1``
    with NaN where no vector could be found.  ``threads`` is accepted for
    compatibility and ignored: all grid points go through one GPU launch (or one
    launch per rank when ``torch.distributed`` is initialised, see sharding.py).

    ``subpixel=True`` (extension): sub-pixel drift vectors (see :func:`use_mcc_batch`).
    ``masked=True`` (extension): vectors next to land and no-data from the masked correlation (see
    :func:`use_mcc_batch`).
    ``outliers=True`` (extension): repair outlier vectors before the post-processing with the normalised median test
    over the grid and the three secondary peaks of every point (see :func:`filter_outliers`; ``outlier_eps`` default
    1.0 px, ``outlier_threshold`` default 2.0): replaced vectors come back in place, rejected ones as NaN.  Needs the
    built-in matcher and one GPU (no process group of more than one rank).  With ``return_flags=True`` an eighth grid
    (int32) holds every point's flag of :func:`filter_outliers`, and -4 where the point was not matched (outside the
    image or its search window).
    ``uncertainty=True`` (extension, needs ``subpixel=True``): two more grids ``su``, ``sv``, appended last (after the
    flags grid with ``return_flags=True``): the standard deviations of u and v, in their units, from the covariance of
    every vector's sub-pixel offsets by correlation statistics (see :func:`use_mcc_batch`), propagated through the
    Jacobian of image-2 pixel -> destination x/y at the vector's end point (the affine map's linear part on the device
    path, central differences of ``n2.transform_points`` at +-0.5 px on the host path).  NaN where u is NaN, where the
    peak lies on its map's edge, and, with ``outliers=True``, where a vector was replaced or rejected (its record
    describes the primary peak).  Needs the built-in matcher and one GPU."""
    from .sharding import use_mcc_batch_sharded, _dist
    outliers = kwargs.get('outliers', False)
    uncertainty = kwargs.get('uncertainty', False)
    for option in ('outliers', 'uncertainty'):
        if kwargs.get(option) and not _is_builtin_matcher(kwargs.get('template_matcher')):
            raise ValueError("%s=True needs the built-in matcher (template_matcher None, match_template or "
                             "cv2.matchTemplate)" % option)
        if kwargs.get(option) and _dist() is not None:
            raise ValueError("%s=True runs on one GPU: it is not supported under a process group of more than one "
                             "rank" % option)
    flags_from_options(kwargs)                  # uncertainty without subpixel: ValueError before any device work
    eps, threshold = kwargs.get('outlier_eps', OUTLIER_EPS), kwargs.get('outlier_threshold', OUTLIER_THRESHOLD)
    return_flags = kwargs.get('return_flags', False)
    if return_flags and not outliers:
        raise ValueError("return_flags=True needs outliers=True")
    t0 = time.time()
    img1, img2 = n1[1], n2[1]
    dst_shape = lon_pm1.shape

    c2pm1, r2pm1 = n2.transform_points(lon_pm1.flatten(), lat_pm1.flatten(), 1)
    c2pm1i, r2pm1i = np.round([c2pm1, r2pm1])
    lon1i, lat1i = n2.transform_points(c2pm1i, r2pm1i)
    c1pm1i, r1pm1i = n1.transform_points(lon1i, lat1i, 1)

    c2fg, r2fg, brd2 = prepare_first_guess(c2pm1i, r2pm1i, n1, c1, r1, n2, c2, r2, img_size, **kwargs)

    hws = round(img_size / 2) + 1
    hws_hypot = np.hypot(hws, hws)
    shape1, shape2 = n1.shape(), n2.shape()
    gpi = ((c2fg - brd2 - hws - margin > 0) *
           (r2fg - brd2 - hws - margin > 0) *
           (c2fg + brd2 + hws + margin < shape2[1]) *
           (r2fg + brd2 + hws + margin < shape2[0]) *
           (c1pm1i - hws_hypot - margin > 0) *
           (r1pm1i - hws_hypot - margin > 0) *
           (c1pm1i + hws_hypot + margin < shape1[1]) *
           (r1pm1i + hws_hypot + margin < shape1[0]))
    alpha0 = get_initial_rotation(n1, n2)
    grid_shape = _grid_shape(dst_shape)
    flag_grid = np.full(dst_shape, -4, np.int32)

    def finish(grids, flags=None, sigma=None):
        out = tuple(grids)
        if return_flags:
            if flags is not None:
                flag_grid.ravel()[np.flatnonzero(gpi)] = flags
            out += (flag_grid,)
        if uncertainty:
            if sigma is None:
                sigma = (np.full(dst_shape, np.nan), np.full(dst_shape, np.nan))
            out += tuple(sigma)
        return out

    def sigma_grids(unc, jac, flags):
        """su, sv grids from the (N, 3) records and the (N, 2, 2) Jacobians pixel -> x/y of the valid points"""
        vc, vr, cv = unc[:, 0], unc[:, 1], unc[:, 2]
        sig = []
        for k in range(2):
            j0, j1 = jac[:, k, 0], jac[:, k, 1]
            s = np.sqrt(j0 * j0 * vc + 2.0 * j0 * j1 * cv + j1 * j1 * vr)
            if flags is not None:
                s[(flags != 0) & (flags != -2)] = np.nan    # replaced / rejected: the record is the primary peak's
            sig.append(_fill_gpi(dst_shape, gpi, s))
        return sig

    # Affine geolocation (an object exposing ``affine_maps(srs) -> (pixel->x/y, pixel->lon/lat)`` 2 x 3 matrices, e.g.
    # synthetic.ArrayDomain): the post-processing below (reference pmlib.py:462-497) runs on the device too, on the
    # table the kernels left there -- the (N, 5) table never visits the host.  Real Nansat objects (GDAL, possibly
    # thin-plate-spline geolocation) take the host path.
    affine = getattr(n2, 'affine_maps', None)
    if (affine is not None and _dist() is None and kwargs.get('device_epilogue', True) and gpi.any()
            and _is_builtin_matcher(kwargs.get('template_matcher'))):
        xy, ll = affine(srs)
        ctx = _ctx(kwargs)
        flags = flags_from_options(kwargs) | (_lib.SID_PEAKS if outliers else 0)
        n_valid = int(np.count_nonzero(gpi))
        ctx.run_pair(img1, img2, c1pm1i[gpi], r1pm1i[gpi], c2fg[gpi], r2fg[gpi], brd2[gpi], img_size,
                     list(kwargs.get('angles', [-3, 0, 3])), alpha0, kwargs.get('rot_order', 0), flags,
                     kwargs.get('mtype', TM_CCOEFF_NORMED), keep_on_device=True)
        unc = ctx.uncertainty(n_valid) if uncertainty else None
        out_flags = None
        if outliers:
            out_flags = ctx.filter_outliers(grid_shape, gpi, c2pm1, r2pm1, eps=eps, threshold=threshold, in_place=True)[1]
        grids = ctx.pm_epilogue_affine(gpi, c2pm1, r2pm1, xy, ll)
        sigma = None
        if uncertainty:
            jac = np.broadcast_to(np.asarray(xy, dtype=np.float64).reshape(2, 3)[:, :2], (n_valid, 2, 2))
            sigma = sigma_grids(unc, jac, out_flags)
        print('\n', 'Pattern matching - OK! (%3.0f sec)' % (time.time() - t0))
        return finish((grid.reshape(dst_shape) for grid in grids), out_flags, sigma)
    out_flags = None
    unc = None
    if outliers or uncertainty:
        extra = use_mcc_batch(c1pm1i[gpi], r1pm1i[gpi], c2fg[gpi], r2fg[gpi], brd2[gpi],
                              img1, img2, img_size, alpha0, **dict(kwargs, peaks=outliers))
        results = extra[0]
        unc = extra[-1] if uncertainty else None
        if outliers and len(results):
            results, out_flags = _ctx(kwargs).filter_outliers(grid_shape, gpi, c2pm1, r2pm1, results, extra[1], eps,
                                                              threshold)
    else:
        results = use_mcc_batch_sharded(c1pm1i[gpi], r1pm1i[gpi], c2fg[gpi], r2fg[gpi], brd2[gpi],
                                        img1, img2, img_size, alpha0, **kwargs)

    print('\n', 'Pattern matching - OK! (%3.0f sec)' % (time.time() - t0))
    if len(results) == 0:
        nan_grid = np.zeros(dst_shape) + np.nan
        return finish(nan_grid.copy() for _ in range(7))

    c2pm2 = results[:, 0] + (c2pm1 - c2pm1i)[gpi]
    r2pm2 = results[:, 1] + (r2pm1 - r2pm1i)[gpi]
    nsr = _nsr(srs)
    xpm1, ypm1 = n2.transform_points(c2pm1, r2pm1, 0, nsr)
    xpm2, ypm2 = n2.transform_points(c2pm2, r2pm2, 0, nsr)
    lon_pm2, lat_pm2 = n2.transform_points(c2pm2, r2pm2, 0)
    u = _fill_gpi(dst_shape, gpi, xpm2) - xpm1.reshape(dst_shape)
    v = _fill_gpi(dst_shape, gpi, ypm2) - ypm1.reshape(dst_shape)
    a = _fill_gpi(dst_shape, gpi, results[:, 2])
    r = _fill_gpi(dst_shape, gpi, results[:, 3])
    h = _fill_gpi(dst_shape, gpi, results[:, 4])
    sigma = None
    if uncertainty:
        # Jacobian of pixel -> x/y at the end point (c2pm2, r2pm2) by central differences at +-0.5 px
        jac = np.empty((len(results), 2, 2))
        for k, (dc, dr) in enumerate(((0.5, 0.0), (0.0, 0.5))):
            xp, yp = n2.transform_points(c2pm2 + dc, r2pm2 + dr, 0, nsr)
            xm, ym = n2.transform_points(c2pm2 - dc, r2pm2 - dr, 0, nsr)
            jac[:, 0, k] = np.asarray(xp) - np.asarray(xm)
            jac[:, 1, k] = np.asarray(yp) - np.asarray(ym)
        sigma = sigma_grids(unc, jac, out_flags)
    return finish((u, v, a, r, h, _fill_gpi(dst_shape, gpi, lon_pm2), _fill_gpi(dst_shape, gpi, lat_pm2)), out_flags,
                  sigma)
