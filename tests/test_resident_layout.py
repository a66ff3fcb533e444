"""Every result depends only on the image bytes it covers.

A resident image has the row pitch of ``sid_pair_layout`` (round_up(cols, 16) + 16: 16 ... 31 bytes of padding per row)
and 4096 bytes of tail slack past its last row.  The kernels read some of these bytes (whole words of the window rows,
16-byte chunks of the downsampler, TMA boxes), and the bytes hold whatever was there before: the caller's data in an
adopted buffer, the previous (larger) pair's pixels in a reused owned buffer, the previous pair's rows in the upload
bands that have not arrived yet.  The reference samples 0 outside image 1 (scipy's ``cval=0``), so a kernel that read
such a byte where the reference reads 0 would pass on zero padding and fail here.

A. Adopted pairs whose whole allocation is first filled with a poison (0xFF, or a seeded pattern without zero bytes)
   and then gets the image in ``[:rows, :cols]``, with the minimal pitch and with 48 bytes more; widths with
   cols % 16 in {1, 15} and rows1 != rows2.  One dispatch row per kernel variant, with points whose templates cross
   image 1's right and bottom edge by 1 ... hws px (NaN rows) or end exactly on / just before its last column and row
   (valid rows), at relative angles 0 and +-45 degrees, and windows clipped at image 2's right and bottom edge.  Also
   run_maps, the sub-pixel flag, run_device and the downsampler for every factor 2 ... 16.
B. One owned context that first holds a large zero-free pair and then gets smaller ones (fewer rows, narrower pitch)
   through every upload path, the single-call functions after a larger resident pair, and the series driver with
   pairs in shrinking order.
C. Upload-band edges: the band plan of ``run_host`` restated in Python; points whose last template or window row is
   the row before or the first row of each band, the reading coordinate in 0.25 px steps, on a pair whose
   not-yet-arrived rows hold another pair's pixels, and pairs of points whose launch count shows which band run_host
   gave the point at a boundary.  The template term of the bound, r1 + 0.707 (s + 2) + 3, lies 4.1 rows (plus the
   rounding) beyond the last row a template reads (r1 + 0.707 (s - 1) + 1 at a relative angle of -45 degrees), so a
   bound up to 4 rows tighter is still safe; the launch-count test pins the bound itself.

Every GPU table equals the exact C oracle (status included) and the same call on zero-padded buffers, bit for bit."""
import functools
import math
import os
import re

import numpy as np
import pytest

from sea_ice_drift_b200 import _lib
from sea_ice_drift_b200 import synthetic as syn
from oracle import c_oracle as co
from tests.helpers import assert_equals_exact_oracle
from tests.test_coarse_tracking import downsample_ref
from tests.test_gpu_maps import window_rule
from tests.test_size_dispatch_sweep import (ROWS, WS, TC, IMMA, DP4A, A3, speckle_pair, speckle_points, opts_of,
                                            flags_of, launch_lines, check_launch)

TAIL_SLACK = 4096                            # IMG_TAIL_SLACK: bytes of sid_pair_layout past the last row
SHAPE1, SHAPE2 = (560, 545), (553, 559)      # cols % 16 = 1 / 15, rows1 != rows2
ALPHAS = (0.0, 45.0, -45.0)                  # relative angles 0 and -+45 degrees for the angle lists around 0
POISONS = ("ff", "rand")
EXTRA_PITCH = (0, 48)


def padded_pitch(cols):
    return (cols + 15) // 16 * 16 + 16


def layout_bytes(rows, cols, pitch=None):
    pitch = padded_pitch(cols) if pitch is None else pitch
    return pitch, pitch * rows + TAIL_SLACK


def poison_bytes(kind, n, seed):
    if kind == "ff":
        return np.full(n, 0xFF, np.uint8)
    return np.random.default_rng(seed).integers(1, 256, n).astype(np.uint8)


@functools.lru_cache(maxsize=None)
def layout_pair():
    img1, img2 = speckle_pair()
    return (np.ascontiguousarray(img1[:SHAPE1[0], :SHAPE1[1]]), np.ascontiguousarray(img2[:SHAPE2[0], :SHAPE2[1]]))


# ------------------------------------------------------------------------------------------------ template geometry
def template_extent(c1, r1, s, angle, alpha0):
    """(largest sample row, largest sample column) of the template of (c1, r1): the four corners of the affine map,
    in the C oracle's arithmetic (row = (off0 + i cos) + j sin, col = (off1 + i (-sin)) + j cos, no FMA)."""
    cs, sn, sh0, sh1 = _lib.angle_table([angle], alpha0, s)[0]
    off0, off1 = r1 - sh0, c1 - sh1
    corners = [(float(i), float(j)) for i in (0, s - 1) for j in (0, s - 1)]
    rows = [(off0 + i * cs) + j * sn for i, j in corners]
    cols = [(off1 + i * (-sn)) + j * cs for i, j in corners]
    return max(rows), max(cols)


def place_edge(s, angles, alpha0, axis, other, target, crossing):
    """Row (axis 0) or column (axis 1) of the point whose template reaches ``target`` along that axis: crossing, every
    angle's largest sample coordinate is >= target; otherwise every angle's is <= target (the other coordinate is
    ``other``)."""
    def reach(v):
        pos = (other, v) if axis == 0 else (v, other)
        return [template_extent(pos[0], pos[1], s, a, alpha0)[axis] for a in angles]
    v = target - (min(reach(0.0)) if crossing else max(reach(0.0)))
    for _ in range(64):
        ext = reach(v)
        if (min(ext) >= target) if crossing else (max(ext) <= target):
            return v
        v = np.nextafter(v, np.inf if crossing else -np.inf)
    raise AssertionError("no placement for %r" % ((s, angles, alpha0, axis, target),))


def crossings(hws):
    """1 ... hws px: all of them for small templates, a spread for large ones."""
    return sorted({d for d in (1, 2, 3, 4, 5, 7, 8, 11, 15, 16, hws // 2, hws - 1, hws) if 1 <= d <= hws})


def layout_points(s, lo, hi, angles, alpha0):
    """speckle_points (grid, NaN row, rejected rows, clipped windows, fractional values; border hi sizes the launch)
    on the layout pair, plus: templates crossing image 1's right / bottom edge by 1 ... hws px (NaN rows), templates
    whose last sample column / row is the last one or lies just before it (valid rows; with rot_order=1 the bilinear
    neighbours are the last column / row), and windows clipped at image 2's right / bottom edge.
    Returns (pts, roles): roles maps "nan_edge" / "last_line" / "clipped" to point indices."""
    (rows1, cols1), (rows2, cols2) = SHAPE1, SHAPE2
    hws = int(s / 2.)
    c1, r1, c2, r2, brd = [list(v) for v in speckle_points(s, lo, hi)]
    roles = {"nan_edge": [], "last_line": [], "clipped": []}
    mid1r, mid1c, mid2r, mid2c = rows1 / 2., cols1 / 2., float(rows2 // 2), float(cols2 // 2)

    def add(role, a, b, c, d, e=lo):
        roles[role].append(len(c1))
        c1.append(a), r1.append(b), c2.append(c), r2.append(d), brd.append(float(e))
    for d in crossings(hws):
        add("nan_edge", place_edge(s, angles, alpha0, 1, mid1r, cols1 - 1 + d, True), mid1r, mid2c, mid2r)
        add("nan_edge", mid1c, place_edge(s, angles, alpha0, 0, mid1c, rows1 - 1 + d, True), mid2c, mid2r)
    for f in (0.0, 0.25, 0.5, 0.75):
        add("last_line", place_edge(s, angles, alpha0, 1, mid1r + 3, cols1 - 1 - f, False), mid1r + 3, mid2c, mid2r)
        add("last_line", mid1c - 3, place_edge(s, angles, alpha0, 0, mid1c - 3, rows1 - 1 - f, False), mid2c, mid2r)
    for e in sorted({1, lo // 2 + 1, lo}):
        far_c, far_r = float(cols2 - 1 - hws - lo + e), float(rows2 - 1 - hws - lo + e)
        add("clipped", mid1c - 5, mid1r + 5, far_c, mid2r - 7)
        add("clipped", mid1c + 5, mid1r - 5, mid2c + 7, far_r)
        add("clipped", mid1c + 9, mid1r + 9, far_c, far_r)
    pts = [np.asarray(v, dtype=np.float64) for v in (c1, r1, c2, r2, brd)]
    return pts, {k: np.asarray(v, dtype=np.int64) for k, v in roles.items()}


def check_roles(pts, roles, st, s, img2):
    """The inputs reach the special rows they claim (judged on a status that equals the oracle's)."""
    assert roles["nan_edge"].size >= 2 and (st[roles["nan_edge"]] == 0).all(), st[roles["nan_edge"]]
    assert (st[roles["last_line"]] == 1).all(), st[roles["last_line"]]
    hws = int(s / 2.)
    for i in roles["clipped"]:
        rule = window_rule(img2, s, *[p[i] for p in pts])
        full = 2 * hws + 2 * int(math.ceil(pts[4][i])) + 1 - s + 1
        assert st[i] == 1 and rule is not None and min(rule) < full, (i, rule, full)
    assert (st == 0).sum() > roles["nan_edge"].size and (st == -1).sum() >= 2


@functools.lru_cache(maxsize=None)
def layout_oracle(s, angles, lo, hi, flag_set, alpha0):
    img1, img2 = layout_pair()
    pts, _ = layout_points(s, lo, hi, list(angles), alpha0)
    return co.use_mcc_batch(*pts, img1, img2, s, alpha0, angles=list(angles), **opts_of(flag_set))


# One dispatch row per kernel variant (rows of the img_size sweep; the dp4a row is forced through SID_PM_PATH)
A_ROW_IDS = ["s35_ws3_b21", "s35_ws2_b22", "s80_ws2_b7", "s2_tc_smem_b24", "s4_tc_smem_b26", "s4_tc_global_b27",
             "s35_tc_split_b37", "s35_tc_fused_b38", "s96_imma_b48", "s112_imma_b16", "s128_imma_ldg_b39"]
A_ROWS = [r for r in ROWS if r[0] in A_ROW_IDS] + \
    [("s35_dp4a_b21", 35, A3, (19, 21), "rot_order1", {"SID_PM_PATH": "dp4a"}, DP4A, dict())]


# ==================================================================================================== CPU tests
def test_a_rows_cover_every_variant():
    assert len(A_ROWS) == len(A_ROW_IDS) + 1
    kinds = {(r[6], r[7].get("nstat"), r[7].get("kidx"), r[7].get("tma"), r[7].get("tail") is None) for r in A_ROWS}
    assert {(WS, 3), (WS, 2)} <= {(k[0], k[1]) for k in kinds}
    assert {(TC, 9), (TC, 8)} <= {(k[0], k[2]) for k in kinds}
    assert {(IMMA, 1), (IMMA, 0)} <= {(k[0], k[3]) for k in kinds}
    assert {True, False} <= {k[4] for k in kinds if k[0] == TC}
    assert any(r[6] == DP4A for r in A_ROWS) and any(r[4] == "rot_order1" for r in A_ROWS)


def test_layout_shapes_and_pitches():
    (rows1, cols1), (rows2, cols2) = SHAPE1, SHAPE2
    assert {cols1 % 16, cols2 % 16} == {1, 15} and rows1 != rows2
    assert padded_pitch(cols1) - cols1 == 31 and padded_pitch(cols2) - cols2 == 17
    for cols in (1, 15, 16, 17, 545, 559):
        assert _lib.pair_layout(7, cols) == layout_bytes(7, cols)


@pytest.mark.parametrize("row", A_ROWS, ids=[r[0] for r in A_ROWS])
def test_layout_points_reach_their_rows(row):
    """Every point set of part A holds NaN rows from image-1 edges, valid rows on the last column / row and clipped
    windows, judged on the exact oracle's table; the crossing templates really cross and the others really do not."""
    rid, s, angles, (lo, hi), fs, env, kernel, attrs = row
    img1, img2 = layout_pair()
    for alpha0 in ALPHAS:
        pts, roles = layout_points(s, lo, hi, angles, alpha0)
        assert np.nanmax(np.ceil(pts[4])) == hi and pts[0].size < 256
        tab, st = layout_oracle(s, tuple(angles), lo, hi, fs, alpha0)
        check_roles(pts, roles, st, s, img2)
        for i in roles["nan_edge"]:
            ext = [template_extent(pts[0][i], pts[1][i], s, a, alpha0) for a in angles]
            assert min(max(e[0] - (SHAPE1[0] - 1), e[1] - (SHAPE1[1] - 1)) for e in ext) > 0
        for i in roles["last_line"]:
            ext = [template_extent(pts[0][i], pts[1][i], s, a, alpha0) for a in angles]
            assert max(e[0] for e in ext) <= SHAPE1[0] - 1 and max(e[1] for e in ext) <= SHAPE1[1] - 1
            assert max(max(e[0] for e in ext) - (SHAPE1[0] - 1), max(e[1] for e in ext) - (SHAPE1[1] - 1)) >= -0.75 - 1e-9


# ------------------------------------------------------------------------------------------------ C: the band plan
MAX_BANDS = 16


def band_weights(max_rows, plan=None, bands=None):
    """run_host's band weights: the default taper, SID_BANDS=n equal bands, SID_BAND_PLAN="w0,w1,..." (positive
    values only, at most MAX_BANDS)."""
    if max_rows >= 8192:
        w = [6, 6, 6, 6, 6, 5, 4, 3, 2, 1]
    else:
        w = [1.0] * max(1, min(8, max_rows // 512))
    if bands is not None:
        w = [1.0] * max(1, min(MAX_BANDS, int(bands)))
    if plan is not None:
        v = []
        for tok in plan.split(","):                 # strtod up to the first token that is no number
            try:
                x = float(tok)
            except ValueError:
                break
            if x > 0.0 and len(v) < MAX_BANDS:
                v.append(x)
        if v:
            w = v
    return [float(x) for x in w]


def band_lo(max_rows, weights):
    """First row of each band (multiples of 64) and max_rows at the end, as run_host computes them."""
    nb = len(weights)
    lo = [0] * (nb + 1)
    total, acc = sum(weights), 0.0
    for k in range(1, nb):
        acc += weights[k - 1]
        y = int(float(max_rows) * acc / total / 64.0 + 0.5) * 64
        lo[k] = max(lo[k - 1], min(max_rows, y))
    lo[nb] = max_rows
    return lo


def band_ext(s):
    """Template reach around (c1, r1) that run_host allows for, incl. rounding and bilinear neighbours."""
    return 0.5 * math.sqrt(2.0) * (s + 2) + 3.0


def point_need(r1, r2fg, border, s):
    """Last image row (+ margin) a point may read: its band is the first one holding that row."""
    v = int(math.ceil(border)) if np.isfinite(border) and 0.0 <= border < 4096.0 else 0
    if not (np.isfinite(r1) and np.isfinite(r2fg)):
        return 0.0
    return max(r1 + band_ext(s), r2fg + s // 2 + v + 2.0)


def point_band(lo, need):
    nb = len(lo) - 1
    max_rows = lo[-1]
    of64 = [nb - 1] * (max_rows // 64 + 2)
    j = 0
    for k in range(nb):
        while j * 64 < lo[k + 1] and j < len(of64):
            of64[j] = k
            j += 1
    if need <= 0.0:
        return 0
    return of64[int(min(float(len(of64) - 1), need / 64.0))]


def predicted_launches(lo, pts, s, limit):
    """The (band, class) pairs run_host launches: one launch per non-empty pair; the small class (borders <= the
    pm_ws_kernel limit) is split off only when it has >= 256 points, one border >= 1 and a larger border exists."""
    c1, r1, c2, r2, b = pts
    ib = [int(math.ceil(x)) if np.isfinite(x) and 0.0 <= x < 4096.0 else 0 for x in b]
    bands = [point_band(lo, point_need(r1[i], r2[i], b[i], s)) if len(lo) > 2 else 0 for i in range(c1.size)]
    small = [limit is not None and v <= limit for v in ib]
    two = limit is not None and limit < max(ib) and sum(small) >= 256 and max(v for v in ib if v <= limit) >= 1
    pairs = {(k, bool(sm) and two) for k, sm in zip(bands, small)}
    return pairs, bands


def test_band_plan_restatement_hand_cases():
    assert band_weights(1700) == [1.0] * 3 and band_weights(511) == [1.0] and band_weights(9000)[0] == 6
    assert band_weights(1700, plan="2,0,x") == [2.0] and band_weights(1700, bands=40) == [1.0] * MAX_BANDS
    assert band_lo(1700, [1.0] * 3) == [0, 576, 1152, 1700]
    assert band_lo(1700, [1.0] * 12) == [0, 128, 256, 448, 576, 704, 832, 960, 1152, 1280, 1408, 1536, 1700]
    assert band_lo(100, [1.0] * 4) == [0, 0, 64, 64, 100]                 # empty bands are kept
    assert band_lo(10400, band_weights(10400))[:3] == [0, 1408, 2752]     # 10400 * 6 / 45 / 64 = 21.7 -> 22 * 64
    lo = band_lo(1700, [1.0] * 3)
    assert band_ext(35) == pytest.approx(29.163, abs=1e-3)
    assert point_need(100.0, 90.0, 20.5, 35) == 90.0 + 17 + 21 + 2.0         # window-limited, border ceiled
    assert point_need(100.0, 90.0, 2.0, 35) == 100.0 + band_ext(35)          # template-limited
    assert point_need(np.nan, 90.0, 2.0, 35) == 0.0 and point_need(100.0, 90.0, np.inf, 35) == 100.0 + band_ext(35)
    assert [point_band(lo, x) for x in (-5.0, 0.0, 575.99, 576.0, 1151.9, 1152.0, 1699.0, 1800.0, 9e9)] == \
        [0, 0, 0, 1, 1, 2, 2, 2, 2]
    pts = [np.zeros(300), np.full(300, 10.0), np.zeros(300), np.full(300, 10.0), np.full(300, 4.0)]
    pts[4][:10] = 30.0
    pairs, _ = predicted_launches(lo, pts, 35, 22)
    assert pairs == {(0, False), (0, True)}
    assert predicted_launches(lo, [p[:200] for p in pts], 35, 22)[0] == {(0, False)}       # < 256 small points


BAND_SHAPE1, BAND_SHAPE2 = (1700, 700), (1690, 703)
BAND_PLANS = {"plan12": "1,1,1,1,1,1,1,1,1,1,1,1", "default": None}
BAND_STEPS = (0.0, 0.25, 0.5, 0.75)
BAND_ALPHA0, BAND_ANGLES = 45.0, [-3, 0, 3]
# (img_size, border of the template-limited points, border of the window-limited points, filler border, ws limit or
#  None) -- s = 2 and 35 split each band into the pm_ws_kernel class and the larger borders (limits 23 and 22 at three
#  angles: the img_size sweep's rows s2_ws_b23 / s2_tc_smem_b24 and s35_ws2_b22 / s35_tc_b23)
BAND_SIZES = [(2, 1, 24, 3, 23), (34, 2, 30, 4, None), (35, 2, 24, 4, 22), (128, 2, 30, 2, None)]


def template_read_row(c1, r1, s, angles, alpha0, rot_order):
    """The last image-1 row a point's templates read: the largest corner row over the angles, rounded (rot_order 0)
    or its bilinear neighbour below (rot_order 1)."""
    m = max(template_extent(c1, r1, s, a, alpha0)[0] for a in angles)
    return math.floor(m) + 1 if rot_order else math.floor(m + 0.5)


def window_read_row(r2fg, border, s, rows2):
    """The last image-2 row of a point's search window (``window``'s slice, clipped at the image)."""
    return min(int(r2fg + s // 2 + border + 1) - 1, rows2 - 1)


@functools.lru_cache(maxsize=None)
def band_pair():
    rng = np.random.default_rng(77)
    img1 = syn.speckle_image(BAND_SHAPE1, seed=41)
    img2 = syn.warp_pair(syn.speckle_image(BAND_SHAPE2, seed=41), syn.rotation_matrix(BAND_SHAPE2, 1.0), seed=41)
    poison1 = rng.integers(1, 256, BAND_SHAPE1).astype(np.uint8)
    poison2 = rng.integers(1, 256, BAND_SHAPE2).astype(np.uint8)
    return img1, img2, poison1, poison2


def band_boundaries(s=None, b_win=0):
    """Inner band boundaries of both plans; with ``s``, those far enough from row 0 for a template (at 45 degrees) and
    a window of border ``b_win`` to end there."""
    max_rows = max(BAND_SHAPE1[0], BAND_SHAPE2[0])
    ys = set()
    for plan in BAND_PLANS.values():
        ys |= set(band_lo(max_rows, band_weights(max_rows, plan=plan))[1:-1])
    if s is not None:
        ys = {y for y in ys if y - 2 - band_ext(s) - 0.75 * s - 2 >= 0 and y - 2 - 2 * (s // 2) - 2 * b_win - 2 >= 0}
    return sorted(ys)


def place_read_row(s, angles, alpha0, rot_order, x, m):
    """r1 of the point at column ``x`` whose largest template corner row over the angles is ``m`` (or the next double
    above it)."""
    def reach(v):
        return max(template_extent(x, v, s, a, alpha0)[0] for a in angles)
    v = m - reach(0.0)
    for _ in range(64):
        if reach(v) >= m:
            return v
        v = np.nextafter(v, np.inf)
    raise AssertionError("no placement for %r" % ((s, alpha0, m),))


def band_points(s, b_tpl, b_win, b_fill, limit, rot_order):
    """Points at every band boundary y of both plans, four kinds: "tpl_reach" / "win_reach" put the last row the
    template / the window reads at y - 1 and at y, the reading coordinate in 0.25 px steps (a bound that falls short
    of the true reach launches the row-y points one band early, before row y has arrived); "tpl_need" / "win_need" put
    run_host's need term itself at y - 0.5 ... y + 0.25 (points on both sides of the boundary in its own terms).  A
    filler grid of small borders puts >= 256 points in the pm_ws_kernel class where the size has one.
    Returns (pts, roles): roles maps each kind to (index, boundary) pairs."""
    hws, ext = s // 2, band_ext(s)
    c1, r1, c2, r2, brd = [], [], [], [], []
    roles = {"tpl_reach": [], "win_reach": [], "tpl_need": [], "win_need": []}

    def add(role, y, a, b, c, d, e):
        if role:
            roles[role].append((len(c1), y))
        c1.append(a), r1.append(b), c2.append(c), r2.append(d), brd.append(float(e))
    cols = min(BAND_SHAPE1[1], BAND_SHAPE2[1])
    xs = np.linspace(hws + 40 + 0.71 * s, cols - hws - 40 - 0.71 * s, 7)
    base = -1.0 if rot_order else -0.5                  # corner rows [R + base, R + base + 1) read row R
    for y in band_boundaries(s, b_win):
        for k, (row, dy) in enumerate([(row, dy) for row in (y - 1, y) for dy in BAND_STEPS]):
            x = xs[k % 7]
            r = place_read_row(s, BAND_ANGLES, BAND_ALPHA0, rot_order, x, row + base + dy)
            add("tpl_reach", y, x, r, round(x), round(r) - 2, b_tpl)     # the window ends rows above
            rw = row + dy - hws - b_win                 # the window's last row: floor(r2fg + hws + b)
            add("win_reach", y, xs[(k + 3) % 7], math.floor(rw), xs[(k + 3) % 7], rw, b_win)
        for k, dy in enumerate((-0.5, -0.25, 0.0, 0.25)):
            r = y + dy - ext
            add("tpl_need", y, xs[k % 7], r, round(xs[k % 7]), round(r), b_tpl)
            rw = y + dy - hws - b_win - 2
            add("win_need", y, xs[(k + 3) % 7], math.floor(rw), xs[(k + 3) % 7], rw, b_win)
    if limit is not None:
        need = 256 + 8 - sum(1 for b in brd if b <= limit)
        rows = np.linspace(hws + b_fill + 60, BAND_SHAPE2[0] - hws - b_fill - 60, max(0, -(-need // 7)))
        for y in rows:
            for x in xs:
                add(None, None, x, y, round(x), round(y), b_fill)
    pts = [np.asarray(v, dtype=np.float64) for v in (c1, r1, c2, r2, brd)]
    return pts, roles


@functools.lru_cache(maxsize=None)
def band_oracle(s, rot_order):
    img1, img2, _, _ = band_pair()
    case = next(c for c in BAND_SIZES if c[0] == s)
    pts, _ = band_points(*case, rot_order)
    return co.use_mcc_batch(*pts, img1, img2, s, BAND_ALPHA0, angles=BAND_ANGLES, rot_order=rot_order)


@pytest.mark.parametrize("rot_order", [0, 1])
@pytest.mark.parametrize("case", BAND_SIZES, ids=["s%d" % c[0] for c in BAND_SIZES])
def test_band_points_reach_every_boundary(case, rot_order):
    """Every point's restated band holds the last row it reads, in both images; the reach points read row y - 1 or
    row y of every boundary y of each plan through the term they claim; the need points sit on both sides of it;
    where a size has a pm_ws_kernel class some band gets two launches."""
    s, b_tpl, b_win, b_fill, limit = case
    pts, roles = band_points(*case, rot_order)
    c1, r1, c2, r2, b = pts
    max_rows = max(BAND_SHAPE1[0], BAND_SHAPE2[0])
    t_row = [template_read_row(c1[i], r1[i], s, BAND_ANGLES, BAND_ALPHA0, rot_order) for i in range(c1.size)]
    w_row = [window_read_row(r2[i], b[i], s, BAND_SHAPE2[0]) for i in range(c1.size)]
    for term, mine, other in (("tpl", t_row, w_row), ("win", w_row, t_row)):
        by_y = {}
        for i, y in roles[term + "_reach"]:
            assert other[i] < mine[i], (term, i)                   # this term sets the reach
            by_y.setdefault(y, []).append(mine[i])
        assert sorted(by_y) == band_boundaries(s, b_win)
        for y, read in by_y.items():
            assert sorted(read) == [y - 1] * 4 + [y] * 4, (term, y, read)
    for plan in BAND_PLANS.values():
        lo = band_lo(max_rows, band_weights(max_rows, plan=plan))
        pairs, bands = predicted_launches(lo, pts, s, limit)
        for i in range(c1.size):
            assert max(t_row[i], w_row[i]) < lo[bands[i] + 1], (i, t_row[i], w_row[i], bands[i])
        for term in ("tpl_need", "win_need"):
            for y in band_boundaries(s, b_win):
                if y in lo:
                    k = lo.index(y)
                    assert {bands[i] for i, yy in roles[term] if yy == y} == {k - 1, k}, (term, y)
        if limit is not None:
            assert any((k, True) in pairs and (k, False) in pairs for k in range(len(lo) - 1)), pairs
        else:
            assert all(not small for _, small in pairs)
    _, st = band_oracle(s, rot_order)
    n_edge = sum(len(v) for v in roles.values())
    assert (st == 1).sum() >= n_edge - 4, st


def sentinel_calls(lo, s, b_tpl, b_win):
    """For every inner boundary y of ``lo`` and each need term: pairs of points whose restated bands are (k-1, k-1)
    (need y - 0.25 and y - 40.25), (k, k) (y + 0.25, y + 40.25) and (k-1, k) (y - 0.25, y + 40.25) -- one, one and two
    launches -- so that run_host assigning the point at the boundary to another band changes the launch count."""
    hws, ext = s // 2, band_ext(s)
    x = 350.0
    calls = []
    for y in lo[1:-1]:
        if y not in band_boundaries(s, b_win) or y + 41 > min(BAND_SHAPE1[0], BAND_SHAPE2[0]) - s:
            continue
        for term in ("tpl", "win"):
            for n1, n2 in ((y - 0.25, y - 40.25), (y + 0.25, y + 40.25), (y - 0.25, y + 40.25)):
                pts = [[], [], [], [], []]
                for need in (n1, n2):
                    if term == "tpl":
                        r, rw, b = need - ext, round(need - ext), b_tpl
                    else:
                        rw, b = need - hws - b_win - 2, b_win
                        r = math.floor(rw)
                    for col, v in zip(pts, (x, r, x, rw, b)):
                        col.append(float(v))
                calls.append((y, term, [np.asarray(v) for v in pts]))
    return calls


def test_sentinel_calls_predict_one_or_two_launches():
    max_rows = max(BAND_SHAPE1[0], BAND_SHAPE2[0])
    s, b_tpl, b_win = 35, 2, 24
    for plan in BAND_PLANS.values():
        lo = band_lo(max_rows, band_weights(max_rows, plan=plan))
        calls = sentinel_calls(lo, s, b_tpl, b_win)
        assert len(calls) == 6 * (len(lo) - 2)
        for y, term, pts in calls:
            k = lo.index(y)
            pairs, bands = predicted_launches(lo, pts, s, None)
            assert bands in ([k - 1, k - 1], [k, k], [k - 1, k]), (y, term, bands)
            assert len(pairs) == len(set(bands))


# ==================================================================================================== GPU helpers
def adopt_poisoned(ctx, img1, img2, poison, extra):
    """Caller-owned buffers in sid_pair_layout form (pitch + ``extra``), filled with the poison first and then with
    the image in [:rows, :cols], adopted by ``ctx``.  Returns the buffers (torch tensors: keep them alive)."""
    import torch
    bufs = []
    for k, img in enumerate((img1, img2)):
        rows, cols = img.shape
        pitch, nbytes = layout_bytes(rows, cols, padded_pitch(cols) + extra)
        t = torch.from_numpy(poison_bytes(poison, nbytes, seed=17 + k)).cuda()
        assert t.data_ptr() % 256 == 0
        t[:pitch * rows].view(rows, pitch)[:, :cols] = torch.from_numpy(img).cuda()
        bufs.append((t, pitch, nbytes))
    torch.cuda.synchronize()
    (t1, p1, n1), (t2, p2, n2) = bufs
    ctx.adopt_pair_device(t1.data_ptr(), img1.shape, p1, n1, t2.data_ptr(), img2.shape, p2, n2)
    return bufs


@pytest.fixture(scope="module")
def layout_ctxs():
    """{"zero": a context with the layout pair uploaded into fresh (zeroed) buffers, (poison, extra pitch): a context
    that adopted the poisoned buffers}."""
    img1, img2 = layout_pair()
    out, keep = {}, []
    zero = _lib.Context(0)
    zero.set_pair(img1, img2)
    out["zero"] = zero
    for poison in POISONS:
        for extra in EXTRA_PITCH:
            ctx = _lib.Context(0)
            keep.append(adopt_poisoned(ctx, img1, img2, poison, extra))
            out[(poison, extra)] = ctx
    yield out
    for ctx in out.values():
        ctx.close()
    del keep


def run_logged(ctx, capfd, pts, s, angles, alpha0, rot_order, flags):
    capfd.readouterr()
    before = ctx.launch_count
    got, st = ctx.run(*pts, s, angles, alpha0, rot_order, flags, want_status=True)
    return got, st, ctx.launch_count - before, launch_lines(capfd.readouterr().err)


def check_row_launch(lines, launched, kernel, attrs):
    if "tail" not in attrs:                 # a row that does not pin the tail: take it from the launch lines
        tail = [d["threads"] for d in lines if d["kernel"] == "tail"]
        attrs = dict(attrs, tail=tail[0] if tail else None)
    check_launch(lines, launched, kernel, attrs)


# ==================================================================================================== A. adopted pairs
@pytest.mark.gpu
@pytest.mark.parametrize("row", A_ROWS, ids=[r[0] for r in A_ROWS])
def test_kernel_rows_on_poisoned_adopted_pairs(layout_ctxs, monkeypatch, capfd, row):
    rid, s, angles, (lo, hi), fs, env, kernel, attrs = row
    monkeypatch.setenv("SID_DEBUG", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    _, img2 = layout_pair()
    o = opts_of(fs)
    for alpha0 in ALPHAS:
        pts, roles = layout_points(s, lo, hi, angles, alpha0)
        ref, st_ref = layout_oracle(s, tuple(angles), lo, hi, fs, alpha0)
        zero, st0, launched, lines = run_logged(layout_ctxs["zero"], capfd, pts, s, angles, alpha0, o["rot_order"],
                                                flags_of(o))
        assert layout_ctxs["zero"].last_kernel_name == kernel, (rid, layout_ctxs["zero"].last_kernel_name, lines)
        check_row_launch(lines, launched, kernel, attrs)
        assert_equals_exact_oracle(zero, ref, st0, st_ref)
        check_roles(pts, roles, st0, s, img2)
        for key in [(p, e) for p in POISONS for e in EXTRA_PITCH]:
            ctx = layout_ctxs[key]
            got, st, launched, lines = run_logged(ctx, capfd, pts, s, angles, alpha0, o["rot_order"], flags_of(o))
            assert ctx.last_kernel_name == kernel, (rid, key, ctx.last_kernel_name)
            check_row_launch(lines, launched, kernel, attrs)
            assert got.tobytes() == zero.tobytes() and np.array_equal(st, st0), (rid, key, alpha0)


MAP_ROWS = [r for r in A_ROWS if r[0] in ("s35_ws3_b21", "s4_tc_smem_b26", "s128_imma_ldg_b39")]


@pytest.mark.gpu
@pytest.mark.parametrize("row", MAP_ROWS, ids=[r[0] for r in MAP_ROWS])
def test_maps_subpixel_and_device_run_on_poisoned_adopted_pairs(layout_ctxs, row):
    """run_maps (table, every map, every template), the sub-pixel flag and run_device on the poisoned pairs: bit for
    bit the zero-padded context's, whose tables equal the exact oracle."""
    import torch
    rid, s, angles, (lo, hi), fs, env, kernel, attrs = row
    o = opts_of(fs)
    flags = flags_of(o)
    zero_ctx = layout_ctxs["zero"]
    for alpha0 in (0.0, 45.0):
        pts, roles = layout_points(s, lo, hi, angles, alpha0)
        ref, st_ref = layout_oracle(s, tuple(angles), lo, hi, fs, alpha0)
        tab0, maps0, tpls0, st0 = zero_ctx.run_maps(*pts, s, angles, alpha0, o["rot_order"], flags, want_status=True)
        assert zero_ctx.last_kernel_name == kernel
        assert_equals_exact_oracle(tab0, ref, st0, st_ref)
        sub0, sst0 = zero_ctx.run(*pts, s, angles, alpha0, o["rot_order"], flags | _lib.SID_SUBPIXEL, want_status=True)
        assert np.array_equal(sst0, st_ref)
        assert np.array_equal(sub0[:, 2:], tab0[:, 2:], equal_nan=True)
        assert np.array_equal(np.isnan(sub0), np.isnan(tab0))
        ok = st0 == 1
        assert np.all(np.abs(sub0[ok, :2] - tab0[ok, :2]) <= 0.5)
        n = pts[0].size
        dev = torch.device("cuda", 0)
        d_pts = torch.from_numpy(np.stack(pts)).to(dev)
        for key in [(p, e) for p in POISONS for e in EXTRA_PITCH]:
            ctx = layout_ctxs[key]
            tab, maps, tpls, st = ctx.run_maps(*pts, s, angles, alpha0, o["rot_order"], flags, want_status=True)
            assert tab.tobytes() == tab0.tobytes() and np.array_equal(st, st0), (rid, key)
            assert tpls.tobytes() == tpls0.tobytes(), (rid, key)
            for i in range(n):
                assert (maps[i] is None) == (maps0[i] is None)
                if maps[i] is not None:
                    assert maps[i].tobytes() == maps0[i].tobytes(), (rid, key, i)
            sub, sst = ctx.run(*pts, s, angles, alpha0, o["rot_order"], flags | _lib.SID_SUBPIXEL, want_status=True)
            assert sub.tobytes() == sub0.tobytes() and np.array_equal(sst, sst0), (rid, key)
            d_out = torch.full((n, 5), -7.0, dtype=torch.float64, device=dev)
            d_st = torch.full((n,), 7, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            ctx.run_device(n, *[d_pts[i].data_ptr() for i in range(5)], hi, s, angles, alpha0, d_out.data_ptr(),
                           d_st.data_ptr(), o["rot_order"], flags)
            assert ctx.last_kernel_name == kernel
            ctx.synchronize()
            assert d_out.cpu().numpy().tobytes() == tab0.tobytes() and np.array_equal(d_st.cpu().numpy(), st0)


def ds_shapes(k):
    """Image 1: output width exactly one or two full CTA tiles; image 2: a partial last tile.  Rows: more than one
    CTA row group, not a multiple of the factor."""
    tile = (256 * 16 // k) // 16 * 16
    rows_cta = 1 if k >= 8 else 8 // k
    full = tile * (2 if k >= 8 else 1)
    return (k * (2 * rows_cta + 1) + (k - 1), k * full + 1), (k * (3 * rows_cta) + 1, k * (tile + 5) + k - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("content", ["random", "all255"])
def test_downsample_every_factor_on_poisoned_adopted_pairs(content):
    """sid_downsample_pair for every factor 2 ... 16 on adopted pairs with poisoned padding and tail slack, into
    poisoned output buffers: the image bytes equal the NumPy restatement, the output padding keeps its poison, and the
    zero-padded upload gives the same bytes.  All-255 content puts 16 * 255 in every 16-bit lane at k = 16."""
    import torch
    for k in range(2, 17):
        rng = np.random.default_rng(300 + k)
        imgs = []
        for shape in ds_shapes(k):
            if content == "all255":
                img = np.full(shape, 255, np.uint8)
            else:
                img = rng.integers(1, 256, shape).astype(np.uint8)
                img[rng.integers(0, shape[0], 30), rng.integers(0, shape[1], 30)] = 0
            imgs.append(img)
        img1, img2 = imgs
        outs = [(img.shape[0] // k, img.shape[1] // k) for img in imgs]
        assert outs[0][1] % ((256 * 16 // k) // 16 * 16) == 0 and outs[1][1] % ((256 * 16 // k) // 16 * 16) != 0
        results = {}
        for key in ["zero"] + [(p, e) for p in POISONS for e in EXTRA_PITCH]:
            ctx = _lib.Context(0)
            keep = ctx.set_pair(img1, img2) if key == "zero" else adopt_poisoned(ctx, img1, img2, *key)
            bufs = []
            for j, shape in enumerate(outs):
                pitch, nbytes = layout_bytes(*shape)
                fill = poison_bytes("rand", nbytes, seed=900 + j)
                bufs.append((torch.from_numpy(fill).cuda(), pitch, nbytes, fill))
            torch.cuda.synchronize()
            ctx.downsample_pair(k, *[(t.data_ptr(), p, n) for t, p, n, _ in bufs])
            ctx.synchronize()
            got = []
            for (t, pitch, nbytes, fill), shape, img in zip(bufs, outs, imgs):
                raw = t.cpu().numpy()
                view = raw[:pitch * shape[0]].reshape(shape[0], pitch)
                assert np.array_equal(view[:, :shape[1]], downsample_ref(img, k)), (k, key, shape)
                inside = np.zeros(nbytes, bool)
                inside[:pitch * shape[0]].reshape(shape[0], pitch)[:, :shape[1]] = True
                assert np.array_equal(raw[~inside], fill[~inside]), (k, key)          # nothing written outside
                got.append(view[:, :shape[1]].tobytes())
            results[key] = got
            ctx.close()
            del keep
        assert all(v == results["zero"] for v in results.values()), k


# ==================================================================================================== B. owned reuse
B_ROWS = [r for r in A_ROWS if r[0] in ("s35_ws3_b21", "s35_tc_split_b37", "s112_imma_b16", "s128_imma_ldg_b39",
                                        "s35_dp4a_b21")]


@functools.lru_cache(maxsize=None)
def large_noise_pair():
    rng = np.random.default_rng(5)
    return (rng.integers(1, 256, (1400, 1230)).astype(np.uint8), rng.integers(1, 256, (1380, 1250)).astype(np.uint8))


@pytest.mark.gpu
def test_owned_context_reused_with_shrinking_pairs(monkeypatch):
    """A large zero-free noise pair first, then the smaller layout pair (fewer rows, narrower pitch: the old pixels lie
    in the new padding, the tail slack and past the new last row) through set_pair, set_pair_device and run_pair from
    pinned and from pageable memory: every table equals the exact oracle and a fresh context's."""
    import torch
    big1, big2 = large_noise_pair()
    img1, img2 = layout_pair()
    assert padded_pitch(big1.shape[1]) > padded_pitch(img1.shape[1]) and big1.shape[0] > img1.shape[0]
    assert padded_pitch(big2.shape[1]) > padded_pitch(img2.shape[1]) and big2.shape[0] > img2.shape[0]
    d1, d2 = torch.from_numpy(img1).cuda(), torch.from_numpy(img2).cuda()
    p1, p2 = torch.from_numpy(img1).pin_memory().numpy(), torch.from_numpy(img2).pin_memory().numpy()
    fresh = _lib.Context(0)
    fresh.set_pair(img1, img2)
    ctx = _lib.Context(0)

    def uploads():
        yield "set_pair", lambda pts, *a: ctx.set_pair(img1, img2).run(*pts, *a, want_status=True)
        yield "set_pair_device", lambda pts, *a: ctx.set_pair_device(
            d1.data_ptr(), img1.shape, img1.shape[1], d2.data_ptr(), img2.shape, img2.shape[1]).run(
            *pts, *a, want_status=True)
        yield "run_pair_pageable", lambda pts, *a: ctx.run_pair(img1, img2, *pts, *a, want_status=True)
        yield "run_pair_pinned", lambda pts, *a: ctx.run_pair(p1, p2, *pts, *a, want_status=True)
    torch.cuda.synchronize()
    for rid, s, angles, (lo, hi), fs, env, kernel, attrs in B_ROWS:
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            o = opts_of(fs)
            for alpha0 in (0.0, 45.0):
                pts, roles = layout_points(s, lo, hi, angles, alpha0)
                ref, st_ref = layout_oracle(s, tuple(angles), lo, hi, fs, alpha0)
                want, st_want = fresh.run(*pts, s, angles, alpha0, o["rot_order"], flags_of(o), want_status=True)
                assert fresh.last_kernel_name == kernel
                assert_equals_exact_oracle(want, ref, st_want, st_ref)
                check_roles(pts, roles, st_want, s, img2)
                for name, call in uploads():
                    ctx.set_pair(big1, big2)
                    ctx.run(*pts[:4], np.full(pts[0].size, 3.0), s, angles, alpha0)
                    got, st = call(pts, s, angles, alpha0, o["rot_order"], flags_of(o))
                    assert ctx.last_kernel_name == kernel, (rid, name, ctx.last_kernel_name)
                    assert got.tobytes() == want.tobytes() and np.array_equal(st, st_want), (rid, name, alpha0)
    fresh.close()
    ctx.close()


@pytest.mark.gpu
def test_single_call_functions_after_a_larger_resident_pair():
    """get_template, match_template and rotate_and_match upload into the context's image buffers: after a larger
    zero-free pair the stale bytes around the new image must not reach their results (templates crossing the image
    edge: zeros where the reference samples outside)."""
    big1, big2 = large_noise_pair()
    img1, img2 = layout_pair()
    ctx = _lib.Context(0)
    s, angles = 35, [-3, 0, 3]
    for alpha0 in (0.0, 45.0):
        for rot_order in (0, 1):
            pts, roles = layout_points(s, 19, 21, angles, alpha0)
            for i in list(roles["nan_edge"]) + list(roles["last_line"]):
                for a in angles:
                    ctx.set_pair(big1, big2)
                    got = ctx.get_template(img1, pts[0][i], pts[1][i], a - alpha0, s, rot_order)
                    want = co.get_template(img1, pts[0][i], pts[1][i], a - alpha0, s, rot_order)
                    assert np.array_equal(got, want), (i, a, alpha0, rot_order)
            nan_seen = 0
            for i in list(roles["nan_edge"][:4]) + list(roles["last_line"]):
                win = img2[int(pts[3][i] - 17 - 19):int(pts[3][i] + 17 + 19 + 1),
                           int(pts[2][i] - 17 - 19):int(pts[2][i] + 17 + 19 + 1)]
                ctx.set_pair(big1, big2)
                got = ctx.rotate_and_match(img1, pts[0][i], pts[1][i], s, win, angles, alpha0, rot_order)
                want = co.rotate_and_match(img1, pts[0][i], pts[1][i], s, win, alpha0, angles=angles,
                                           rot_order=rot_order)
                if got is None:
                    nan_seen += 1
                    assert not isinstance(want[5], np.ndarray), (i, want[:5])
                    continue
                assert (got[0], got[1], angles[got[2]], got[3]) == (want[0], want[1], want[2], want[3])
                assert abs(got[4] - want[4]) <= 4e-6 * (1 + abs(want[4]))
                assert got[5].tobytes() == np.asarray(want[5], np.float32).tobytes()
                assert np.array_equal(got[6], want[6])
            assert nan_seen == 4
    # match_template on a window at image 2's far corner with a template from image 1's last rows / columns
    for h, w in ((50, 61), (41, 37)):
        win = np.ascontiguousarray(img2[-h:, -w:])
        tpl = np.ascontiguousarray(img1[-35:, -33:])
        ctx.set_pair(big1, big2)
        got = ctx.match_template(win, tpl)
        assert got.tobytes() == np.asarray(co.match_template(win, tpl), np.float32).tobytes()
    ctx.close()


@pytest.mark.gpu
def test_series_driver_with_shrinking_pairs():
    """sharding.use_mcc_series with pairs in shrinking order (the series test of tests/test_gpu_parity.py run the
    other way round): every pair lands in buffers that held a larger one."""
    from sea_ice_drift_b200.sharding import use_mcc_series
    items = []
    for k in range(5):
        img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=30 + k, side=792 - 48 * k, grid=22 - 3 * k)
        items.append((img1, img2, c1, r1, c2, r2, b))
    for n_contexts in (1, 2):
        tables = use_mcc_series(items, 35, 0.0, n_contexts=n_contexts, angles=[-3, 0, 3])
        assert len(tables) == 5
        for (img1, img2, c1, r1, c2, r2, b), got in zip(items, tables):
            ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=[-3, 0, 3])
            assert_equals_exact_oracle(got, ref)


# ==================================================================================================== C. band edges
@pytest.mark.gpu
@pytest.mark.parametrize("rot_order", [0, 1])
@pytest.mark.parametrize("case", BAND_SIZES, ids=["s%d" % c[0] for c in BAND_SIZES])
def test_upload_band_edges(monkeypatch, capfd, case, rot_order):
    """run_pair from pageable memory with one host copy thread on a context whose buffers hold a same-shaped poison
    pair (no fresh zero fill): band k + 1 is copied on the host only after band k's launches are enqueued, so a point
    launched with a band before the last row it reads has arrived would read poison.  Two plans (12 short bands, the
    default); the table equals the exact oracle.  The launch count equals the restated plan's non-empty (band, class)
    pairs -- a coarse tie of the restatement to the C code (most single misassignments keep every pair non-empty);
    the sharp one is test_band_assignment_matches_the_restatement."""
    s, b_tpl, b_win, b_fill, limit = case
    img1, img2, poison1, poison2 = band_pair()
    pts, roles = band_points(*case, rot_order)
    ref, st_ref = band_oracle(s, rot_order)
    max_rows = max(img1.shape[0], img2.shape[0])
    monkeypatch.setenv("SID_DEBUG", "1")
    monkeypatch.setenv("SID_UPLOAD_THREADS", "1")
    ctx = _lib.Context(0)
    two_launch_bands = 0
    for name, plan in BAND_PLANS.items():
        with monkeypatch.context() as mp:
            if plan is not None:
                mp.setenv("SID_BAND_PLAN", plan)
            ctx.set_pair(poison1, poison2)
            ctx.synchronize()
            capfd.readouterr()
            before = ctx.launch_count
            got, st = ctx.run_pair(img1, img2, *pts, s, BAND_ANGLES, BAND_ALPHA0, rot_order, want_status=True)
            launched = ctx.launch_count - before
            lines = launch_lines(capfd.readouterr().err)
        assert_equals_exact_oracle(got, ref, st, st_ref)
        lo = band_lo(max_rows, band_weights(max_rows, plan=plan))
        assert len(lo) - 1 == (12 if plan else 3)
        pairs, bands = predicted_launches(lo, pts, s, limit)
        main = [d for d in lines if d["kernel"] != "tail"]
        assert len(main) == len(pairs), (name, len(main), sorted(pairs))
        assert launched == len(lines), (name, launched, lines)
        n_ws = sum(1 for d in main if d["kernel"] == "ws")
        assert n_ws == sum(1 for _, small in pairs if small) or limit is None, (name, n_ws, sorted(pairs))
        two_launch_bands += sum(1 for k in range(len(lo) - 1) if (k, True) in pairs and (k, False) in pairs)
        reach_y = {y for i, y in roles["tpl_reach"]}
        assert {y for y in lo[1:-1] if y in band_boundaries(s, b_win)} <= reach_y
    assert (two_launch_bands > 0) == (limit is not None)
    ctx.close()


@pytest.mark.gpu
def test_band_assignment_matches_the_restatement(monkeypatch, capfd):
    """Two points per run_pair call at every boundary of both plans, for each need term: the call launches one kernel
    per band the restatement puts a point in, so run_host giving the point at the boundary another band than the
    restated one changes the count (one launch where two are predicted, or two where one is)."""
    img1, img2, _, _ = band_pair()
    s, b_tpl, b_win = 35, 2, 24
    max_rows = max(img1.shape[0], img2.shape[0])
    monkeypatch.setenv("SID_DEBUG", "1")
    ctx = _lib.Context(0)
    n_calls = 0
    for name, plan in BAND_PLANS.items():
        lo = band_lo(max_rows, band_weights(max_rows, plan=plan))
        with monkeypatch.context() as mp:
            if plan is not None:
                mp.setenv("SID_BAND_PLAN", plan)
            for y, term, pts in sentinel_calls(lo, s, b_tpl, b_win):
                pairs, bands = predicted_launches(lo, pts, s, None)
                capfd.readouterr()
                ctx.run_pair(img1, img2, *pts, s, BAND_ANGLES, BAND_ALPHA0)
                main = [d for d in launch_lines(capfd.readouterr().err) if d["kernel"] != "tail"]
                assert len(main) == len(pairs), (name, y, term, bands, len(main))
                n_calls += 1
    assert n_calls == 6 * (12 - 1) + 6 * (3 - 1)
    ctx.close()
