"""Parity on degenerate image content: flat patches, exact ties and low contrast.

Speckle (the content of every other parity test) gives correlation maps without repeated values, so it never reaches
the branches that handle them: a flat template (the whole map is 1, the peak is index 0, h is 0/0 under hes_norm),
several positions or several angles at the same maximum (the lowest row-major index and the first angle win), a median
whose 20-bit histogram bin holds more than 64 Hessian values (the wide select of hes_norm_fast), and valid rows with NaN
r or h.  The content below is built to reach them, and ``test_content_reaches_the_degenerate_branches`` checks that it
still does.

The CPU tests pin the exact oracle against an independent float64 NCC, the NumPy Hessian and the cv2 port of the
reference; the GPU tests (``-m gpu``) pin every correlation kernel against the exact oracle, bit for bit."""
import functools

import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

from sea_ice_drift_b200 import synthetic as syn
from oracle import c_oracle as co
from tests.helpers import classify, make_exact_lookup, assert_parity, assert_equals_exact_oracle

SIDE = 400
FLT_EPSILON = float(np.finfo(np.float32).eps)
FLAG_SETS = {"default": dict(), "raw_hes": dict(hes_norm=False), "hes_smth": dict(hes_smth=True),
             "mcc_norm": dict(mcc_norm=True)}
CLASSES = ("plateaus", "periodic", "lowcontrast")


def opts_of(flag_set):
    o = dict(rot_order=0, hes_norm=True, hes_smth=False, mcc_norm=False)
    o.update(FLAG_SETS[flag_set])
    return o


# ---------------------------------------------------------------------------------------------------- content
# img1 plateau (flat templates), img2 plateau (flat search windows)
P1 = (100, 230)
P2 = (200, 380)


@functools.lru_cache(maxsize=None)
def images(kind):
    """Seeded image pairs, SIDE x SIDE uint8."""
    if kind == "plateaus":
        base = syn.speckle_image((SIDE, SIDE), seed=0)
        img1 = base.copy()
        img2 = syn.warp_pair(base, syn.shift_matrix(2.0, -1.0), seed=0).copy()
        img1[P1[0]:P1[1], P1[0]:P1[1]] = 128
        img2[P2[0]:P2[1], P2[0]:P2[1]] = 200
        img1[300:340, 40:100] = 255                    # saturated patch in img1, near-black one in img2
        img2[40:90, 260:330] = 1
        return img1, img2
    if kind == "periodic":
        tile = np.random.default_rng(1).integers(1, 256, (7, 9), dtype=np.uint8)
        img1 = np.ascontiguousarray(np.tile(tile, (SIDE // 7 + 1, SIDE // 9 + 1))[:SIDE, :SIDE])
        return img1, np.ascontiguousarray(np.roll(img1, (1, 2), axis=(0, 1)))
    if kind == "lowcontrast":
        rng = np.random.default_rng(2)
        img1 = np.full((SIDE, SIDE), 100, np.uint8)
        ii = rng.integers(0, SIDE, (SIDE * SIDE // 200, 2))
        img1[ii[:, 0], ii[:, 1]] = 101
        img2 = np.full((SIDE, SIDE), 100, np.uint8)
        jj = rng.integers(0, SIDE, (SIDE * SIDE // 300, 2))
        img2[jj[:, 0], jj[:, 1]] = 101
        return img1, img2
    raise KeyError(kind)


def _rows(kind, s):
    """The points of a class for img_size ``s``, placed on purpose: (tag, border -> (c1, r1, c2fg, r2fg))."""
    centre, hws = int(s / 2.) + 1, int(s / 2.)
    rows = []
    if kind == "plateaus":
        mid = (P1[0] + P1[1]) // 2
        # templates wholly inside the img1 plateau: flat at every angle
        for c in (mid - 23, mid, mid + 23):
            for r in (mid - 23, mid + 23):
                rows.append(("flat", lambda b, c=c, r=r: (c, r, c + 2, r - 1)))
        # templates straddling the plateau's top / left edge: one row of texture at every angle (k = -1), flat at
        # angle 0 only (k = 0), flat at every angle (k = 1, 2)
        for k in (-1, 0, 1, 2):
            tag = "nearly_flat" if k < 0 else "edge"
            rows.append((tag, lambda b, k=k: (mid, P1[0] + centre + k, mid + 2, P1[0] + centre + k - 1)))
            rows.append((tag, lambda b, k=k: (P1[0] + centre + k, mid + 7, P1[0] + centre + k + 2, mid + 6)))
        # search windows more than half inside the img2 plateau (NCC 0 over most of the map), and one wholly inside
        for frac in (0.25, 0.5, 0.75):
            rows.append(("window_mostly_flat", lambda b, f=frac: (288, 260, 290, P2[0] + hws + int(f * b))))
            rows.append(("window_mostly_flat", lambda b, f=frac: (258, 290, P2[0] + hws + int(f * b), 291)))
        rows.append(("window_flat", lambda b: (288, 290, 290, 290)))
        # the saturated / near-black patches, and plain speckle
        rows.append(("saturated", lambda b: (70, 300, 72, 299)))
        rows.append(("saturated", lambda b: (300, 65, 302, 64)))
        rows.append(("speckle", lambda b: (60, 60, 62, 59)))
        rows.append(("speckle", lambda b: (330, 150, 332, 149)))
    elif kind == "periodic":
        # every window holds exact copies of the template at several positions (r == 1 ties)
        for c in (80, 143, 210, 297):
            for r in (90, 171, 250, 320):
                rows.append(("periodic", lambda b, c=c, r=r: (c, r, c + 2, r + 1)))
    elif kind == "lowcontrast":
        for c in (80, 170, 260, 330):
            for r in (85, 200, 310):
                rows.append(("lowcontrast", lambda b, c=c, r=r: (c, r, c + 1, r - 2)))
        for c, r in MEDIAN_RANK_POINTS:
            rows.append(("median_rank", lambda b, c=c, r=r: (c, r, c, r)))
    else:
        raise KeyError(kind)
    return rows


def points(kind, s, border):
    """The points of a class for img_size ``s`` and the per-point ``border`` array (its length is the point count;
    the point list is cycled).  Returns c1, r1, c2fg, r2fg, border."""
    rows = _rows(kind, s)
    border = np.asarray(border, dtype=np.float64)
    tab = np.array([rows[i % len(rows)][1](int(np.ceil(border[i]))) for i in range(border.size)], dtype=np.float64)
    return [tab[:, 0], tab[:, 1], tab[:, 2], tab[:, 3], border]


def tags(kind):
    return np.array([t for t, _ in _rows(kind, 35)])


def n_points(kind):
    return len(_rows(kind, 35))


# plateau rows where cv2's float32 correlation, not the oracle, limits the agreement in h: templates with one row of
# texture and search windows mostly on the img2 plateau; see test_exact_oracle_equals_cv2_port
CV2_LIMITED = ("nearly_flat", "window_mostly_flat")


# low-contrast points whose Hessian median (s 35, border 20, hes_norm) sits in a 20-bit bin of more than 64 values AND
# differs from its lower neighbour in rank by more than the h tolerance: only there does the rank the wide select
# takes show in h.  Found by scanning a 3-px grid of the low-contrast pair with the oracle (25 of 8 836 points).
MEDIAN_RANK_POINTS = ((87, 303), (99, 117), (114, 201), (174, 93), (228, 180), (252, 231), (297, 138), (315, 261))



def window_of(pts, i, img2, s):
    c1, r1, c2, r2, brd = pts
    hws = int(s / 2.)
    y0, y1 = int(r2[i] - hws - brd[i]), int(r2[i] + hws + brd[i] + 1)
    x0, x1 = int(c2[i] - hws - brd[i]), int(c2[i] + hws + brd[i] + 1)
    return img2[y0:y1, x0:x1]


# ---------------------------------------------------------------------------------------------------- float64 NCC
def ncc_float64(win, tpl):
    """TM_CCOEFF_NORMED with OpenCV's rules, directly in float64 over NumPy windows (no integral images)."""
    w = np.asarray(win, dtype=np.float64)
    t = np.asarray(tpl, dtype=np.float64)
    n = t.size
    t0 = t - t.mean()
    tnorm2 = (t0 * t0).sum()
    views = sliding_window_view(w, t.shape)
    out_shape = views.shape[:2]
    if tnorm2 / n < np.finfo(np.float64).eps:
        return np.ones(out_shape)
    num = np.einsum("yxij,ij->yx", views, t0)
    wsum = views.sum(axis=(2, 3))
    wsq = (views * views).sum(axis=(2, 3))
    diff2 = np.maximum(wsq - wsum * wsum / n, 0.0)
    thr = np.minimum(0.5, 10.0 * FLT_EPSILON * wsq)
    den = np.where(diff2 <= thr, 0.0, np.sqrt(diff2) * np.sqrt(tnorm2))
    an = np.abs(num)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(an < den, num / den, np.where(an < 1.125 * den, np.sign(num), 0.0))


def template_cases():
    """(name, window, template) pairs of every class: flat template, flat window, straddling edges, periodic copies,
    low contrast."""
    out = []
    pl1, pl2 = images("plateaus")
    out.append(("flat_template", pl2[60:135, 60:135], pl1[140:175, 150:185]))
    out.append(("flat_window", pl2[250:325, 250:325], pl1[20:55, 30:65]))
    out.append(("window_half_flat", pl2[170:245, 250:325], pl1[20:55, 30:65]))
    out.append(("template_straddles_edge", pl2[80:155, 140:215], pl1[98:133, 150:185]))
    out.append(("template_saturated", pl2[20:100, 250:340], pl1[290:325, 50:85]))
    pe1, pe2 = images("periodic")
    out.append(("periodic", pe2[100:175, 100:175], pe1[120:155, 118:153]))
    out.append(("periodic_even", pe2[50:120, 70:150], pe1[60:110, 80:130]))
    lc1, lc2 = images("lowcontrast")
    out.append(("lowcontrast", lc2[100:175, 100:175], lc1[120:155, 118:153]))
    out.append(("lowcontrast_self", lc1[100:175, 100:175], lc1[120:155, 118:153]))
    out.append(("lowcontrast_s21", lc2[200:261, 40:101], lc1[210:231, 50:71]))
    return out


# ---------------------------------------------------------------------------------------------------- map statistics
def degenerate_branches(kind, s, angles, border, flag_set="default"):
    """Counts, over the valid points of a class, of the degenerate branches the oracle's maps hit."""
    img1, img2 = images(kind)
    pts = points(kind, s, np.full(n_points(kind), float(border)))
    o = opts_of(flag_set)
    c = dict(flat_template=0, flat_at_some_angles=0, position_ties=0, angle_ties=0, median_bin_gt64=0,
             median_rank_matters=0, nan_h=0)
    for i in range(len(pts[0])):
        win = window_of(pts, i, img2, s)
        per_angle = [co.rotate_and_match(img1, pts[0][i], pts[1][i], s, win, 0.0, angles=[a], **o) for a in angles]
        if not isinstance(per_angle[0][5], np.ndarray):
            continue
        peaks = [float(p[5].max()) for p in per_angle]
        win_k = int(np.argmax(peaks))
        m = per_angle[win_k][5]
        res = co.rotate_and_match(img1, pts[0][i], pts[1][i], s, win, 0.0, angles=angles, **o)
        c["flat_template"] += int(bool(np.all(m == 1.0)))
        flat = [bool(np.all(p[5] == 1.0)) for p in per_angle]
        c["flat_at_some_angles"] += int(any(flat) and not all(flat))     # the screening must keep the flat angle
        c["position_ties"] += int((m == m.max()).sum() >= 2)
        c["angle_ties"] += int(peaks.count(max(peaks)) >= 2)
        c["nan_h"] += int(np.isnan(res[4]))
        hes = np.sort(co.get_hessian(m, hes_norm=False).ravel())
        n = hes.size
        key = hes.view(np.uint32) >> 11
        if (key == key[n // 2]).sum() > 64:
            c["median_bin_gt64"] += 1
            with np.errstate(invalid="ignore", divide="ignore"):
                gap = (hes[n // 2] - hes[n // 2 - 1]) / np.std(hes)
            c["median_rank_matters"] += int(gap > 3 * 4e-6 * (1 + abs(res[4])))
    return c


# ==================================================================================================== CPU tests
@pytest.mark.parametrize("name,win,tpl", template_cases(), ids=[c[0] for c in template_cases()])
def test_match_template_equals_float64_ncc(name, win, tpl):
    got = co.match_template(np.ascontiguousarray(win), np.ascontiguousarray(tpl)).astype(np.float64)
    ref = ncc_float64(win, tpl)
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 1e-6, (name, np.abs(got - ref).max())
    special = np.isin(ref, (1.0, -1.0, 0.0))
    assert np.array_equal(got[special], ref[special]), name


def hessian_maps():
    rng = np.random.default_rng(5)
    maps = {"constant_one": np.ones((41, 41), np.float32), "constant_zero": np.zeros((41, 41), np.float32),
            "constant_third": np.full((33, 47), 1.0 / 3.0, np.float32)}
    half_zero = np.zeros((41, 41), np.float32)
    half_zero[:15, :] = rng.uniform(-1, 1, (15, 41))
    maps["mostly_zero"] = half_zero
    zero_with_peak = np.zeros((51, 51), np.float32)
    zero_with_peak[20:25, 30:35] = np.float32(0.75)
    maps["zero_with_plateau"] = zero_with_peak
    maps["quantised"] = (rng.integers(-2, 5, (41, 41)) * 0.25).astype(np.float32)
    maps["quantised_even"] = (rng.integers(0, 3, (40, 36)) * 0.5).astype(np.float32)
    return maps


@pytest.mark.parametrize("name", sorted(hessian_maps()))
@pytest.mark.parametrize("hes_norm,hes_smth", [(True, False), (False, False), (True, True), (False, True)])
def test_hessian_on_degenerate_maps_equals_numpy(name, hes_norm, hes_smth):
    from oracle import pm_oracle as po
    ccm = hessian_maps()[name]
    got = co.get_hessian(ccm, hes_norm=hes_norm, hes_smth=hes_smth)
    ref = po.peak_sharpness(ccm, hes_norm=hes_norm, hes_smth=hes_smth)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), name
    fin = np.isfinite(ref)
    assert np.array_equal(got[~fin], ref[~fin], equal_nan=True), name
    if fin.any():
        assert np.abs(got[fin] - ref[fin]).max() <= 2e-6 * (1 + np.abs(ref[fin]).max()), name


@pytest.mark.parametrize("flag_set", sorted(FLAG_SETS))
@pytest.mark.parametrize("kind", ["plateaus", "periodic"])
def test_exact_oracle_equals_cv2_port(kind, flag_set):
    """Low contrast is left out on purpose: there cv2's float32 correlation is wrong (tests/helpers.py).  On the plateau
    points in CV2_LIMITED cv2 is off by 4e-6 ... 1.1e-5 from a float64 NCC (the exact side: < 3e-8), and the h
    normalisation, with a small Hessian spread on maps that are mostly flat, turns that into |dh| up to 5e-4 at
    |h| ~ 2 ... 4.
    Those rows are held to everything but the h budget here; their h is pinned against float64 by
    test_exact_rows_equal_float64_pipeline."""
    from oracle import pm_oracle as po
    img1, img2 = images(kind)
    o = opts_of(flag_set)
    for s, angles, border in ((35, [-3, 0, 3], 20), (21, [2, 2, 2], 12)):
        pts = points(kind, s, np.full(n_points(kind), float(border)))
        got, _ = co.use_mcc_batch(*pts, img1, img2, s, 0.0, angles=angles, **o)
        ref = po.run_points(*pts, img1, img2, s, 0.0, angles=angles, **o)
        lookup = make_exact_lookup(co, pts, img1, img2, s, 0.0, angles, o)
        lim = np.isin(tags(kind), CV2_LIMITED)
        for sel, full in ((~lim, True), (lim, False)):
            if not sel.any():
                continue
            idx = np.nonzero(sel)[0]
            stats = classify(got[sel], ref[sel], lambda i, *a: lookup(idx[i], *a))
            assert stats["exact"] + stats["ties"] == int((~np.isnan(ref[sel, 0])).sum()), stats
            if full:
                assert_parity(stats)
            else:
                assert stats["nan_equal"] and not stats["unexplained"] and stats["max_dr"] <= 1e-4, stats


@pytest.mark.parametrize("flag_set", sorted(FLAG_SETS))
@pytest.mark.parametrize("kind", ["plateaus", "lowcontrast"])
def test_exact_rows_equal_float64_pipeline(kind, flag_set):
    """Where cv2 cannot serve as the reference (low contrast, CV2_LIMITED), each oracle row is checked against float64:
    its winning map against the float64 NCC of its template, its peak against that map's maximum over all angles (under
    mcc_norm r against the normalisation of the float64 map), and its h against NumPy's Hessian of the float64 map at
    the oracle's peak."""
    from oracle import pm_oracle as po
    img1, img2 = images(kind)
    o = opts_of(flag_set)
    angles = [-3, 0, 3]
    pts = points(kind, 35, np.full(n_points(kind), 20.0))
    rows = np.nonzero(np.isin(tags(kind), CV2_LIMITED))[0] if kind == "plateaus" else range(n_points(kind))
    table, _ = co.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=angles, **o)
    for i in rows:
        win = window_of(pts, i, img2, 35)
        dc, dr, a, r, h, m, tpl = co.rotate_and_match(img1, pts[0][i], pts[1][i], 35, win, 0.0, angles=angles, **o)
        assert (pts[2][i] + dc, pts[3][i] + dr, a, r) == tuple(table[i, :4])
        f64 = ncc_float64(win, tpl)
        assert np.abs(m - f64).max() <= 1e-6, i
        best = max(float(ncc_float64(win, co.get_template(img1, pts[0][i], pts[1][i], x, 35)).max()) for x in angles)
        peak = (int(round(dr + (win.shape[0] - 35) / 2.)), int(round(dc + (win.shape[1] - 35) / 2.)))
        assert abs(f64[peak] - best) <= 1e-6, i
        if o["mcc_norm"]:
            f32 = f64.astype(np.float32)
            r64 = (np.float32(best) - np.median(f32)) / np.std(f32)
            assert np.isnan(r) == np.isnan(r64) and (np.isnan(r) or abs(r - r64) <= 1e-5 * (1 + abs(r64))), (i, r, r64)
        else:
            assert abs(r - best) <= 1e-6, i
        h64 = po.peak_sharpness(f64.astype(np.float32), **o)[peak]
        assert np.isnan(h) == np.isnan(h64) and (np.isnan(h) or abs(h - h64) <= 1e-5 * (1 + abs(h64))), (i, h, h64)


def test_content_reaches_the_degenerate_branches():
    """The content must keep hitting the branches it is here for; speckle hits none of them."""
    pl = degenerate_branches("plateaus", 35, [-3, 0, 3], 20)
    assert pl["flat_template"] >= 6 and pl["nan_h"] >= 6 and pl["angle_ties"] >= 6, pl
    assert pl["position_ties"] >= 6 and pl["median_bin_gt64"] >= 4 and pl["flat_at_some_angles"] >= 2, pl
    pe = degenerate_branches("periodic", 35, [-3, 0, 3], 20)
    assert pe["position_ties"] == n_points("periodic"), pe
    lc = degenerate_branches("lowcontrast", 35, [-3, 0, 3], 20)
    assert lc["median_bin_gt64"] >= 4 and lc["median_rank_matters"] >= len(MEDIAN_RANK_POINTS), lc
    rep = degenerate_branches("periodic", 35, [2, 2, 2], 20)
    assert rep["angle_ties"] == n_points("periodic"), rep
    seven = degenerate_branches("plateaus", 35, [-9, -6, -3, 0, 3, 6, 9], 20)
    assert seven["flat_template"] >= 6 and seven["angle_ties"] >= 6 and seven["flat_at_some_angles"] >= 2, seven
    sp1 = syn.speckle_image((300, 300), seed=3)
    sp2 = syn.warp_pair(sp1, syn.shift_matrix(2.0, -1.0), seed=3)
    for c, r in ((100, 100), (150, 200), (200, 120)):
        m = co.rotate_and_match(sp1, c, r, 35, sp2[r - 38:r + 37, c - 36:c + 39], 0.0)[5]
        assert (m == m.max()).sum() == 1 and m.max() < 1.0


# ==================================================================================================== GPU tests
def _flags(o):
    from sea_ice_drift_b200 import _lib
    return _lib.flags_from_kwargs(o["hes_norm"], o["hes_smth"], o["mcc_norm"])


def _run_vs_oracle(gpu_ctx, kind, s, angles, brd, flag_set, kernel, path=None, monkeypatch=None):
    img1, img2 = images(kind)
    pts = points(kind, s, brd)
    o = opts_of(flag_set)
    if path is not None:
        monkeypatch.setenv("SID_PM_PATH", path)
    gpu_ctx.set_pair(img1, img2)
    got, st = gpu_ctx.run(*pts, s, angles, 0.0, o["rot_order"], _flags(o), want_status=True)
    assert gpu_ctx.last_kernel_name == kernel, gpu_ctx.last_kernel_name
    ref, st_ref = co.use_mcc_batch(*pts, img1, img2, s, 0.0, angles=angles, **o)
    assert_equals_exact_oracle(got, ref, st, st_ref)
    assert np.isfinite(ref[:, 0]).sum() >= len(brd) // 2
    return got


# (family, img_size, angles, border range, SID_PM_PATH, kernel name)
FAMILIES = [
    ("ws", 35, [-3, 0, 3], (16, 20), None, "sid::pm_ws_kernel"),
    ("ws_repeated_angle", 35, [2, 2, 2], (20, 20), None, "sid::pm_ws_kernel"),
    ("ws_7angles", 35, [-9, -6, -3, 0, 3, 6, 9], (18, 20), None, "sid::pm_ws_kernel"),
    ("tc", 35, [-3, 0, 3], (30, 40), None, "sid::pm_tc_kernel"),
    ("imma_s35", 35, [-3, 0, 3], (20, 30), "imma", "sid::pm_points_kernel<imma>"),
    ("imma_s50", 50, [-3, 0, 3], (15, 25), "imma", "sid::pm_points_kernel<imma>"),
    ("imma_s21", 21, [-3, 0, 3], (10, 16), "imma", "sid::pm_points_kernel<imma>"),
    ("dp4a_s35", 35, [-3, 0, 3], (20, 30), "dp4a", "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s50", 50, [-3, 0, 3], (15, 25), "dp4a", "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s21", 21, [-3, 0, 3], (10, 16), "dp4a", "sid::pm_points_kernel<dp4a>"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", sorted(FLAG_SETS))
@pytest.mark.parametrize("kind", CLASSES)
@pytest.mark.parametrize("family", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_kernels_equal_exact_oracle(gpu_ctx, monkeypatch, family, kind, flag_set):
    name, s, angles, (lo, hi), path, kernel = family
    n = n_points(kind)
    brd = lo + np.arange(n) % (hi - lo + 1)
    _run_vs_oracle(gpu_ctx, kind, s, angles, brd.astype(np.float64), flag_set, kernel, path, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", sorted(FLAG_SETS))
@pytest.mark.parametrize("kind", CLASSES)
def test_mixed_border_classes_equal_exact_oracle(gpu_ctx, kind, flag_set):
    """Borders 20 and 30 ... 45 in one call: two launches (row-loop kernel + pm_ws_kernel), one table."""
    n = 24 * n_points(kind)
    k = np.arange(n)
    brd = np.where(k % 3 == 2, 30 + k % 16, 20).astype(np.float64)
    assert (brd == 20).sum() >= 256
    _run_vs_oracle(gpu_ctx, kind, 35, [-3, 0, 3], brd, flag_set, "sid::pm_tc_kernel + sid::pm_ws_kernel")


@pytest.mark.gpu
@pytest.mark.parametrize("path,kernel", [(None, "sid::pm_ws_kernel"), ("tc", "sid::pm_tc_kernel"),
                                         ("imma", "sid::pm_points_kernel<imma>")])
def test_median_rank_of_the_wide_select(gpu_ctx, monkeypatch, path, kernel):
    """MEDIAN_RANK_POINTS at border 20, hes_norm only (the fast Hessian normalisation): many Hessian values share the
    median's histogram bin, so the wide select decides the median, and its neighbour in rank would change h."""
    c = np.array([p[0] for p in MEDIAN_RANK_POINTS], dtype=np.float64)
    r = np.array([p[1] for p in MEDIAN_RANK_POINTS], dtype=np.float64)
    img1, img2 = images("lowcontrast")
    if path is not None:
        monkeypatch.setenv("SID_PM_PATH", path)
    gpu_ctx.set_pair(img1, img2)
    got, st = gpu_ctx.run(c, r, c, r, np.full(c.size, 20.0), 35, [-3, 0, 3], 0.0, want_status=True)
    assert gpu_ctx.last_kernel_name == kernel, gpu_ctx.last_kernel_name
    ref, st_ref = co.use_mcc_batch(c, r, c, r, np.full(c.size, 20.0), img1, img2, 35, 0.0, angles=[-3, 0, 3])
    assert_equals_exact_oracle(got, ref, st, st_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", CLASSES)
def test_run_pair_equals_exact_oracle(gpu_ctx, kind):
    img1, img2 = images(kind)
    brd = 20 + np.arange(n_points(kind)) % 21
    pts = points(kind, 35, brd.astype(np.float64))
    got, st = gpu_ctx.run_pair(img1, img2, *pts, 35, [-3, 0, 3], 0.0, want_status=True)
    ref, st_ref = co.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[-3, 0, 3])
    assert_equals_exact_oracle(got, ref, st, st_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("name,win,tpl", template_cases(), ids=[c[0] for c in template_cases()])
def test_single_call_match_template_equals_exact_oracle(gpu_ctx, name, win, tpl):
    got = gpu_ctx.match_template(win, tpl)
    assert np.array_equal(got, co.match_template(np.ascontiguousarray(win), np.ascontiguousarray(tpl))), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(hessian_maps()))
def test_single_call_get_hessian_equals_exact_oracle(gpu_ctx, name):
    from sea_ice_drift_b200 import _lib
    ccm = hessian_maps()[name]
    for hn in (False, True):
        for hs in (False, True):
            got = gpu_ctx.get_hessian(ccm, _lib.flags_from_kwargs(hn, hs, False))
            ref = co.get_hessian(ccm, hes_norm=hn, hes_smth=hs)
            assert np.array_equal(np.isnan(got), np.isnan(ref)), (name, hn, hs)
            fin = np.isfinite(ref)
            assert np.array_equal(got[~fin], ref[~fin], equal_nan=True), (name, hn, hs)
            assert np.all(np.abs(got[fin] - ref[fin]) <= 4e-6 * (1 + np.abs(ref[fin]))), (name, hn, hs)


@pytest.mark.gpu
@pytest.mark.parametrize("s,border", [(35, 20), (35, 33), (21, 9), (50, 14)])
def test_single_call_rotate_and_match_flat_template(s, border):
    """A flat template: the map is all 1, so the peak is index 0 of the first angle, r == 1 and h = 0/0."""
    import sea_ice_drift_b200 as sid
    img1, img2 = images("plateaus")
    mid = (P1[0] + P1[1]) // 2
    hws = int(s / 2.)
    win = img2[mid - hws - border:mid + hws + border + 1, mid - hws - border + 3:mid + hws + border + 4]
    angles = [-3, 0, 3]
    for mcc in (False, True):
        dc, dr, a, r, h, ccm, tpl = sid.rotate_and_match(img1, mid, mid, s, win, 0.0, angles=angles, mcc_norm=mcc)
        assert np.all(tpl == 128) and np.all(ccm == 1.0)
        assert (dc, dr, a) == (-(win.shape[1] - s) / 2., -(win.shape[0] - s) / 2., angles[0])
        assert np.isnan(h)
        assert (np.isnan(r) if mcc else r == 1.0)
    raw = sid.rotate_and_match(img1, mid, mid, s, win, 0.0, angles=angles, hes_norm=False)
    assert raw[:4] == (dc, dr, angles[0], 1.0) and raw[4] == 0.0
