"""Per-vector drift uncertainty (SID_UNCERT, Context.uncertainty, use_mcc_batch(uncertainty=True),
pattern_matching(..., subpixel=True, uncertainty=True)).

``record`` below restates the rule of include/sid_b200.h with Python integers for the exact sums (``float(int)`` is
correctly rounded, Python floats are IEEE doubles without contraction).  It reads the exact oracle's winning maps and
templates and the search window as ``use_mcc`` slices it.  On the CPU it is checked against an independent float64
computation, closed forms, the NaN rules and a calibration probe with a known noise level; the GPU must match it bit
for bit on every kernel family and through every entry point."""
import math

import numpy as np
import pytest

from sea_ice_drift_b200 import _lib, pmlib, sharding
from sea_ice_drift_b200 import synthetic as syn
from sea_ice_drift_b200.seaicedrift import SeaIceDrift
from oracle import c_oracle as co
from tests import masked_oracle as mo
from tests import test_degenerate_content as dg
from tests.test_gpu_maps import window, window_rule
from tests.test_masked_matching import _land_pair, _land_points
from tests.test_subpixel import peak_offsets

NAN = float("nan")
# positions in the rule's order: P0, X-, X+, Y-, Y+ (row, column offsets from the peak)
OFFSETS = ((0, 0), (0, -1), (0, 1), (-1, 0), (1, 0))


# ---------------------------------------------------------------------------------------------------- restatement
def _exact_dot(x, y):
    """sum x_k y_k of two int64 arrays with |x|, |y| < 2^44, exactly: 22-bit halves keep every partial sum in int64."""
    xh, xl = np.divmod(x, 1 << 22)
    yh, yl = np.divmod(y, 1 << 22)
    hh = int(np.dot(xh, yh))
    mid = int(np.dot(xh, yl)) + int(np.dot(xl, yh))
    return (hh << 44) + (mid << 22) + int(np.dot(xl, yl))


def integer_sums(tpl, win, bi, bj, masked):
    """n, Vt and per used position P: w_k(P) (None where unused), A(P), V(P); x_k(P) = t_k w_k(P).  Positions off the
    map, or on an axis whose peak lies on the map's edge, are unused."""
    s = tpl.shape[0]
    RH, RW = win.shape[0] - s + 1, win.shape[1] - s + 1
    T = tpl.astype(np.int64).ravel()
    M = (T > 0) if masked else np.ones(T.size, bool)
    n = int(M.sum())
    St = int(T[M].sum())
    t = np.where(M, n * T - St, 0)
    ux, uy = 0 < bj < RW - 1, 0 < bi < RH - 1
    used = (True, ux, ux, uy, uy)
    x, A, V = [None] * 5, [0] * 5, [0] * 5
    for p, (di, dj) in enumerate(OFFSETS):
        if not used[p]:
            continue
        Wp = win[bi + di:bi + di + s, bj + dj:bj + dj + s].astype(np.int64).ravel()
        Sw = int(Wp[M].sum())
        w = np.where(M, n * Wp - Sw, 0)
        x[p] = t * w
        A[p] = int(x[p].sum())
        V[p] = int(np.dot(w, w))
    return n, int(np.dot(t, t)), t, used, x, A, V


def ieee_div(a, b):
    """a / b with IEEE semantics for b = 0 (a flat template has Vt = 0 and a zero numerator: NaN)"""
    if b == 0.0:
        return NAN if a == 0.0 or math.isnan(a) else math.copysign(math.inf, a) * math.copysign(1.0, b)
    return a / b


def covariance_k(tpl, win, bi, bj, masked):
    """The 5 x 5 K of the rule (NaN where a position is unused or has V = 0), evaluated once per unordered pair with
    P the earlier position."""
    n, Vt, _, used, x, A, V = integer_sums(tpl, win, bi, bj, masked)
    K = np.full((5, 5), NAN)
    for p in range(5):
        for q in range(p, 5):
            if used[p] and used[q] and V[p] and V[q]:
                num = n * _exact_dot(x[p], x[q]) - A[p] * A[q]
                k = ieee_div(float(num), ((float(n) * float(Vt)) * math.sqrt(float(V[p]))) * math.sqrt(float(V[q])))
                K[p, q] = K[q, p] = k
    return K


def vertex_grad(a, b, c):
    a, b, c = float(a), float(b), float(c)
    p, q = b - a, b - c
    w = (p + q) * (p + q)
    return (-q / w, (q - p) / w, p / w)


def quad(K, ul, g, vl, gp):
    h = [(K[u, vl[0]] * gp[0] + K[u, vl[1]] * gp[1]) + K[u, vl[2]] * gp[2] for u in ul]
    return (g[0] * h[0] + g[1] * h[1]) + g[2] * h[2]


def record(ccm, tpl, win, masked=False, peak=None):
    """(var_c, var_r, cov_cr) of one row from its raw winning map, template and search window."""
    m = np.asarray(ccm, dtype=np.float32)
    bi, bj = np.unravel_index(int(np.argmax(m)), m.shape) if peak is None else peak
    K = covariance_k(tpl, win, bi, bj, masked)
    RH, RW = m.shape
    ux, uy = 0 < bj < RW - 1, 0 < bi < RH - 1
    lx, ly = (1, 0, 2), (3, 0, 4)
    gx = vertex_grad(m[bi, bj - 1], m[bi, bj], m[bi, bj + 1]) if ux else None
    gy = vertex_grad(m[bi - 1, bj], m[bi, bj], m[bi + 1, bj]) if uy else None
    var_c = quad(K, lx, gx, lx, gx) if ux else NAN
    var_r = quad(K, ly, gy, ly, gy) if uy else NAN
    cov = quad(K, lx, gx, ly, gy) if ux and uy else NAN
    return var_c, var_r, cov


def recover_peak(m, e_c, e_r):
    """The kernel's peak recovery: integers within 0.5 + 1e-6 of the table's position in map coordinates, the largest
    map value among them, ties to the lowest flat index."""
    RH, RW = m.shape
    cand_c = [j for j in range(math.ceil(e_c - 0.5 - 1e-6), math.floor(e_c + 0.5 + 1e-6) + 1) if 0 <= j < RW][:2]
    cand_r = [i for i in range(math.ceil(e_r - 0.5 - 1e-6), math.floor(e_r + 0.5 + 1e-6) + 1) if 0 <= i < RH][:2]
    best, at = -np.inf, None
    for i in cand_r:
        for j in cand_c:
            if m[i, j] > best:
                best, at = m[i, j], (i, j)
    return at


def table_position(m, c2fg, r2fg, H, W, s):
    """c2, r2 as the kernels write them with SID_SUBPIXEL, and e_c, e_r as the pass reads them back."""
    bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)
    dx, dy = peak_offsets(m)
    c2 = (c2fg + (float(bj) - (W - s) / 2.0)) + float(dx)
    r2 = (r2fg + (float(bi) - (H - s) / 2.0)) + float(dy)
    return (c2 - c2fg) + (W - s) / 2.0, (r2 - r2fg) + (H - s) / 2.0


def expected(img1, img2, pts, s, angles, o, masked=False):
    """(n, 3) records of the rule from the exact oracle (the masked oracle with ``masked``), NaN for other rows."""
    c1, r1, c2, r2, b = pts
    _, st = (mo if masked else co).use_mcc_batch(*pts, img1, img2, s, 0.0, angles=angles, **o)
    out = np.full((c1.size, 3), NAN)
    for i in np.flatnonzero(st > 0):
        win = window(img2, s, c2[i], r2[i], b[i])
        ora = mo if masked else co
        res = ora.rotate_and_match(img1, c1[i], r1[i], s, win, 0.0, angles=angles, **o)
        out[i] = record(res[5], res[6], win, masked=bool(masked and res[7] == 2))
    return out, st


def float64_k(tpl, win, bi, bj, masked):
    """Independent float64 K: explicit per-pixel contributions x_k(P) and NumPy's population covariance, times n."""
    T = tpl.astype(np.float64).ravel()
    M = (T > 0) if masked else np.ones(T.size, bool)
    n = M.sum()
    s = tpl.shape[0]
    tc = np.where(M, T - T[M].mean(), 0.0)
    xs = []
    for di, dj in OFFSETS:
        Wp = win[bi + di:bi + di + s, bj + dj:bj + dj + s].astype(np.float64).ravel()
        wc = np.where(M, Wp - Wp[M].mean(), 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):              # flat patches: NaN, as the rule's V = 0
            xs.append((tc * wc / (np.sqrt(np.sum(tc * tc)) * np.sqrt(np.sum(wc * wc))))[M])
    return n * np.cov(np.array(xs), bias=True), [x.sum() for x in xs]


# ---------------------------------------------------------------------------------------------------- CPU
def _speckle_rows(s=35, border=6, n_side=5, noise=6.0, seed=3):
    img1 = syn.speckle_image((300, 300), seed)
    img2 = syn.warp_pair(img1, syn.shift_matrix(2.4, -1.7), seed, noise_sd=noise)
    g = np.linspace(60, 230, n_side)
    c1, r1 = [a.ravel() for a in np.meshgrid(g, g)]
    pts = [c1, r1, np.round(c1 + 2.4), np.round(r1 - 1.7), np.full(c1.size, float(border))]
    return img1, img2, pts


def _rows_of(img1, img2, pts, s, angles=(0,), masked=False):
    """(map, template, window, masked) of every valid (or masked) row by the exact oracle"""
    c1, r1, c2, r2, b = pts
    ora = mo if masked else co
    out = []
    for i in range(c1.size):
        if window_rule(img2, s, c1[i], r1[i], c2[i], r2[i], b[i]) is None:
            continue
        win = window(img2, s, c2[i], r2[i], b[i])
        res = ora.rotate_and_match(img1, c1[i], r1[i], s, win, 0.0, angles=list(angles))
        if masked and res[7] == 0 or not masked and not np.isfinite(res[0]):
            continue
        out.append((res[5], res[6], win, bool(masked and res[7] == 2)))
    return out


def _check_float64(rows):
    checked = 0
    for m, tpl, win, msk in rows:
        bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)
        if not (0 < bi < m.shape[0] - 1 and 0 < bj < m.shape[1] - 1):
            continue
        K = covariance_k(tpl, win, bi, bj, msk)
        K64, sums = float64_k(tpl, win, bi, bj, msk)
        ok = np.isfinite(np.diag(K))
        if not ok.all():
            continue
        scale = np.sqrt(np.outer(np.diag(K), np.diag(K)))
        assert np.all(np.abs(K - K64) <= 1e-9 * scale + 1e-300), (K, K64)
        # the contributions sum to the map value (the oracle's float32 map; OpenCV's formula rounds differently)
        for p, (di, dj) in enumerate(OFFSETS):
            assert abs(sums[p] - float(m[bi + di, bj + dj])) <= 2e-6, (sums[p], m[bi + di, bj + dj])
        checked += 1
    return checked


def test_restatement_equals_independent_float64_on_speckle():
    img1, img2, pts = _speckle_rows()
    assert _check_float64(_rows_of(img1, img2, pts, 35, (-3, 0, 3))) >= 20


def test_restatement_equals_independent_float64_on_masked_rows():
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 12)
    rows = [r for r in _rows_of(img1, img2, pts, 35, (-3, 0, 3), masked=True) if r[3]]
    assert len(rows) >= 5
    assert _check_float64(rows) >= 5


@pytest.mark.parametrize("kind", dg.CLASSES)
def test_restatement_on_degenerate_content(kind):
    """Flat windows, periodic ties and low contrast: the float64 check where every K entry exists, and the NaN rules
    (V = 0, flat templates, edge peaks) elsewhere."""
    img1, img2 = dg.images(kind)
    pts = dg.points(kind, 35, np.full(dg.n_points(kind), 8.0))
    rows = _rows_of(img1, img2, pts, 35, (-3, 0, 3))
    assert rows
    _check_float64(rows)
    for m, tpl, win, msk in rows:
        rec = record(m, tpl, win, msk)
        bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)
        _, Vt, _, used, _, _, V = integer_sums(tpl, win, bi, bj, msk)
        zero = [p for p in range(5) if used[p] and V[p] == 0]
        if not used[1] or any(p in (0, 1, 2) for p in zero) or Vt == 0:
            assert math.isnan(rec[0]) and math.isnan(rec[2])
        if not used[3] or any(p in (0, 3, 4) for p in zero) or Vt == 0:
            assert math.isnan(rec[1]) and math.isnan(rec[2])
        if used[1] and used[3] and not zero and Vt:
            assert all(math.isfinite(v) for v in rec)


def test_closed_forms_and_nan_rules():
    rng = np.random.default_rng(0)
    for _ in range(200):
        a, c = rng.uniform(-1, 1, 2).astype(np.float32)
        b = np.float32(max(a, c) + rng.uniform(1e-6, 1))
        g = vertex_grad(a, b, c)
        assert abs(sum(g)) <= 1e-12 * max(abs(v) for v in g)
    img1, img2, pts = _speckle_rows(n_side=3)
    for m, tpl, win, msk in _rows_of(img1, img2, pts, 35):
        bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)
        K = covariance_k(tpl, win, bi, bj, msk)
        assert np.allclose(K, K.T, equal_nan=True)
        assert np.linalg.eigvalsh(K).min() >= -1e-9 * np.abs(K).max()          # positive semi-definite
        var_c, var_r, cov = record(m, tpl, win)
        assert var_c > 0 and var_r > 0 and cov * cov <= var_c * var_r * (1 + 1e-9)
    # a peak on the map's first column / last row: that axis and the covariance are NaN
    m, tpl, win, _ = _rows_of(img1, img2, pts, 35)[0]
    mm = m.copy()
    bi = mm.shape[0] - 1
    mm[bi, 0] = 2.0
    rec = record(mm, tpl, win)
    assert math.isnan(rec[0]) and math.isnan(rec[1]) and math.isnan(rec[2])
    mm = m.copy()
    mm[4, 0] = 2.0
    rec = record(mm, tpl, win)
    assert math.isnan(rec[0]) and math.isfinite(rec[1]) and math.isnan(rec[2])
    # V = 0: a flat window patch at X+
    win2 = win.copy()
    bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)
    win2[bi:bi + 35, bj + 1:bj + 36] = 77
    rec = record(m, tpl, win2, peak=(bi, bj))
    assert math.isnan(rec[0]) and math.isfinite(rec[1]) and math.isnan(rec[2])


def test_peak_recovery_on_constructed_maps():
    """dx = +0.5 exactly (a tie with the right-hand neighbour), peaks below 1e-6 and negative maps: the recovery rule
    returns np.argmax's first maximum."""
    rng = np.random.default_rng(1)
    s, W, H = 35, 35 + 12, 35 + 10
    n_half = n_tiny = 0
    for k in range(3000):
        m = rng.normal(0, 1, (H - s + 1, W - s + 1)).astype(np.float32)
        if k % 3 == 0:
            m *= np.float32(1e-7)
        i0, j0 = rng.integers(0, m.shape[0]), rng.integers(0, m.shape[1])
        m[i0, j0] = m.max() + np.float32(abs(m.max()) * 0.01 + 1e-9)
        if k % 2 == 0 and j0 + 1 < m.shape[1]:
            m[i0, j0 + 1] = m[i0, j0]                                         # dx = +0.5
        if k % 5 == 0 and i0 + 1 < m.shape[0]:
            m[i0 + 1, j0] = m[i0, j0]                                         # dy = +0.5
        c2fg, r2fg = float(rng.integers(100, 5000)), float(rng.integers(100, 5000))
        e_c, e_r = table_position(m, c2fg, r2fg, H, W, s)
        n_half += abs(e_c - round(e_c)) == 0.5
        n_tiny += m.max() < 1e-6
        assert recover_peak(m, e_c, e_r) == np.unravel_index(int(np.argmax(m)), m.shape)
    assert n_half >= 300 and n_tiny >= 300


def test_peak_recovery_on_oracle_tables():
    img1, img2, pts = _speckle_rows(n_side=6)
    cases = [(img1, img2, pts)]
    for kind in dg.CLASSES:
        i1, i2 = dg.images(kind)
        cases.append((i1, i2, dg.points(kind, 35, np.full(dg.n_points(kind), 8.0))))
    n = 0
    for i1, i2, p in cases:
        c1, r1, c2, r2, b = p
        for i in range(c1.size):
            win = window(i2, 35, c2[i], r2[i], b[i])
            res = co.rotate_and_match(i1, c1[i], r1[i], 35, win, 0.0, angles=[-3, 0, 3])
            if not np.isfinite(res[0]):
                continue
            e_c, e_r = table_position(res[5], c2[i], r2[i], win.shape[0], win.shape[1], 35)
            assert recover_peak(res[5], e_c, e_r) == np.unravel_index(int(np.argmax(res[5])), res[5].shape)
            n += 1
    assert n >= 60


NOISE = (3.0, 6.0, 12.0, 24.0)
SHIFT = (2.35, -1.6)


def calibration(noise_sd, n_seeds=20, n_side=6, s=35, border=4):
    """Per grid point: the refined column / row offsets over noise seeds, and the predicted sigma per seed."""
    img1 = syn.speckle_image((360, 360), 21)
    g = np.linspace(70, 280, n_side)
    c1, r1 = [a.ravel() for a in np.meshgrid(g, g)]
    c2, r2 = np.round(c1 + SHIFT[0]), np.round(r1 + SHIFT[1])
    pos = np.full((n_seeds, c1.size, 2), NAN)
    sig = np.full((n_seeds, c1.size, 2), NAN)
    for k in range(n_seeds):
        img2 = syn.warp_pair(img1, syn.shift_matrix(*SHIFT), 100 + k, noise_sd=noise_sd)
        for i in range(c1.size):
            win = window(img2, s, c2[i], r2[i], border)
            res = co.rotate_and_match(img1, c1[i], r1[i], s, win, 0.0, angles=[0])
            dx, dy = peak_offsets(res[5])
            pos[k, i] = (c2[i] + res[0]) + dx, (r2[i] + res[1]) + dy
            rec = record(res[5], res[6], win)
            sig[k, i] = math.sqrt(rec[0]), math.sqrt(rec[1])
    return pos, sig


@pytest.fixture(scope="module")
def calibration_runs():
    return {sd: calibration(sd) for sd in NOISE}


def calibration_ratios(calibration_runs, sd):
    """(RMS error against the known shift over points, axes and seeds, median seed-to-seed spread per point and axis)
    over the median predicted sigma"""
    pos, sig = calibration_runs[sd]
    g = np.linspace(70, 280, 6)
    c1, r1 = [a.ravel() for a in np.meshgrid(g, g)]
    # the table's c2 / r2 of a point moved by SHIFT: c1 + dx - 1 (the template's centre is int(s / 2) + 1)
    err = pos - np.stack([c1 + SHIFT[0] - 1, r1 + SHIFT[1] - 1], -1)[None]
    med = np.nanmedian(sig)
    return np.sqrt(np.nanmean(err ** 2)) / med, np.median(np.nanstd(pos, axis=0)) / med


def test_calibration_probe(calibration_runs):
    """Known sub-pixel shift, independent pixel noise of known sd, 20 seeds on a 6 x 6 grid.  The predicted sigma rises
    with the noise; at noise 6 and 12 the RMS error against the known shift is within 3x of the median predicted sigma.
    The seed-to-seed spread alone is well below it (ratio ~0.1 ... 0.2, DESIGN 4.1g): the per-pixel mismatch the rule
    sees includes the deterministic part (bilinear resampling of the moved image), which every seed shares."""
    med = [np.nanmedian(calibration_runs[sd][1]) for sd in NOISE]
    assert all(a < b for a, b in zip(med, med[1:])), med
    for sd in (6.0, 12.0):
        rms_ratio, spread_ratio = calibration_ratios(calibration_runs, sd)
        assert 1 / 3 <= rms_ratio <= 3, (sd, rms_ratio)
        assert spread_ratio < 1, (sd, spread_ratio)


def test_uncertainty_keyword_refusals():
    calls = []

    def matcher(*a):
        calls.append(a)
        return np.zeros((3, 3), np.float32)

    img = syn.speckle_image((120, 120), 1)
    with pytest.raises(ValueError, match="subpixel"):
        _lib.flags_from_options(dict(uncertainty=True))
    assert _lib.flags_from_options(dict(subpixel=True, uncertainty=True)) == \
        _lib.SID_HES_NORM | _lib.SID_SUBPIXEL | _lib.SID_UNCERT
    assert _lib.flags_from_options(dict(subpixel=True)) & _lib.SID_UNCERT == 0
    with pytest.raises(ValueError, match="subpixel"):
        pmlib.use_mcc_batch([60.0], [60.0], [60.0], [60.0], [10.0], img, img, 35, 0.0, uncertainty=True)
    with pytest.raises(ValueError, match="uncertainty=True needs the built-in matcher"):
        pmlib.use_mcc_batch([60.0], [60.0], [60.0], [60.0], [10.0], img, img, 35, 0.0, template_matcher=matcher,
                            uncertainty=True)
    for fn in (sharding.use_mcc_batch_split, sharding.use_mcc_batch_sharded):
        with pytest.raises(ValueError, match="uncertainty=True runs on one GPU"):
            fn([60.0], [60.0], [60.0], [60.0], [10.0], img, img, 35, 0.0, subpixel=True, uncertainty=True)
    with pytest.raises(ValueError, match="uncertainty=True runs on one GPU"):
        sharding.use_mcc_series([], 35, subpixel=True, uncertainty=True)
    n = syn.ArrayDomain(img)
    lon, lat = n.transform_points(np.array([[60.0]]), np.array([[60.0]]))
    with pytest.raises(ValueError, match="uncertainty=True"):
        pmlib.pattern_matching(lon, lat, n, [60.0], [60.0], n, [60.0], [60.0], template_matcher=matcher,
                               subpixel=True, uncertainty=True)
    with pytest.raises(ValueError, match="subpixel"):
        pmlib.pattern_matching(lon, lat, n, [60.0], [60.0], n, [60.0], [60.0], uncertainty=True)
    assert not calls


def test_under_a_process_group_pattern_matching_refuses(monkeypatch):
    import sea_ice_drift_b200.sharding as sh
    monkeypatch.setattr(sh, "_dist", lambda: object())
    img = syn.speckle_image((120, 120), 1)
    n = syn.ArrayDomain(img)
    lon, lat = n.transform_points(np.array([[60.0]]), np.array([[60.0]]))
    with pytest.raises(ValueError, match="uncertainty=True runs on one GPU"):
        pmlib.pattern_matching(lon, lat, n, [60.0], [60.0], n, [60.0], [60.0], subpixel=True, uncertainty=True)


def test_abi_exports_sid_get_uncertainty():
    assert "sid_get_uncertainty" in _lib.EXPORTS
    assert _lib.SID_UNCERT == 64
    lib = _lib.load_library()
    assert hasattr(lib, "sid_get_uncertainty")


# ---------------------------------------------------------------------------------------------------- GPU
def flags_of(o, masked=False, uncertainty=True):
    return _lib.flags_from_kwargs(o.get("hes_norm", True), o.get("hes_smth", False), o.get("mcc_norm", False), True,
                                  masked, uncertainty)


def assert_records(got, exp):
    assert got.shape == exp.shape
    assert np.array_equal(np.isnan(got), np.isnan(exp)), np.flatnonzero((np.isnan(got) != np.isnan(exp)).any(1))
    ok = ~np.isnan(exp)
    bad = np.flatnonzero(((got.view(np.uint64) != exp.view(np.uint64)) & ok).any(axis=1))
    assert bad.size == 0, (bad[:5], got[bad[:3]], exp[bad[:3]])


# (name, img_size, angles, border, environment)
FAMILIES = [
    ("ws", 35, [-3, 0, 3], 16, {}),
    ("tc", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "tc"}),
    ("imma", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "imma"}),
    ("dp4a", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "dp4a"}),
    ("ws_even_1angle", 34, [0], 14, {}),
    ("tc_even_7angles", 50, [-9, -6, -3, 0, 3, 6, 9], 22, {"SID_PM_PATH": "tc"}),
    ("dp4a_odd_7angles", 21, [-9, -6, -3, 0, 3, 6, 9], 14, {"SID_PM_PATH": "dp4a"}),
    ("imma_s96", 96, [-3, 0, 3], 12, {"SID_PM_PATH": "imma"}),
]
OPTION_SETS = {"default": {}, "all": dict(hes_smth=True, mcc_norm=True, rot_order=1), "raw_rot1": dict(hes_norm=False,
                                                                                                     rot_order=1)}
CASES = [(f, o) for f in FAMILIES for o in (OPTION_SETS if f[0] in ("ws", "tc", "dp4a") else ("default",))]


@pytest.mark.gpu
@pytest.mark.parametrize("family,option_set", CASES, ids=["%s-%s" % (f[0], o) for f, o in CASES])
def test_every_kernel_family_equals_restatement(gpu_ctx, monkeypatch, family, option_set):
    """Masked land rows, rejected rows, templates crossing image 1's edges: the records equal the restatement on the
    exact masked oracle's maps bit for bit; the table and status equal the call without the flag, which issues one
    launch fewer."""
    name, s, angles, border, env = family
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    o = OPTION_SETS[option_set]
    img1, img2 = _land_pair()
    pts = _land_points(img1, s, border)
    gpu_ctx.set_pair(img1, img2)
    rot = o.get("rot_order", 0)
    n0 = gpu_ctx.launch_count
    plain, st_plain = gpu_ctx.run(*pts, s, angles, 0.0, rot, flags_of(o, True, False), want_status=True)
    n_plain = gpu_ctx.launch_count - n0
    kernel = gpu_ctx.last_kernel_name
    got, st = gpu_ctx.run(*pts, s, angles, 0.0, rot, flags_of(o, True), want_status=True)
    assert gpu_ctx.launch_count - n0 - n_plain == n_plain + 1
    assert gpu_ctx.last_kernel_name == kernel
    assert got.tobytes() == plain.tobytes() and np.array_equal(st, st_plain)
    oo = {k: v for k, v in o.items()}
    exp, st_exp = expected(img1, img2, pts, s, angles, oo, masked=True)
    assert np.array_equal(st, st_exp)
    assert (st == 2).sum() >= 3 and (st == 1).sum() >= 5
    assert_records(gpu_ctx.uncertainty(pts[0].size), exp)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", dg.CLASSES)
@pytest.mark.parametrize("path", (None, "tc", "imma", "dp4a"))
def test_degenerate_content_equals_restatement(gpu_ctx, monkeypatch, kind, path):
    if path:
        monkeypatch.setenv("SID_PM_PATH", path)
    img1, img2 = dg.images(kind)
    pts = dg.points(kind, 35, np.full(dg.n_points(kind), 12.0))
    gpu_ctx.set_pair(img1, img2)
    gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, 0, flags_of({}))
    exp, _ = expected(img1, img2, pts, 35, [-3, 0, 3], {})
    assert_records(gpu_ctx.uncertainty(pts[0].size), exp)


@pytest.mark.gpu
def test_edge_peaks_equal_restatement(gpu_ctx):
    """First guesses off by the whole border: peaks on the map's edges give NaN axes."""
    img1, img2, pts = _speckle_rows(n_side=6, border=3)
    c1, r1, c2, r2, b = pts
    off = np.tile([[3, 0], [-3, 0], [0, 3], [0, -3], [3, 3], [0, 0]], (6, 1))[:c1.size]
    pts = [c1, r1, c2 + off[:, 0], r2 + off[:, 1], b]
    gpu_ctx.set_pair(img1, img2)
    gpu_ctx.run(*pts, 35, [0], 0.0, 0, flags_of({}))
    exp, _ = expected(img1, img2, pts, 35, [0], {})
    got = gpu_ctx.uncertainty(c1.size)
    assert_records(got, exp)
    assert np.isnan(got[:, 0]).sum() >= 5 and np.isfinite(got[:, 0]).sum() >= 5


def _two_class_points(img1):
    pts = _land_points(img1, 35, 20, seed=1)
    c1, r1, c2, r2, _ = pts
    reps = 12                                                           # >= 512 points: run_device splits classes
    k = np.arange(c1.size * reps)
    brd = np.where(k % 4 == 3, 21 + k % 20, 16).astype(np.float64)
    return [np.tile(c1, reps), np.tile(r1, reps), np.tile(c2, reps), np.tile(r2, reps), brd]


@pytest.mark.gpu
def test_entry_points_give_identical_records(gpu_ctx, monkeypatch):
    import torch
    img1, img2 = _land_pair(side=420, seed=5)
    pts = _two_class_points(img1)
    n = pts[0].size
    flags = flags_of({}, True)
    gpu_ctx.set_pair(img1, img2)
    ref, st = gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, 0, flags, want_status=True)
    assert " + " in gpu_ctx.last_kernel_name                            # two border classes
    rec = gpu_ctx.uncertainty(n)
    exp, _ = expected(img1, img2, pts, 35, [-3, 0, 3], {}, masked=True)
    assert_records(rec, exp)
    assert np.isfinite(rec[st == 2]).all(axis=1).sum() >= 10
    for bands in ("3", "8"):
        monkeypatch.setenv("SID_BANDS", bands)
        got = gpu_ctx.run_pair(img1, img2, *pts, 35, [-3, 0, 3], 0.0, 0, flags)
        assert got.tobytes() == ref.tobytes()
        assert gpu_ctx.uncertainty(n).tobytes() == rec.tobytes()
    monkeypatch.delenv("SID_BANDS")
    out, maps, tpls = gpu_ctx.run_maps(*pts, 35, [-3, 0, 3], 0.0, 0, flags)
    assert out.tobytes() == ref.tobytes() and gpu_ctx.uncertainty(n).tobytes() == rec.tobytes()
    plain_maps = gpu_ctx.run_maps(*pts, 35, [-3, 0, 3], 0.0, 0, flags_of({}, True, False))
    assert all((a is None and b is None) or a.tobytes() == b.tobytes() for a, b in zip(maps, plain_maps[1]))
    assert tpls.tobytes() == plain_maps[2].tobytes()
    dev = torch.device("cuda", gpu_ctx.device)
    d_pts = torch.from_numpy(np.stack(pts)).to(dev)
    for with_status in (True, False):
        d_out = torch.full((n, 5), -7.0, dtype=torch.float64, device=dev)
        d_st = torch.full((n,), 9, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        gpu_ctx.run_device(n, *[d_pts[j].data_ptr() for j in range(5)], 40, 35, [-3, 0, 3], 0.0, d_out.data_ptr(),
                           d_st.data_ptr() if with_status else 0, flags=flags)
        gpu_ctx.synchronize()
        assert d_out.cpu().numpy().tobytes() == ref.tobytes()
        assert gpu_ctx.uncertainty(n).tobytes() == rec.tobytes()


@pytest.mark.gpu
def test_with_peaks_the_peaks_are_unchanged(gpu_ctx):
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 16)
    n = pts[0].size
    gpu_ctx.set_pair(img1, img2)
    a = gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, 0, flags_of({}, True, False) | _lib.SID_PEAKS)
    pa = gpu_ctx.peaks(n)
    b = gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, 0, flags_of({}, True) | _lib.SID_PEAKS)
    assert a.tobytes() == b.tobytes() and gpu_ctx.peaks(n).tobytes() == pa.tobytes()
    t, p, u = pmlib.use_mcc_batch(*pts, img1, img2, 35, 0.0, subpixel=True, masked=True, peaks=True, uncertainty=True,
                                  angles=[-3, 0, 3])
    assert t.tobytes() == a.tobytes() and p.tobytes() == pa.tobytes() and u.shape == (n, 3)


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(gpu_ctx):
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 16)
    n = pts[0].size
    gpu_ctx.set_pair(img1, img2)
    n0 = gpu_ctx.launch_count
    with pytest.raises(ValueError, match="SID_SUBPIXEL"):
        gpu_ctx.run(*pts, 35, [0], 0.0, 0, _lib.SID_HES_NORM | _lib.SID_UNCERT)
    with pytest.raises(ValueError, match="SID_SUBPIXEL"):
        gpu_ctx.run_maps(*pts, 35, [0], 0.0, 0, _lib.SID_HES_NORM | _lib.SID_UNCERT)
    assert gpu_ctx.launch_count == n0
    with pytest.raises(ValueError, match="SID_UNCERT"):
        gpu_ctx.uncertainty(n)                                          # the failed call reset the records
    gpu_ctx.run(*pts, 35, [0], 0.0, 0, flags_of({}))
    rec = gpu_ctx.uncertainty(n)
    with pytest.raises(ValueError, match="SID_UNCERT"):
        gpu_ctx.uncertainty(n - 1)
    with pytest.raises(ValueError):
        gpu_ctx.rotate_and_match(img1, 100.0, 100.0, 35, img2[60:140, 60:140], [0], 0.0, flags=flags_of({}))
    gpu_ctx.run(*[np.zeros(0)] * 5, 35, [0], 0.0, 0, flags_of({}))
    assert gpu_ctx.uncertainty(0).shape == (0, 3)
    gpu_ctx.run(*pts, 35, [0], 0.0, 0, _lib.SID_HES_NORM | _lib.SID_SUBPIXEL)
    with pytest.raises(ValueError, match="SID_UNCERT"):
        gpu_ctx.uncertainty(n)
    gpu_ctx.run(*pts, 35, [0], 0.0, 0, flags_of({}))
    assert gpu_ctx.uncertainty(n).tobytes() == rec.tobytes()


def _drop_in_scene(side=900, grid=24):
    img1 = syn.speckle_image((side, side), 7)
    m = syn.shift_matrix(5.3, 3.6)
    img2 = syn.warp_pair(img1, m, 7)
    for im in (img1, img2):
        im[:140, :200] = 0                                              # a no-data corner: NaN vectors
    n1, n2 = syn.ArrayDomain(img1, lat0=0.0), syn.ArrayDomain(img2, lat0=0.0)
    rng = np.random.default_rng(2)
    kx, ky = rng.uniform(220, side - 40, 3000), rng.uniform(160, side - 40, 3000)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    gx, gy = np.meshgrid(np.linspace(60, side - 60, grid), np.linspace(60, side - 60, grid))
    lon, lat = n2.transform_points(gx, gy)
    ll = (*n1.transform_points(kx, ky), *n2.transform_points(k2x + rng.normal(0, 0.5, kx.size),
                                                             k2y + rng.normal(0, 0.5, ky.size)))
    return n1, n2, lon, lat, ll


@pytest.mark.gpu
def test_get_drift_pm_uncertainty_device_and_host_paths(gpu_ctx):
    n1, n2, lon, lat, ll = _drop_in_scene()
    sid = SeaIceDrift(n1, n2)
    kw = dict(angles=[-3, 0, 3], img_size=35, subpixel=True)
    base = sid.get_drift_PM(lon, lat, *ll, **kw)
    dev = sid.get_drift_PM(lon, lat, *ll, uncertainty=True, **kw)
    host = sid.get_drift_PM(lon, lat, *ll, uncertainty=True, device_epilogue=False, **kw)
    assert len(dev) == 9 and len(host) == 9
    for a, b in zip(base, dev[:7]):
        assert a.tobytes() == b.tobytes()
    u, su, sv = dev[0], dev[7], dev[8]
    assert np.isnan(u).sum() >= 10 and np.isfinite(u).sum() >= 300
    assert np.all(np.isnan(su[np.isnan(u)])) and np.all(np.isnan(sv[np.isnan(u)]))
    assert np.isfinite(su[np.isfinite(u)]).mean() >= 0.95 and np.isfinite(sv[np.isfinite(u)]).mean() >= 0.95
    for a, b in ((su, host[7]), (sv, host[8])):
        assert np.array_equal(np.isnan(a), np.isnan(b))
        ok = np.isfinite(a)
        assert np.all(np.abs(a[ok] - b[ok]) <= 1e-12 * np.abs(a[ok]))
    # sigma in degrees of the stand-in's lon / lat: the pixel covariance through the 1e-3 deg / px geolocation
    assert 1e-6 < np.nanmedian(su) < 1e-3 and 1e-6 < np.nanmedian(sv) < 1e-3
    # outliers: replaced and rejected rows get NaN sigma, the others keep theirs
    out = sid.get_drift_PM(lon, lat, *ll, uncertainty=True, outliers=True, return_flags=True, **kw)
    assert len(out) == 10
    flags, su2 = out[7], out[8]
    changed = np.isin(flags, (1, 2, 3, -1))
    assert np.all(np.isnan(su2[changed]))
    keep = (flags == 0) | (flags == -2)
    assert su2[keep].tobytes() == su[keep].tobytes()
