"""Outlier repair: the secondary peaks of every row's winning map (SID_PEAKS) and the normalised median test with
replacement (sid_filter_outliers, pmlib.filter_outliers, pattern_matching(outliers=True)).

The NumPy restatements below are the exact definitions of include/sid_b200.h: ``secondary_peaks`` on a raw winning map
(the oracle's ``rotate_and_match(...)[5]`` or what ``sid_run_maps`` returns) with the oracle's ``get_hessian``, and
``median_test`` on a table and its peaks.  The GPU must match both bit for bit.  The CPU probes run the restatements
on the exact oracle's tables and pin what the default eps / threshold do on a decoy scene and on clean scenes."""
import functools

import numpy as np
import pytest

from sea_ice_drift_b200 import _lib, pmlib
from sea_ice_drift_b200 import synthetic as syn
from oracle import c_oracle as co
from tests import test_degenerate_content as dg
from tests import test_gpu_maps as gm

N_PEAKS = 3


# ---------------------------------------------------------------------------------------------------- restatements
def peak_mask(m):
    """Peaks of a map: every in-map 8-neighbour with a lower flat index is strictly smaller, every one with a higher
    flat index is not larger (a plateau counts once, at its first index: np.argmax's rule)."""
    m = np.asarray(m, dtype=np.float32)
    rows, cols = m.shape
    pad = np.full((rows + 2, cols + 2), -np.inf, np.float32)
    pad[1:-1, 1:-1] = m
    ok = np.ones(m.shape, bool)
    for di in (-1, 0, 1):
        for dj in (-1, 0, 1):
            if di == 0 and dj == 0:
                continue
            q = pad[1 + di:1 + di + rows, 1 + dj:1 + dj + cols]
            ok &= (q < m) if (di < 0 or (di == 0 and dj < 0)) else (q <= m)
    return ok


def peak_ranks(m):
    """Flat indices of the secondary peaks in rank order: value descending, flat index ascending."""
    m = np.asarray(m, dtype=np.float32)
    mask = peak_mask(m).ravel()
    mask[int(np.argmax(m))] = False
    idx = np.flatnonzero(mask)
    vals = m.ravel()[idx]
    return idx[np.lexsort((idx, -vals.astype(np.float64)))]


def std32(v):
    """np.std of a float32 map as the library (and the oracle) compute it: float32 mean / deviations / squares,
    sequential sums in double."""
    v = np.asarray(v, dtype=np.float32).ravel()
    mean = np.float32(np.add.accumulate(v.astype(np.float64))[-1] / v.size)
    d = (v - mean).astype(np.float32)
    q = np.add.accumulate((d * d).astype(np.float32).astype(np.float64))[-1]
    return np.float32(np.sqrt(np.float32(q / v.size)))


def median32(v):
    v = np.sort(np.asarray(v, dtype=np.float32).ravel())
    n = v.size
    return v[n // 2] if n & 1 else np.float32(np.float32(v[n // 2 - 1] + v[n // 2]) * np.float32(0.5))


def parabola(a, b, c):
    p, q = np.float64(b) - np.float64(a), np.float64(b) - np.float64(c)
    return (p - q) / (2.0 * (p + q))


def secondary_peaks(ccm, s, c2fg, r2fg, H, W, hes_norm=True, hes_smth=False, mcc_norm=False, subpixel=False):
    """(N_PEAKS, 4) records c2, r2, r, h of a raw winning map, NaN where missing (include/sid_b200.h, SID_PEAKS)."""
    m = np.asarray(ccm, dtype=np.float32)
    rows, cols = m.shape
    out = np.full((N_PEAKS, 4), np.nan)
    ranks = peak_ranks(m)[:N_PEAKS]
    if ranks.size == 0:
        return out
    hes = co.get_hessian(m, hes_norm, hes_smth)
    for k, p in enumerate(ranks):
        i, j = divmod(int(p), cols)
        c2 = c2fg + (j - (W - s) / 2.0)
        r2 = r2fg + (i - (H - s) / 2.0)
        if subpixel:
            if 0 < j < cols - 1:
                c2 = c2 + parabola(m[i, j - 1], m[i, j], m[i, j + 1])
            if 0 < i < rows - 1:
                r2 = r2 + parabola(m[i - 1, j], m[i, j], m[i + 1, j])
        r = m[i, j]
        if mcc_norm:
            r = np.float32(np.float32(r - median32(m)) / std32(m))
        out[k] = (c2, r2, np.float64(r), np.float64(hes[i, j]))
    return out


def _median(v):
    v = sorted(v)
    k = len(v)
    return v[k // 2] if k & 1 else (v[k // 2 - 1] + v[k // 2]) * 0.5


def median_test(table, peaks, gpi, c2pm1, r2pm1, eps=1.0, threshold=2.0):
    """The rule of sid_filter_outliers, by definition (one Python loop per row).  ``gpi``: 2-D boolean grid."""
    gpi = np.asarray(gpi, dtype=bool)
    rows, cols = gpi.shape
    idx = np.flatnonzero(gpi)
    inv = np.full(gpi.size, -1)
    inv[idx] = np.arange(idx.size)
    c2pm1, r2pm1 = np.asarray(c2pm1, np.float64).ravel(), np.asarray(r2pm1, np.float64).ravel()
    out = np.array(table, dtype=np.float64, copy=True).reshape(-1, 5)
    flags = np.zeros(idx.size, np.int32)
    thr2 = threshold * threshold

    def disp(c2, r2, g):
        return c2 - np.round(c2pm1[g]), r2 - np.round(r2pm1[g])

    def outlier(d, m, rm):
        ex = abs(d[0] - m[0]) / (rm[0] + eps)
        ey = abs(d[1] - m[1]) / (rm[1] + eps)
        return ex * ex + ey * ey > thr2

    for k, g in enumerate(idx):
        row = table[k]
        if not np.isfinite(row[0]):
            flags[k] = -3
            continue
        gr, gc = divmod(int(g), cols)
        nb = []
        for di in (-1, 0, 1):
            for dj in (-1, 0, 1):
                y, x = gr + di, gc + dj
                if (di or dj) and 0 <= y < rows and 0 <= x < cols and inv[y * cols + x] >= 0:
                    q = inv[y * cols + x]
                    if np.isfinite(table[q, 0]):
                        nb.append(disp(table[q, 0], table[q, 1], y * cols + x))
        if len(nb) < 3:
            flags[k] = -2
            continue
        m = [_median([d[a] for d in nb]) for a in (0, 1)]
        rm = [_median([abs(d[a] - m[a]) for d in nb]) for a in (0, 1)]
        if not outlier(disp(row[0], row[1], g), m, rm):
            continue
        flags[k] = -1
        for rank in range(N_PEAKS):
            pk = peaks[k, rank]
            if np.isfinite(pk[0]) and not outlier(disp(pk[0], pk[1], g), m, rm):
                out[k, [0, 1, 3, 4]] = pk
                flags[k] = rank + 1
                break
        if flags[k] == -1:
            out[k] = np.nan
    return out, flags


# ---------------------------------------------------------------------------------------------------- CPU: closed forms
def test_peak_rule_plateau_border_ties_flat():
    m = np.zeros((5, 7), np.float32)
    m[2, 3] = 0.9                                      # primary
    m[0, 0] = 0.5                                      # corner peak
    m[4, 5] = m[4, 6] = 0.7                            # plateau on the bottom border: first index only
    m[1, 5] = 0.6
    m[1, 6] = 0.6                                      # horizontal tie: (1, 5) counts, (1, 6) does not
    assert list(peak_ranks(m)) == [4 * 7 + 5, 1 * 7 + 5, 0]
    rec = secondary_peaks(m, 3, 100.0, 50.0, 7, 9)
    assert rec[0, 0] == 100.0 + 5 - 3 and rec[0, 1] == 50.0 + 4 - 2 and rec[0, 2] == np.float32(0.7)
    assert rec[2, 0] == 100.0 - 3 and rec[2, 1] == 50.0 - 2
    # flat map: the primary is index 0 and nothing else is a peak
    assert peak_ranks(np.ones((6, 6), np.float32)).size == 0
    assert np.isnan(secondary_peaks(np.ones((6, 6), np.float32), 3, 0.0, 0.0, 8, 8)).all()
    # fewer than three: NaN records behind the ones that exist
    m2 = np.zeros((4, 4), np.float32)
    m2[0, 0], m2[3, 3] = 1.0, 0.5
    rec2 = secondary_peaks(m2, 3, 0.0, 0.0, 6, 6)
    assert np.isfinite(rec2[0]).all() and np.isnan(rec2[1:]).all()
    # exact ties between separate peaks: lower flat index first
    m3 = np.zeros((5, 5), np.float32)
    m3[0, 0] = 2.0
    m3[4, 0] = m3[2, 4] = m3[0, 4] = 1.0
    assert list(peak_ranks(m3)) == [4, 14, 20]


def test_peak_rule_is_argmax_rule_and_primary_is_a_peak():
    rng = np.random.default_rng(3)
    for _ in range(50):
        m = np.round(rng.normal(size=(rng.integers(2, 9), rng.integers(2, 9))), 1).astype(np.float32)
        assert peak_mask(m).ravel()[int(np.argmax(m))]
        for p in np.flatnonzero(peak_mask(m)):
            i, j = divmod(int(p), m.shape[1])
            blk = m[max(i - 1, 0):i + 2, max(j - 1, 0):j + 2]
            assert m[i, j] == blk.max()


def _brute_median_test(table, gpi, c2pm1, r2pm1, eps, threshold):
    """Independent definition with NumPy medians, decisions only (flags 0 / -2 / -3 / outlier)."""
    rows, cols = gpi.shape
    grid_c = np.full(gpi.shape, np.nan)
    grid_r = np.full(gpi.shape, np.nan)
    grid_c[gpi] = table[:, 0] - np.round(c2pm1.reshape(gpi.shape)[gpi])
    grid_r[gpi] = table[:, 1] - np.round(r2pm1.reshape(gpi.shape)[gpi])
    res = []
    for (y, x) in zip(*np.nonzero(gpi)):
        if not np.isfinite(grid_c[y, x]):
            res.append(-3)
            continue
        nc = grid_c[max(y - 1, 0):y + 2, max(x - 1, 0):x + 2].copy()
        nr = grid_r[max(y - 1, 0):y + 2, max(x - 1, 0):x + 2].copy()
        cy, cx = min(y, 1), min(x, 1)
        nc[cy, cx] = nr[cy, cx] = np.nan
        ok = np.isfinite(nc)
        if ok.sum() < 3:
            res.append(-2)
            continue
        mc, mr = np.median(nc[ok]), np.median(nr[ok])
        rc, rr = np.median(np.abs(nc[ok] - mc)), np.median(np.abs(nr[ok] - mr))
        e = (abs(grid_c[y, x] - mc) / (rc + eps)) ** 2 + (abs(grid_r[y, x] - mr) / (rr + eps)) ** 2
        res.append(9 if e > threshold ** 2 else 0)
    return np.array(res)


def random_field(seed, rows=9, cols=11, holes=0.15, outliers=0.15):
    """A grid field with NaN holes, points outside gpi, outliers and random secondary peaks."""
    rng = np.random.default_rng(seed)
    gpi = rng.random((rows, cols)) > 0.1
    c2pm1 = rng.uniform(0, 1000, rows * cols)
    r2pm1 = rng.uniform(0, 1000, rows * cols)
    # exact half-integers: rint rounds them to even (np.round), not away from zero
    half = rng.random(rows * cols) < 0.3
    c2pm1[half] = np.floor(c2pm1[half]) + 0.5
    r2pm1[half[::-1]] = np.floor(r2pm1[half[::-1]]) + 0.5
    n = int(gpi.sum())
    g = np.flatnonzero(gpi)
    table = np.empty((n, 5))
    table[:, 0] = np.round(c2pm1[g]) + 3.0 + rng.normal(0, 0.4, n)
    table[:, 1] = np.round(r2pm1[g]) - 2.0 + rng.normal(0, 0.4, n)
    table[:, 2] = rng.choice([-3.0, 0.0, 3.0], n)
    table[:, 3:] = rng.uniform(0, 1, (n, 2))
    bad = rng.random(n) < outliers
    table[bad, 0] += rng.uniform(5, 30, bad.sum()) * rng.choice([-1, 1], bad.sum())
    table[rng.random(n) < holes] = np.nan
    peaks = np.full((n, N_PEAKS, 4), np.nan)
    for k in range(n):
        cnt = rng.integers(0, N_PEAKS + 1)
        for r in range(cnt):
            good = rng.random() < 0.5
            dx = rng.normal(0, 0.4) if good else rng.uniform(-20, 20)
            peaks[k, r] = (np.round(c2pm1[g[k]]) + 3.0 + dx, np.round(r2pm1[g[k]]) - 2.0 + rng.normal(0, 0.4),
                           rng.uniform(0, 1), rng.uniform(0, 1))
    return table, peaks, gpi, c2pm1, r2pm1


@pytest.mark.parametrize("seed", range(6))
def test_median_test_against_brute_force(seed):
    table, peaks, gpi, c2pm1, r2pm1 = random_field(seed, holes=0.1 + 0.1 * seed)
    out, flags = median_test(table, peaks, gpi, c2pm1, r2pm1)
    brute = _brute_median_test(table, gpi, c2pm1, r2pm1, 1.0, 2.0)
    assert np.array_equal(flags == 0, brute == 0) and np.array_equal(flags == -2, brute == -2)
    assert np.array_equal(flags == -3, brute == -3) and np.array_equal(flags > 0, (brute == 9) & (flags > 0))
    assert ((flags == -1) | (flags > 0)).sum() == (brute == 9).sum() > 0
    assert (flags == -2).any() and (flags > 0).any() and (flags == -1).any()
    assert np.array_equal(out[flags == 0], table[flags == 0])
    assert np.isnan(out[flags == -1]).all() and np.isnan(out[flags == -3]).all()
    for k in np.flatnonzero(flags > 0):
        assert np.array_equal(out[k, [0, 1, 3, 4]], peaks[k, flags[k] - 1]) and out[k, 2] == table[k, 2]
    assert set(np.unique(flags)) <= {-3, -2, -1, 0, 1, 2, 3}


def test_median_test_edges_and_corners():
    """A full 3 x 3 grid of equal displacements: corners have 3 neighbours, edges 5, the centre 8; a 2 x 1 grid has
    fewer than 3 everywhere; with eps 1.0 a vector one pixel off on both axes is kept (e^2 = 2 <= 4)."""
    gpi = np.ones((3, 3), bool)
    c2pm1 = np.arange(9, dtype=np.float64) * 100
    r2pm1 = np.arange(9, dtype=np.float64) * 50
    table = np.column_stack([c2pm1 + 2, r2pm1 - 1, np.zeros(9), np.ones(9), np.ones(9)])
    table[4, :2] += 1.0
    out, flags = median_test(table, np.full((9, 3, 4), np.nan), gpi, c2pm1, r2pm1)
    assert (flags == 0).all() and np.array_equal(out, table)
    table[4, 0] += 1.0                                     # 2 px and 1 px: e^2 = 5 > 4
    out, flags = median_test(table, np.full((9, 3, 4), np.nan), gpi, c2pm1, r2pm1)
    assert flags[4] == -1 and np.isnan(out[4]).all() and (np.delete(flags, 4) == 0).all()
    out, flags = median_test(table[:2], np.full((2, 3, 4), np.nan), np.ones((2, 1), bool), c2pm1[:2], r2pm1[:2])
    assert (flags == -2).all()


# ---------------------------------------------------------------------------------------------------- CPU: probes
PROBE_SIDE, PROBE_STEP, PROBE_S, PROBE_BORDER = 760, 100, 35, 40


@functools.lru_cache(maxsize=None)
def probe_scene(rotation=2.0, seed=5):
    img1 = syn.speckle_image((PROBE_SIDE, PROBE_SIDE), seed)
    m = syn.shift_matrix(4.0, -3.0)
    rot = syn.rotation_matrix(img1.shape, rotation)
    full = np.vstack([rot, [0, 0, 1]]) @ np.vstack([m, [0, 0, 1]])
    m = full[:2]
    img2 = syn.warp_pair(img1, m, seed)
    inset = 130
    xs = np.arange(inset, PROBE_SIDE - inset + 1, PROBE_STEP, dtype=np.float64)
    gx, gy = np.meshgrid(xs, xs)
    tx, ty = syn.apply_affine(m, gx.ravel(), gy.ravel())
    return img1, img2, m, gx.shape, gx.ravel(), gy.ravel(), np.round(tx), np.round(ty), tx, ty


def oracle_rows(img1, img2, c1, r1, c2, r2, subpixel=False):
    """Table rows and secondary peaks from the exact oracle's rotate_and_match and the restatement."""
    s, b = PROBE_S, PROBE_BORDER
    table = np.full((c1.size, 5), np.nan)
    peaks = np.full((c1.size, N_PEAKS, 4), np.nan)
    for k in range(c1.size):
        win = gm.window(img2, s, c2[k], r2[k], b)
        res = co.rotate_and_match(img1, c1[k], r1[k], s, win, 0.0, angles=[-3, 0, 3])
        if not np.isfinite(res[0]):
            continue
        H, W = win.shape
        m = res[5]
        c, r = c2[k] + res[0], r2[k] + res[1]
        if subpixel:
            i, j = divmod(int(np.argmax(m)), m.shape[1])
            if 0 < j < m.shape[1] - 1:
                c = c + parabola(m[i, j - 1], m[i, j], m[i, j + 1])
            if 0 < i < m.shape[0] - 1:
                r = r + parabola(m[i - 1, j], m[i, j], m[i + 1, j])
        table[k] = (c, r, res[2], res[3], res[4])
        peaks[k] = secondary_peaks(m, s, c2[k], r2[k], H, W, subpixel=subpixel)
    return table, peaks


@functools.lru_cache(maxsize=None)
def decoy_probe():
    img1, img2, m, shape, c1, r1, c2, r2, tx, ty = probe_scene()
    s, hws = PROBE_S, PROBE_S // 2
    img2 = img2.copy()
    decoys = np.arange(c1.size) % 5 == 2
    for k in np.flatnonzero(decoys):
        win = gm.window(img2, s, c2[k], r2[k], PROBE_BORDER)
        tpl = co.rotate_and_match(img1, c1[k], r1[k], s, win, 0.0, angles=[-3, 0, 3])[6]
        # an exact copy of the winning template, s + 3 px right of (or left of) the true position
        sign = 1 if k % 2 else -1
        x0 = int(c2[k]) - hws + sign * (s + 3)
        y0 = int(r2[k]) - hws
        img2[y0:y0 + s, x0:x0 + s] = tpl
    table, peaks = oracle_rows(img1, img2, c1, r1, c2, r2)
    out, flags = median_test(table, peaks, np.ones(shape, bool), c2, r2)
    return table, peaks, out, flags, decoys, tx, ty


def test_decoy_probe():
    """Every fifth point of a speckle pair (shift (4, -3) and a 2 degree rotation, grid 100 px apart, s = 35, border 40,
    true first guess) gets an exact copy of its winning template one template width from the truth.  The decoy wins
    (r = 1) and the truth becomes a secondary peak: every decoy row is flagged and repaired to within 1 px of the truth
    (after the -1 px template bias), and no other row changes."""
    table, peaks, out, flags, decoys, tx, ty = decoy_probe()
    assert (table[decoys, 3] == 1.0).all()
    assert (flags[decoys] != 0).all()
    err = np.hypot(out[decoys, 0] - (tx[decoys] - 1), out[decoys, 1] - (ty[decoys] - 1))
    assert (flags[decoys] >= 1).mean() >= 0.95 and (err[flags[decoys] >= 1] <= 1.0).mean() >= 0.95
    changed = ~np.all((out == table) | (np.isnan(out) & np.isnan(table)), axis=1)
    assert changed[~decoys].mean() <= 0.01
    assert int(decoys.sum()) == 7 and int(changed[decoys].sum()) == 7 and int(changed[~decoys].sum()) == 0


@pytest.mark.parametrize("subpixel", (False, True))
def test_clean_probe(subpixel):
    """The same scene without decoys: at most 0.5 % of the valid rows change, and no row within 1 px of the truth is
    rejected."""
    img1, img2, m, shape, c1, r1, c2, r2, tx, ty = probe_scene()
    table, peaks = oracle_rows(img1, img2, c1, r1, c2, r2, subpixel)
    out, flags = median_test(table, peaks, np.ones(shape, bool), c2, r2)
    valid = np.isfinite(table[:, 0])
    assert valid.sum() == 36
    changed = ~np.all((out == table) | (np.isnan(out) & np.isnan(table)), axis=1)
    assert changed[valid].mean() <= 0.005
    near = np.hypot(table[:, 0] - (tx - 1), table[:, 1] - (ty - 1)) <= 1.0
    assert not (near & (flags == -1)).any()


# ---------------------------------------------------------------------------------------------------- CPU: plumbing
def test_value_errors_before_device_work():
    img = np.ones((64, 64), np.uint8)
    matcher = lambda im, tp, m: pmlib.match_template(im, tp, m)
    with pytest.raises(ValueError):
        pmlib.use_mcc_batch([30.], [30.], [30.], [30.], [5.], img, img, 9, 0.0, peaks=True, template_matcher=matcher)
    n = syn.ArrayDomain(img)
    lon, lat = n.transform_points(np.array([[30.0]]), np.array([[30.0]]))
    with pytest.raises(ValueError):
        pmlib.pattern_matching(lon, lat, n, [10.], [10.], n, [10.], [10.], outliers=True, template_matcher=matcher)
    with pytest.raises(ValueError):
        pmlib.pattern_matching(lon, lat, n, [10.], [10.], n, [10.], [10.], return_flags=True)


def test_outliers_refused_under_a_process_group(monkeypatch):
    from sea_ice_drift_b200 import sharding
    monkeypatch.setattr(sharding, "_dist", lambda: object())
    img = np.ones((64, 64), np.uint8)
    n = syn.ArrayDomain(img)
    lon, lat = n.transform_points(np.array([[30.0]]), np.array([[30.0]]))
    with pytest.raises(ValueError):
        pmlib.pattern_matching(lon, lat, n, [10.], [10.], n, [10.], [10.], outliers=True)


def test_abi_names():
    assert _lib.SID_PEAKS == 32 and _lib.SID_N_PEAKS == N_PEAKS
    assert {"sid_get_peaks", "sid_filter_outliers"} <= set(_lib.EXPORTS)


# ---------------------------------------------------------------------------------------------------- GPU
def _peaks_equal(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(np.nan_to_num(a, nan=0.0).view(np.uint64), np.nan_to_num(b, nan=0.0).view(np.uint64))


def check_peaks(ctx, img1, img2, pts, s, angles, o, flags_extra=0, kernel=None, oracle=True):
    """Table / status / maps with SID_PEAKS are those without; the peaks equal the restatement on run_maps' maps and
    (valid rows) on the oracle's maps.  Returns (table, status, peaks)."""
    ctx.set_pair(img1, img2)
    flags = gm.flags_of(o) | flags_extra
    ref, st_ref = ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags, want_status=True)
    launches = ctx.launch_count
    tab, st = ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags | _lib.SID_PEAKS, want_status=True)
    launches_peaks = ctx.launch_count - launches
    launches = ctx.launch_count
    ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags, want_status=True)
    assert launches_peaks == ctx.launch_count - launches
    if kernel is not None:
        assert ctx.last_kernel_name == kernel, ctx.last_kernel_name
    assert tab.tobytes() == ref.tobytes() and np.array_equal(st, st_ref)
    n = pts[0].size
    # the previous call did not set the flag
    with pytest.raises(ValueError):
        ctx.peaks(n)
    tab, st = ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags | _lib.SID_PEAKS, want_status=True)
    peaks = ctx.peaks(n)
    with pytest.raises(ValueError):
        ctx.peaks(n + 1)
    tab_m, maps, tpls, st_m = ctx.run_maps(*pts, s, angles, 0.0, o["rot_order"], flags | _lib.SID_PEAKS, want_status=True)
    assert _peaks_equal(ctx.peaks(n), peaks)
    _, maps_ref, _ = ctx.run_maps(*pts, s, angles, 0.0, o["rot_order"], flags)
    assert tab_m.tobytes() == ref.tobytes() and np.array_equal(st_m, st_ref)
    sub = bool(flags & _lib.SID_SUBPIXEL)
    kw = dict(hes_norm=o["hes_norm"], hes_smth=o["hes_smth"], mcc_norm=o["mcc_norm"], subpixel=sub)
    c1, r1, c2, r2, b = pts
    found = 0
    for i in range(n):
        if st[i] not in (_lib.SID_PT_VALID, _lib.SID_PT_MASKED):
            assert np.isnan(peaks[i]).all() and maps[i] is None
            continue
        assert maps[i].tobytes() == maps_ref[i].tobytes()
        H, W = gm.window(img2, s, c2[i], r2[i], b[i]).shape
        want = secondary_peaks(maps[i], s, c2[i], r2[i], H, W, **kw)
        assert _peaks_equal(peaks[i], want), (i, peaks[i], want)
        if oracle and st[i] == _lib.SID_PT_VALID:
            res = co.rotate_and_match(img1, c1[i], r1[i], s, gm.window(img2, s, c2[i], r2[i], b[i]), 0.0, angles=angles, **o)
            assert _peaks_equal(secondary_peaks(res[5], s, c2[i], r2[i], H, W, **kw), want)
        found += int(np.isfinite(peaks[i, 0, 0]))
    assert found > 0
    return tab, st, peaks


PEAK_CASES = gm.CASES + [(f, "subpixel") for f in gm.FAMILIES if f[0] in ("ws", "tc_fused", "imma_fused_global", "tc_split")]


@pytest.mark.gpu
@pytest.mark.parametrize("family,flag_set", PEAK_CASES, ids=["%s-%s" % (f[0], fs) for f, fs in PEAK_CASES])
def test_peaks_equal_restatement(gpu_ctx, monkeypatch, family, flag_set):
    name, s, angles, (lo, hi), env, kernel = family
    gm._setenv(monkeypatch, env)
    img1, img2 = gm.speckle_pair()
    pts = gm.speckle_points(s, lo, hi)
    extra = _lib.SID_SUBPIXEL if flag_set == "subpixel" else 0
    o = gm.opts_of("default" if flag_set == "subpixel" else flag_set)
    check_peaks(gpu_ctx, img1, img2, pts, s, angles, o, extra, kernel)


@pytest.mark.gpu
@pytest.mark.parametrize("family", [f for f in gm.FAMILIES if f[0] in ("ws", "tc_fused", "imma_split")],
                         ids=lambda f: f[0])
def test_peaks_of_masked_rows(gpu_ctx, monkeypatch, family):
    """SID_MASKED rows (status 2) get peaks from their masked maps; the main kernels' rows keep theirs."""
    name, s, angles, (lo, hi), env, kernel = family
    gm._setenv(monkeypatch, env)
    img1, img2 = gm.speckle_pair()
    img1 = img1.copy()
    img1[200:260, 60:120] = 0                                  # land: templates crossing it are masked rows
    pts = gm.speckle_points(s, lo, hi)
    tab, st, peaks = check_peaks(gpu_ctx, img1, img2, pts, s, angles, gm.opts_of("default"), _lib.SID_MASKED, kernel)
    assert (st == _lib.SID_PT_MASKED).sum() >= 2
    assert np.isfinite(peaks[st == _lib.SID_PT_MASKED, 0, 0]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("plateaus", "periodic"))
def test_peaks_on_degenerate_content(gpu_ctx, kind):
    img1, img2 = dg.images(kind)
    n = dg.n_points(kind)
    pts = dg.points(kind, 35, (16 + np.arange(n) % 5).astype(np.float64))
    tab, st, peaks = check_peaks(gpu_ctx, img1, img2, pts, 35, gm.ANGLES, gm.opts_of("default"))
    if kind == "plateaus":
        assert np.isnan(peaks[st == 1]).all(axis=(1, 2)).any()      # flat templates: no secondary peaks


@pytest.mark.gpu
def test_peaks_identical_across_entry_points(gpu_ctx, monkeypatch):
    """sid_run, sid_run_pair (3 bands, two border classes), sid_run_device (two classes, with and without status)."""
    import torch
    img1, img2 = gm.speckle_pair()
    c1, r1, c2, r2, _ = gm.speckle_points(35, 20, 50, n_grid=23)
    k = np.arange(c1.size)
    brd = np.where(k % 4 == 3, 21 + k % 30, 20).astype(np.float64)
    brd[-8:] = 20.0
    pts = [c1, r1, c2, r2, brd]
    n = c1.size
    flags = _lib.SID_HES_NORM | _lib.SID_PEAKS
    gpu_ctx.set_pair(img1, img2)
    tab, st = gpu_ctx.run(*pts, 35, gm.ANGLES, 0.0, 0, flags, want_status=True)
    assert gpu_ctx.last_kernel_name.endswith(" + sid::pm_ws_kernel"), gpu_ctx.last_kernel_name
    ref = gpu_ctx.peaks(n)
    monkeypatch.setenv("SID_BANDS", "3")
    tab2 = gpu_ctx.run_pair(img1, img2, *pts, 35, gm.ANGLES, 0.0, 0, flags)
    assert tab2.tobytes() == tab.tobytes() and _peaks_equal(gpu_ctx.peaks(n), ref)
    dev = [torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda") for a in pts]
    for with_status in (True, False):
        d_out = torch.empty((n, 5), dtype=torch.float64, device="cuda")
        d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        gpu_ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        gpu_ctx.run_device(n, *[t.data_ptr() for t in dev], 50, 35, gm.ANGLES, 0.0, d_out.data_ptr(),
                           d_st.data_ptr() if with_status else 0, 0, flags)
        gpu_ctx.synchronize()
        assert d_out.cpu().numpy().tobytes() == tab.tobytes()
        assert _peaks_equal(gpu_ctx.peaks(n), ref)
        gpu_ctx.set_stream(None)
    # secondary peaks sit in the windows of the valid rows
    ok = st == 1
    assert np.isfinite(ref[ok, 0, 0]).mean() > 0.9


@pytest.mark.gpu
def test_refusals(gpu_ctx):
    img1, img2 = gm.speckle_pair()
    pts = gm.speckle_points(35, 16, 20)
    n = pts[0].size
    gpu_ctx.set_pair(img1, img2)
    gpu_ctx.run(*pts, 35, gm.ANGLES, 0.0, 0, _lib.SID_HES_NORM, keep_on_device=True)
    gpi = np.ones((1, n), bool)
    with pytest.raises(ValueError):
        gpu_ctx.peaks(n)
    with pytest.raises(ValueError):
        gpu_ctx.filter_outliers((1, n), gpi, pts[2], pts[3], in_place=True)
    with pytest.raises(ValueError):
        gpu_ctx.rotate_and_match(img1, 100.0, 100.0, 35, gm.window(img2, 35, 100.0, 100.0, 16), gm.ANGLES, 0.0,
                                 flags=_lib.SID_HES_NORM | _lib.SID_PEAKS)
    # peaks of a sid_run_device call do not go with the table an earlier sid_run left on the device
    import torch
    dev = [torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda") for a in pts]
    d_out = torch.empty((n, 5), dtype=torch.float64, device="cuda")
    gpu_ctx.run(*pts, 35, gm.ANGLES, 0.0, 0, _lib.SID_HES_NORM | _lib.SID_PEAKS, keep_on_device=True)
    gpu_ctx.run_device(n, *[t.data_ptr() for t in dev], 20, 35, gm.ANGLES, 0.0, d_out.data_ptr(), 0, 0,
                       _lib.SID_HES_NORM | _lib.SID_PEAKS)
    gpu_ctx.synchronize()
    assert gpu_ctx.peaks(n).shape == (n, N_PEAKS, 4)
    with pytest.raises(ValueError):
        gpu_ctx.filter_outliers((1, n), gpi, pts[2], pts[3], in_place=True)
    # the context stays usable
    tab = gpu_ctx.run(*pts, 35, gm.ANGLES, 0.0, 0, _lib.SID_HES_NORM | _lib.SID_PEAKS)
    assert gpu_ctx.peaks(n).shape == (n, N_PEAKS, 4) and np.isfinite(tab[:, 0]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_filter_equals_restatement_host_inputs(gpu_ctx, seed):
    table, peaks, gpi, c2pm1, r2pm1 = random_field(seed + 100, rows=23, cols=31, holes=0.05 + 0.1 * seed)
    halves = np.flatnonzero(np.mod(c2pm1, 1.0) == 0.5)
    assert halves.size > 50 and (np.mod(np.round(c2pm1[halves]), 2.0) == 0).all()
    assert (np.round(c2pm1[halves]) != np.floor(c2pm1[halves] + 0.5)).any()      # ties that half-up would round otherwise
    for eps, thr in ((1.0, 2.0), (0.1, 3.0)):
        want, wflags = median_test(table, peaks, gpi, c2pm1, r2pm1, eps, thr)
        got, flags = pmlib.filter_outliers(table, peaks, gpi, c2pm1, r2pm1, eps, thr)
        assert np.array_equal(flags, wflags)
        assert np.array_equal(got, want, equal_nan=True) and np.array_equal(np.isnan(got), np.isnan(want))
        assert np.array_equal(np.nan_to_num(got).view(np.uint64), np.nan_to_num(want).view(np.uint64))


@pytest.mark.gpu
def test_filter_device_resident_in_place(gpu_ctx):
    """The table and peaks a run left on the device, filtered in place, then read by the epilogue."""
    img1, img2, m, shape, c1, r1, c2, r2, tx, ty = probe_scene()
    img2 = img2.copy()
    img2[300:340, 300:340] = img2[100:140, 100:140]               # disturb a few windows
    b = np.full(c1.size, float(PROBE_BORDER))
    gpi = np.ones(shape, bool)
    gpu_ctx.set_pair(img1, img2)
    table = gpu_ctx.run(c1, r1, c2, r2, b, PROBE_S, [-3, 0, 3], 0.0, 0, _lib.SID_HES_NORM | _lib.SID_PEAKS)
    peaks = gpu_ctx.peaks(c1.size)
    want, wflags = median_test(table, peaks, gpi, c2, r2)
    got, flags = gpu_ctx.filter_outliers(shape, gpi, c2, r2)                 # device inputs, host output
    assert np.array_equal(flags, wflags) and np.array_equal(got, want, equal_nan=True)
    got2, flags2 = gpu_ctx.filter_outliers(shape, gpi, c2, r2, in_place=True)
    assert got2 is None and np.array_equal(flags2, wflags)
    xy = ll = np.array([1.0, 0.0, 0.0, 0.0, 1.0, 0.0])
    grids = gpu_ctx.pm_epilogue_affine(gpi, c2, r2, xy, ll)
    grids_host = gpu_ctx.pm_epilogue_affine(gpi, c2, r2, xy, ll, results=want)
    assert grids.tobytes() == grids_host.tobytes()


@pytest.mark.gpu
def test_pattern_matching_outliers_device_equals_host(gpu_ctx):
    from tests.test_subpixel import _drop_in_scene
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = _drop_in_scene(side=1600, grid=30)
    kw = dict(angles=[-3, 0, 3], img_size=35)
    plain = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, **kw)
    dev = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, outliers=True, **kw)
    host = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, outliers=True, device_epilogue=False, **kw)
    for a, b in zip(dev, host):
        assert a.tobytes() == b.tobytes()
    # a clean scene: almost nothing changes
    changed = ~((dev[0] == plain[0]) | (np.isnan(dev[0]) & np.isnan(plain[0])))
    assert changed.mean() <= 0.01
    # without the keyword: the parent's bytes
    again = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, **kw)
    for a, b in zip(again, plain):
        assert a.tobytes() == b.tobytes()
    # outlier_eps / outlier_threshold pass through, and both paths filter: a strict setting rejects and replaces rows
    strict_kw = dict(outliers=True, outlier_eps=0.01, outlier_threshold=0.5, **kw)
    strict = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, **strict_kw)
    strict_host = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, device_epilogue=False, **strict_kw)
    for a, b in zip(strict, strict_host):
        assert a.tobytes() == b.tobytes()
    assert np.isnan(strict[0]).sum() > np.isnan(dev[0]).sum() >= np.isnan(plain[0]).sum()
    # return_flags: the eighth grid explains every difference, on both paths
    for de in (True, False):
        res = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, return_flags=True, device_epilogue=de, **strict_kw)
        assert len(res) == 8 and res[7].shape == lon.shape and res[7].dtype == np.int32
        assert all(a.tobytes() == b.tobytes() for a, b in zip(res[:7], strict))
        fl = res[7]
        assert set(np.unique(fl)) <= {-4, -3, -2, -1, 0, 1, 2, 3} and np.isnan(plain[0][fl == -4]).all()
        assert np.isnan(res[0][fl == -1]).all() and (fl == -1).sum() == (np.isnan(res[0]) & np.isfinite(plain[0])).sum()
        assert np.array_equal(res[0][fl == 0], plain[0][fl == 0])
    # the angle of a row that is not rejected never changes
    kept = np.isfinite(strict[0])
    assert np.array_equal(strict[2][kept], plain[2][kept])


@pytest.mark.gpu
def test_use_mcc_batch_peaks(gpu_ctx):
    img1, img2 = gm.speckle_pair()
    c1, r1, c2, r2, b = gm.speckle_points(35, 16, 20)
    plain = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=gm.ANGLES)
    tab, peaks = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=gm.ANGLES, peaks=True)
    assert tab.tobytes() == plain.tobytes() and peaks.shape == (c1.size, N_PEAKS, 4)
    tab2, maps, tpls, peaks2 = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=gm.ANGLES,
                                                   peaks=True, return_maps=True)
    assert tab2.tobytes() == plain.tobytes() and _peaks_equal(peaks2, peaks)
