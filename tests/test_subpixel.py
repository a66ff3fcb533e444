"""Sub-pixel drift vectors (SID_SUBPIXEL, ``subpixel=True``): the parabola through the peak of the winning raw NCC map
and its two neighbours per axis, added on the device to the unrefined position.

The expected table is the exact oracle's unrefined row (rotate_and_match on the point's window) plus ``peak_offsets``
below, a NumPy float64 restatement of the device arithmetic, applied to the oracle's map for that point, bit for bit;
columns 2-4, the NaN rows and the status must be those of the call without the flag.  The CPU tests pin the estimator
(closed forms), its accuracy on the oracle's maps and the keyword plumbing; the others need a GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

from sea_ice_drift_b200 import _lib, pmlib
from sea_ice_drift_b200 import synthetic as syn
from oracle import c_oracle as co
from tests import test_degenerate_content as dg
from tests.test_gpu_maps import (ANGLES, CASES, DEGENERATE, FLAG_SETS, _setenv, flags_of, opts_of, speckle_pair,
                                 speckle_points, window)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def peak_offsets(ccm):
    """Sub-pixel offsets (dx, dy) of the peak of a raw NCC map (SID_SUBPIXEL, include/sid_b200.h), float64 in the
    kernels' operation order: per axis a, b, c = the lower neighbour, the peak (np.argmax's first maximum) and the
    higher neighbour, p = b - a, q = b - c, d = (p - q) / (2 (p + q)); +0.0 for a peak on the first or last column
    (row).  The refined position is (c2fg + dc) + dx, (r2fg + dr) + dy."""
    m = np.asarray(ccm, dtype=np.float32)
    bi, bj = np.unravel_index(int(np.argmax(m)), m.shape)

    def vertex(a, b, c):
        p, q = np.float64(b) - np.float64(a), np.float64(b) - np.float64(c)
        return (p - q) / (np.float64(2.0) * (p + q))

    dx = vertex(m[bi, bj - 1], m[bi, bj], m[bi, bj + 1]) if 0 < bj < m.shape[1] - 1 else np.float64(0.0)
    dy = vertex(m[bi - 1, bj], m[bi, bj], m[bi + 1, bj]) if 0 < bi < m.shape[0] - 1 else np.float64(0.0)
    return float(dx), float(dy)


def expected_table(img1, img2, pts, s, angles, o, plain, st, alpha0=0.0):
    """For every valid row of ``plain`` (a table computed without the flag) the exact oracle's unrefined row
    (c2fg + dc, r2fg + dr, angle of rotate_and_match on the point's window), checked against ``plain``, and the expected
    refined row: c2 / r2 plus peak_offsets of the oracle's map.  Returns (expected table, offsets); rows that are not
    valid keep ``plain``'s NaN and get NaN offsets."""
    exp = plain.copy()
    offs = np.full((plain.shape[0], 2), np.nan)
    c1, r1, c2, r2, b = pts
    for i in np.flatnonzero(st == 1):
        res = co.rotate_and_match(img1, c1[i], r1[i], s, window(img2, s, c2[i], r2[i], b[i]), alpha0, angles=angles, **o)
        c2u, r2u = c2[i] + res[0], r2[i] + res[1]
        assert (c2u, r2u, res[2]) == tuple(plain[i, :3]), i
        dx, dy = peak_offsets(res[5])
        exp[i, 0], exp[i, 1] = c2u + dx, r2u + dy
        offs[i] = dx, dy
    return exp, offs


def assert_refined(plain, st_plain, sub, st_sub, exp):
    """Columns 2-4, NaN rows and status as without the flag; c2 / r2 equal the expected table bit for bit."""
    assert np.array_equal(st_sub, st_plain)
    assert sub[:, 2:].tobytes() == plain[:, 2:].tobytes()
    assert np.array_equal(np.isnan(sub), np.isnan(plain))
    assert sub[:, :2].tobytes() == exp[:, :2].tobytes(), np.argwhere(sub[:, :2].view(np.uint64) != exp[:, :2].view(np.uint64))


# ---------------------------------------------------------------------------------------------------- CPU
def test_peak_offsets_recovers_parabola_vertex():
    rng = np.random.default_rng(3)
    for _ in range(200):
        x0, y0 = rng.uniform(-0.5, 0.5, 2)
        ax, ay, top = rng.uniform(0.05, 2.0), rng.uniform(0.05, 2.0), rng.uniform(0.5, 1.0)
        j = np.arange(-2, 3)
        # a separable paraboloid sampled on a 5 x 5 grid around its vertex (x0, y0); float32 like a real map
        m = (top - ax * (j[None, :] - x0) ** 2 - ay * (j[:, None] - y0) ** 2).astype(np.float64)
        if np.argmax(m) != 12:                    # the vertex must round to the centre sample
            continue
        dx, dy = peak_offsets(m.astype(np.float32))
        # exact in float64 arithmetic; the float32 samples bound the error
        assert abs(dx - x0) <= 1e-5 * (1 + 1 / ax) and abs(dy - y0) <= 1e-5 * (1 + 1 / ay)
        # float64 samples: the closed form itself
        a, b, c = m[2, 1], m[2, 2], m[2, 3]
        p, q = b - a, b - c
        assert abs((p - q) / (2 * (p + q)) - x0) <= 1e-12


def test_peak_offsets_bounded_ties_and_edges():
    rng = np.random.default_rng(4)
    for _ in range(2000):
        b = np.float32(rng.uniform(-1, 1))
        a = np.float32(b - np.float32(rng.uniform(1e-7, 2)))     # lower-index neighbour strictly smaller (first maximum)
        c = np.float32(b - np.float32(rng.uniform(0, 2)) * rng.integers(0, 2))
        m = np.array([[a - 1, a - 1, a - 1], [a, b, c], [a - 1, a - 1, a - 1]], np.float32)
        if m.argmax() != 4:
            continue
        dx, dy = peak_offsets(m)
        assert abs(dx) <= 0.5 and np.isfinite(dx) and np.isfinite(dy)
    # the higher-index neighbour ties the peak: exactly +0.5 on that axis
    assert peak_offsets(np.array([[0, 0, 0], [0.2, 0.9, 0.9], [0, 0, 0]], np.float32))[0] == 0.5
    assert peak_offsets(np.array([[0, 0.2, 0], [0, 0.9, 0], [0, 0.9, 0]], np.float32))[1] == 0.5
    # a flat map (flat template: all 1.0) peaks at index 0: the edge rule gives +0.0 on both axes
    dx, dy = peak_offsets(np.ones((4, 5), np.float32))
    assert (dx, dy) == (0.0, 0.0) and np.signbit(dx) == np.signbit(dy) == False
    # peaks on the last column / row
    m = np.zeros((3, 4), np.float32)
    m[1, 3] = 1
    assert peak_offsets(m)[0] == 0.0 and np.signbit(peak_offsets(m)[0]) == False
    m = np.zeros((3, 4), np.float32)
    m[2, 1] = 1
    assert peak_offsets(m)[1] == 0.0


def _accuracy(side, warp, angles, grid=12):
    """The method of the issue's CPU experiment on the exact oracle's maps: median 2-D error against the known drift
    (minus the reference's -1 px template-centre bias) of the integer and the refined positions."""
    img1 = syn.speckle_image((side, side), 0)
    m = syn.shift_matrix(*warp[1:]) if warp[0] == "shift" else syn.rotation_matrix((side, side), warp[1])
    img2 = syn.warp_pair(img1, m, 0)
    c1, r1, c2fg, r2fg, brd = syn.hot_loop_inputs(img1, m, grid, 35, 20, 0, subpixel=False)
    tx, ty = syn.apply_affine(m, c1, r1)
    e_int, e_ref = [], []
    for i in range(c1.size):
        res = co.rotate_and_match(img1, c1[i], r1[i], 35, window(img2, 35, c2fg[i], r2fg[i], brd[i]), 0.0, angles=angles)
        if np.isnan(res[0]):
            continue
        dx, dy = peak_offsets(res[5])
        ex, ey = c2fg[i] + res[0] - (tx[i] - 1), r2fg[i] + res[1] - (ty[i] - 1)
        e_int.append(np.hypot(ex, ey))
        e_ref.append(np.hypot(ex + dx, ey + dy))
    assert len(e_int) >= 0.9 * c1.size
    return float(np.median(e_int)), float(np.median(e_ref))


def test_accuracy_on_exact_oracle_shift():
    integer, refined = _accuracy(800, ("shift", 12.3, -7.6), [0])
    assert refined < 0.1 and refined < 0.25 * integer, (integer, refined)


def test_accuracy_on_exact_oracle_rotation():
    integer, refined = _accuracy(1200, ("rot", 2.0), [-3, 0, 3])
    assert refined < 0.15 and refined < integer, (integer, refined)


def test_flags_from_options_sets_subpixel_only_when_asked():
    assert _lib.flags_from_options({}) == _lib.SID_HES_NORM
    assert _lib.flags_from_options({"subpixel": False, "hes_smth": True}) == _lib.SID_HES_NORM | _lib.SID_HES_SMTH
    assert _lib.flags_from_options({"subpixel": True}) == _lib.SID_HES_NORM | _lib.SID_SUBPIXEL
    assert _lib.flags_from_options(dict(hes_norm=False, mcc_norm=True, subpixel=True)) == \
        _lib.SID_MCC_NORM | _lib.SID_SUBPIXEL
    assert _lib.flags_from_kwargs(True, False, False) == _lib.flags_from_options({})
    assert _lib.SID_SUBPIXEL == 8


def test_subpixel_with_user_matcher_is_refused_before_any_device_call():
    img = np.full((60, 60), 7, np.uint8)
    matcher = lambda im, tp, m: np.zeros((im.shape[0] - tp.shape[0] + 1, im.shape[1] - tp.shape[1] + 1), np.float32)
    with pytest.raises(ValueError, match="subpixel"):
        pmlib.rotate_and_match(img, 30.0, 30.0, 21, img[5:40, 5:40], 0.0, template_matcher=matcher, subpixel=True)
    with pytest.raises(ValueError, match="subpixel"):
        pmlib.use_mcc_batch([30.0], [30.0], [30.0], [30.0], [5.0], img, img, 21, 0.0, template_matcher=matcher,
                            subpixel=True)


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("family,flag_set", CASES, ids=["%s-%s" % (f[0], fs) for f, fs in CASES])
def test_every_kernel_family_equals_oracle_plus_offsets(gpu_ctx, monkeypatch, family, flag_set):
    name, s, angles, (lo, hi), env, kernel = family
    _setenv(monkeypatch, env)
    img1, img2 = speckle_pair()
    pts = speckle_points(s, lo, hi)
    o = opts_of(flag_set)
    gpu_ctx.set_pair(img1, img2)
    plain, st = gpu_ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags_of(o), want_status=True)
    ran = gpu_ctx.last_kernel_name
    if kernel is not None:
        assert ran == kernel, ran
    sub, st_sub = gpu_ctx.run(*pts, s, angles, 0.0, o["rot_order"], flags_of(o) | _lib.SID_SUBPIXEL, want_status=True)
    assert gpu_ctx.last_kernel_name == ran
    exp, offs = expected_table(img1, img2, pts, s, angles, o, plain, st)
    assert_refined(plain, st, sub, st_sub, exp)
    valid = st == 1
    assert (st == 0).sum() >= 1 and (st == -1).sum() == 2
    assert np.all(np.abs(offs[valid]) <= 0.5) and np.count_nonzero(offs[valid]) > valid.sum()


def _edge_points(s, border, shift=(7.0, -4.0)):
    """Integer drift, integer c1, first guesses offset by exactly +-border from the truth in one or both axes: the peak
    sits on the first or last column / row of the map."""
    side = 360
    img1 = syn.speckle_image((side, side), 5)
    img2 = syn.warp_pair(img1, syn.shift_matrix(*shift), 5, noise_sd=2.0)
    gx, gy = syn.grid_points((side, side), 4, 35 + 2 * border + 12)
    c1, r1 = np.round(gx), np.round(gy)
    tx, ty = syn.apply_affine(syn.shift_matrix(*shift), c1, r1)
    tc, tr = tx - 1, ty - 1                                 # where the peak is: the truth minus the -1 px template bias
    k = np.arange(c1.size)
    sx = np.array([-1, 1, 0, 0, -1, 1, 1, -1])[k % 8] * border
    sy = np.array([0, 0, -1, 1, -1, 1, -1, 1])[k % 8] * border
    return img1, img2, [c1, r1, tc + sx, tr + sy, np.full(c1.size, float(border))]


EDGE_FAMILIES = [f for f in DEGENERATE if f[0] in ("ws", "tc_fused", "imma_split", "imma_fused", "dp4a_s35_fused")]


@pytest.mark.gpu
@pytest.mark.parametrize("family", EDGE_FAMILIES, ids=[f[0] for f in EDGE_FAMILIES])
def test_peak_on_the_map_edge_keeps_the_unrefined_position(gpu_ctx, monkeypatch, family):
    name, s, angles, (lo, hi), env, kernel = family
    _setenv(monkeypatch, env)
    img1, img2, pts = _edge_points(s, hi)
    gpu_ctx.set_pair(img1, img2)
    plain, st = gpu_ctx.run(*pts, s, angles, 0.0, want_status=True)
    if kernel is not None:
        assert gpu_ctx.last_kernel_name == kernel
    sub, st_sub = gpu_ctx.run(*pts, s, angles, 0.0, flags=_lib.SID_HES_NORM | _lib.SID_SUBPIXEL, want_status=True)
    exp, offs = expected_table(img1, img2, pts, s, angles, opts_of("default"), plain, st)
    assert_refined(plain, st, sub, st_sub, exp)
    c1, r1, c2, r2, b = pts
    on_col = on_row = 0
    for i in np.flatnonzero(st == 1):
        res = co.rotate_and_match(img1, c1[i], r1[i], s, window(img2, s, c2[i], r2[i], b[i]), 0.0, angles=angles)
        bi, bj = np.unravel_index(np.argmax(res[5]), res[5].shape)
        if bj in (0, res[5].shape[1] - 1):
            on_col += 1
            assert offs[i, 0] == 0.0 and sub[i, 0].tobytes() == plain[i, 0].tobytes()
        if bi in (0, res[5].shape[0] - 1):
            on_row += 1
            assert offs[i, 1] == 0.0 and sub[i, 1].tobytes() == plain[i, 1].tobytes()
    assert on_col >= 4 and on_row >= 4, (on_col, on_row)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", dg.CLASSES)
@pytest.mark.parametrize("family", DEGENERATE, ids=[f[0] for f in DEGENERATE])
def test_degenerate_content_offsets_equal_oracle(gpu_ctx, monkeypatch, family, kind):
    """Flat templates (all-1.0 maps), exact position / angle ties and low contrast."""
    name, s, angles, (lo, hi), env, kernel = family
    _setenv(monkeypatch, env)
    img1, img2 = dg.images(kind)
    n = dg.n_points(kind)
    pts = dg.points(kind, s, (lo + np.arange(n) % (hi - lo + 1)).astype(np.float64))
    gpu_ctx.set_pair(img1, img2)
    plain, st = gpu_ctx.run(*pts, s, angles, 0.0, want_status=True)
    sub, st_sub = gpu_ctx.run(*pts, s, angles, 0.0, flags=_lib.SID_HES_NORM | _lib.SID_SUBPIXEL, want_status=True)
    exp, offs = expected_table(img1, img2, pts, s, angles, opts_of("default"), plain, st)
    assert_refined(plain, st, sub, st_sub, exp)
    valid = st == 1
    assert valid.any() and np.all(np.isfinite(offs[valid])) and np.all(np.abs(offs[valid]) <= 0.5)


def _cfg2_small(seed=3, side=1100, grid=14):
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=seed, side=side, grid=grid)
    return img1, img2, [c1, r1, c2, r2, b], cfg


@pytest.mark.gpu
@pytest.mark.parametrize("bands", ("1", "3", "8"))
def test_run_pair_bands(gpu_ctx, monkeypatch, bands):
    monkeypatch.setenv("SID_BANDS", bands)
    img1, img2, pts, cfg = _cfg2_small()
    flags = _lib.SID_HES_NORM | _lib.SID_SUBPIXEL
    plain, st = gpu_ctx.run_pair(img1, img2, *pts, 35, cfg["angles"], 0.0, want_status=True)
    sub, st_sub = gpu_ctx.run_pair(img1, img2, *pts, 35, cfg["angles"], 0.0, flags=flags, want_status=True)
    exp, _ = expected_table(img1, img2, pts, 35, cfg["angles"], opts_of("default"), plain, st)
    assert_refined(plain, st, sub, st_sub, exp)


@pytest.mark.gpu
def test_run_device_and_two_border_classes(gpu_ctx):
    import torch
    img1, img2 = speckle_pair()
    c1, r1, c2, r2, _ = speckle_points(35, 20, 50, n_grid=19)
    k = np.arange(c1.size)
    brd = np.where(k % 4 == 3, 21 + k % 30, 20).astype(np.float64)
    brd[-8:] = 20.0
    pts = [c1, r1, c2, r2, brd]
    flags = _lib.SID_HES_NORM | _lib.SID_SUBPIXEL
    gpu_ctx.set_pair(img1, img2)
    plain, st = gpu_ctx.run(*pts, 35, ANGLES, 0.0, want_status=True)
    sub, st_sub = gpu_ctx.run(*pts, 35, ANGLES, 0.0, flags=flags, want_status=True)
    big, small = gpu_ctx.last_kernel_name.split(" + ")
    assert small == "sid::pm_ws_kernel" and big.startswith("sid::pm_"), gpu_ctx.last_kernel_name
    exp, _ = expected_table(img1, img2, pts, 35, ANGLES, opts_of("default"), plain, st)
    assert_refined(plain, st, sub, st_sub, exp)
    ok = np.isfinite(brd) & np.isfinite(c1)
    dev = torch.device("cuda", gpu_ctx.device)
    d_pts = torch.from_numpy(np.stack([p[ok] for p in pts])).to(dev)
    d_out = torch.full((int(ok.sum()), 5), -7.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    gpu_ctx.run_device(int(ok.sum()), *[d_pts[j].data_ptr() for j in range(5)], 50, 35, ANGLES, 0.0, d_out.data_ptr(),
                       flags=flags)
    gpu_ctx.synchronize()
    assert d_out.cpu().numpy().tobytes() == sub[ok].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", ("default", "hes_smth"))
def test_run_maps_maps_unchanged_table_refined(gpu_ctx, flag_set):
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    o = opts_of(flag_set)
    gpu_ctx.set_pair(img1, img2)
    tab, maps, tpls, st = gpu_ctx.run_maps(*pts, 35, ANGLES, 0.0, o["rot_order"], flags_of(o), want_status=True)
    tab_s, maps_s, tpls_s, st_s = gpu_ctx.run_maps(*pts, 35, ANGLES, 0.0, o["rot_order"],
                                                   flags_of(o) | _lib.SID_SUBPIXEL, want_status=True)
    sub = gpu_ctx.run(*pts, 35, ANGLES, 0.0, o["rot_order"], flags_of(o) | _lib.SID_SUBPIXEL)
    assert tab_s.tobytes() == sub.tobytes() and np.array_equal(st_s, st) and np.array_equal(tpls_s, tpls)
    for i, (m, ms) in enumerate(zip(maps, maps_s)):
        assert (m is None and ms is None) or m.tobytes() == ms.tobytes()
        if st[i] == 1:       # the table is refined from exactly these maps
            dx, dy = peak_offsets(m)
            assert tab_s[i, 0] == tab[i, 0] + dx and tab_s[i, 1] == tab[i, 1] + dy
    # the public wrapper with return_maps
    t2, m2, _ = pmlib.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=ANGLES, return_maps=True, subpixel=True, **FLAG_SETS[flag_set])
    assert t2.tobytes() == tab_s.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", ("default", "hes_smth", "mcc_norm"))
def test_single_call_rotate_and_match(gpu_ctx, flag_set):
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    o = opts_of(flag_set)
    checked = 0
    for i in range(0, pts[0].size, 3):
        c1, r1, c2, r2, b = [p[i] for p in pts]
        if not np.all(np.isfinite([c1, r1])) or int(r2 - 17 - b) < 0 or int(c2 - 17 - b) < 0:
            continue
        win = window(img2, 35, c2, r2, b)
        got = pmlib.rotate_and_match(img1, c1, r1, 35, win, 0.0, angles=ANGLES, template_matcher=None, subpixel=True, **o)
        plain = pmlib.rotate_and_match(img1, c1, r1, 35, win, 0.0, angles=ANGLES, template_matcher=None, **o)
        res = co.rotate_and_match(img1, c1, r1, 35, win, 0.0, angles=ANGLES, **o)
        if np.isnan(res[0]):
            assert np.isnan(got[0])
            continue
        dx, dy = peak_offsets(res[5])
        assert got[0] == res[0] + dx and got[1] == res[1] + dy
        assert got[2:5] == plain[2:5] and got[5].tobytes() == plain[5].tobytes()
        checked += 1
    assert checked >= 5


def _drop_in_scene(side=2400, n_keypoints=20000, grid=40):
    """bench.py's drop_in_ew scene at a moderate size: cfg2's 2-degree rotation, synthetic feature-tracking matches in
    generic position with 0.8 px noise, known drift."""
    rng = np.random.default_rng(7)
    img1 = syn.speckle_image((side, side), 0)
    m = syn.rotation_matrix(img1.shape, syn.CONFIGS["cfg2"]["warp"][1])
    img2 = syn.warp_pair(img1, m, 0)
    kx, ky = rng.uniform(40, side - 40, n_keypoints), rng.uniform(40, side - 40, n_keypoints)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    k2x, k2y = k2x + rng.normal(0, 0.8, n_keypoints), k2y + rng.normal(0, 0.8, n_keypoints)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(150, side - 150, grid), np.linspace(150, side - 150, grid))
    lon, lat = n2.transform_points(gx, gy)
    return n1, n2, kx, ky, k2x, k2y, lon, lat, m


def _median_error(res, n1, n2, lon, lat, m):
    ok = np.isfinite(res[0])
    c2, r2 = n2.transform_points(res[5][ok], res[6][ok], 1)
    c1g, r1g = n1.transform_points(lon[ok], lat[ok], 1)
    tx, ty = syn.apply_affine(m, c1g, r1g)
    return float(np.median(np.hypot(c2 - (tx - 1), r2 - (ty - 1))))


@pytest.mark.gpu
def test_pattern_matching_drop_in(gpu_ctx):
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = _drop_in_scene()
    kw = dict(angles=[-3, 0, 3], img_size=35)
    dev = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, subpixel=True, **kw)
    host = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, subpixel=True, device_epilogue=False, **kw)
    plain = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, **kw)
    for a, b in zip(dev, host):
        assert np.array_equal(a, b, equal_nan=True) and a.tobytes() == b.tobytes()
    for k in (2, 3, 4):                                         # angle, r, h unchanged
        assert dev[k].tobytes() == plain[k].tobytes()
    assert np.array_equal(np.isnan(dev[0]), np.isnan(plain[0])) and np.isfinite(dev[0]).sum() > 0.9 * dev[0].size
    refined, integer = _median_error(dev, n1, n2, lon, lat, m), _median_error(plain, n1, n2, lon, lat, m)
    assert refined <= 0.15 and refined < 0.5 * integer, (refined, integer)


@pytest.mark.gpu
def test_split_over_two_gpus_equals_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29579", os.path.join(ROOT, "tests", "multi_gpu_subpixel.py")]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:]
    assert "subpixel split(2 ranks) == single GPU: True" in res.stdout
