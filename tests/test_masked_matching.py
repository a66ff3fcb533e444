"""Masked correlation for templates with invalid pixels (SID_MASKED, ``masked=True``).

A row the reference returns as NaN because some angle's template holds a 0 pixel (land, no-data, samples outside image
1) is matched by the Pearson correlation over the templates' valid pixels when every angle's template has at least
ceil(s^2 / 2) valid pixels and vt > 0 (include/sid_b200.h); its status is 2.  The exact C oracle of the rule is
tests/masked_oracle.c (sido_match_template_masked / sido_rotate_and_match_ex on top of oracle/mcc_oracle.c); on the CPU it is pinned against a float64 NumPy restatement,
against cv2's masked TM_CCOEFF_NORMED and on an island probe with a known drift.  On the GPU every table, status, map
and template must equal the oracle's bit for bit (sub-pixel offsets: the oracle's map through ``peak_offsets``)."""
import numpy as np
import pytest

from sea_ice_drift_b200 import _lib, pmlib
from sea_ice_drift_b200 import synthetic as syn
from sea_ice_drift_b200.seaicedrift import SeaIceDrift
from oracle import c_oracle as co
from tests import masked_oracle as mo
from tests.test_gpu_maps import window
from tests.test_subpixel import peak_offsets

MASKED_FLAGS = _lib.SID_HES_NORM | _lib.SID_MASKED


def masked_ncc_f64(img, tpl):
    """The masked rule in NumPy: exact int64 sums, then float64 in the rule's order, clamped, float32."""
    img = np.asarray(img, np.int64)
    t = np.asarray(tpl, np.int64)
    s = t.shape[0]
    m = (t > 0).astype(np.int64)
    n, st, stt = m.sum(), t.sum(), (t * t).sum()
    win = np.lib.stride_tricks.sliding_window_view(img, (s, s))
    c = np.einsum("yxij,ij->yx", win, t)
    sw = np.einsum("yxij,ij->yx", win, m)
    sww = np.einsum("yxij,ij->yx", win * win, m)
    num, vt, vw = n * c - st * sw, n * stt - st * st, n * sww - sw * sw
    with np.errstate(invalid="ignore", divide="ignore"):
        r = num.astype(np.float64) / (np.sqrt(np.float64(vt)) * np.sqrt(vw.astype(np.float64)))
    r = np.where(vw == 0, 0.0, np.clip(r, -1.0, 1.0))
    return r.astype(np.float32)


def pearson_f64(img, tpl):
    """Textbook Pearson correlation over the valid template pixels, float64 with means subtracted."""
    s = tpl.shape[0]
    m = tpl > 0
    t = tpl[m].astype(np.float64)
    t = t - t.mean()
    win = np.lib.stride_tricks.sliding_window_view(np.asarray(img, np.float64), (s, s))[..., m]
    w = win - win.mean(axis=-1, keepdims=True)
    den = np.sqrt((w * w).sum(-1)) * np.sqrt((t * t).sum())
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(den > 0, (w * t).sum(-1) / den, 0.0)


def template_with_zeros(rng, s, frac=0.3):
    t = rng.integers(1, 256, (s, s)).astype(np.uint8)
    k = int(frac * s)
    t[:k, :k] = 0
    t[-max(1, k // 2):, s // 2:] = 0
    return t


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("s", (2, 3, 8, 35, 36, 64))
def test_oracle_masked_map_equals_float64_restatement(s):
    rng = np.random.default_rng(s)
    img = rng.integers(0, 256, (s + 23, s + 17)).astype(np.uint8)
    img[3:9, 2:7] = 0                                   # window zeros are data
    tpl = template_with_zeros(rng, s, 0.25) if s > 3 else np.array(rng.integers(1, 256, (s, s)), np.uint8)
    if s <= 3:
        tpl.flat[0] = 0
    got = mo.match_template_masked(img, tpl)
    exp = masked_ncc_f64(img, tpl)
    assert got.tobytes() == exp.tobytes()              # same operations: bit for bit
    # and within float32 rounding of the textbook formula
    assert np.max(np.abs(got - pearson_f64(img, tpl))) <= 2e-7


def test_oracle_equals_cv2_masked_matchtemplate():
    import cv2
    rng = np.random.default_rng(5)
    ties = 0
    for k in range(12):
        s = (35, 21, 50)[k % 3]
        img = syn.speckle_image((s + 40, s + 44), seed=k)
        img[rng.integers(0, s):, :rng.integers(1, 20)] = 0
        tpl = syn.speckle_image((s, s), seed=100 + k)
        tpl[:rng.integers(1, s // 2), :rng.integers(1, s // 2)] = 0
        tpl[-rng.integers(1, s // 3):, -rng.integers(1, s // 2):] = 0
        got = mo.match_template_masked(img, tpl)
        ref = cv2.matchTemplate(img, tpl, cv2.TM_CCOEFF_NORMED, mask=(tpl > 0).astype(np.uint8))
        assert np.max(np.abs(got - ref)) <= 5e-6            # cv2 works in float32
        if got.argmax() != ref.argmax():                    # a near-tie: the exact values at both picks agree
            assert abs(float(got.flat[got.argmax()]) - float(got.flat[ref.argmax()])) <= 1e-5
            ties += 1
    assert ties <= 2


def _land_pair(side=320, seed=3, drift=(6, 4)):
    """A speckle pair with a known integer drift, an island (radius 45) and a no-data corner in both images."""
    big = syn.speckle_image((side + 10, side + 10), seed)
    dx, dy = drift
    img1 = big[1 + dy:1 + dy + side, 1 + dx:1 + dx + side].copy()
    img2 = big[1:1 + side, 1:1 + side].copy()             # img2[y + dy, x + dx] == img1[y, x]
    yy, xx = np.mgrid[:side, :side]
    land = (xx - 0.55 * side) ** 2 + (yy - 0.5 * side) ** 2 < 45 ** 2
    nodata = xx + yy < 0.3 * side
    for im in (img1, img2):
        im[land | nodata] = 0
    return img1, img2


def _land_points(img1, s, border, drift=(6, 4), n_extra=0, seed=0):
    """A grid over the scene, points next to the island and the no-data corner, templates crossing image 1's edges
    (first guesses inside image 2) and two rejected rows."""
    side = img1.shape[0]
    hws = s // 2
    rng = np.random.default_rng(seed)
    lo = hws + border + 8
    g = np.linspace(lo, side - 1 - lo - max(drift), 7)
    gx, gy = [a.ravel() for a in np.meshgrid(g, g)]
    ang = rng.uniform(0, 2 * np.pi, 24)
    rad = rng.uniform(45 - 0.3 * s, 45 + 0.7 * s, ang.size)
    ix, iy = 0.55 * side + rad * np.cos(ang), 0.5 * side + rad * np.sin(ang)
    t = rng.uniform(0.3 * side - 0.4 * s, 0.3 * side + 0.6 * s, 10) / np.sqrt(2)
    cx, cy = t + rng.uniform(-8, 8, t.size), t + rng.uniform(-8, 8, t.size)
    c1 = np.round(np.concatenate([gx, ix, cx]))
    r1 = np.round(np.concatenate([gy, iy, cy]))
    c2, r2 = c1 + drift[0], r1 + drift[1]
    ok = (c2 - hws - border >= 0) & (r2 - hws - border >= 0) & (c2 + hws + border < side) & (r2 + hws + border < side)
    c1, r1, c2, r2 = c1[ok], r1[ok], c2[ok], r2[ok]
    # templates crossing image 1's left / top edge by 1 ... hws px, windows in the middle of image 2
    e = np.arange(1, hws + 1, max(1, hws // 4))
    mid = side / 2.0
    c1 = np.concatenate([c1, e, np.full(e.size, mid - 40), [5.0]])
    r1 = np.concatenate([r1, np.full(e.size, mid + 30), e + 0.5, [5.0]])
    c2 = np.concatenate([c2, np.full(e.size, mid + 40), np.full(e.size, mid - 60), [float(hws + border - 3)]])
    r2 = np.concatenate([r2, np.full(e.size, mid + 50), np.full(e.size, mid + 20), [mid]])
    b = np.full(c1.size, float(border))
    b[::5] = border - 1
    return [np.asarray(v, np.float64) for v in (c1, r1, c2, r2, b)]


def test_rows_without_zeros_are_byte_identical_in_the_oracle():
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 12)
    plain, st = co.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[-3, 0, 3])
    got, st_m = mo.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[-3, 0, 3])
    keep = st != 0
    assert np.array_equal(st_m[keep], st[keep])
    assert got[keep].tobytes() == plain[keep].tobytes()
    assert set(np.unique(st_m[~keep])) <= {0, 2}
    assert (st_m == 2).sum() >= 10 and (st_m[~keep] == 0).sum() >= 1 and (st == -1).sum() >= 1


def _threshold_case(s, n_zero, flat=False):
    """img1 whose angle-0 template at (c, r) has exactly n_zero 0 pixels (row-major from its top-left corner)."""
    rng = np.random.default_rng(s)
    img1 = rng.integers(1, 256, (120, 120)).astype(np.uint8)
    img2 = rng.integers(1, 256, (120, 120)).astype(np.uint8)
    c = r = 60.0
    tc = int(s / 2.) + 1
    rows, cols = np.divmod(np.arange(s * s), s)
    ys, xs = int(r) - tc + rows, int(c) - tc + cols
    if flat:
        img1[ys, xs] = 100
    img1[ys[:n_zero], xs[:n_zero]] = 0
    assert (co.get_template(img1, c, r, 0.0, s) == 0).sum() == n_zero
    return img1, img2, [np.array([v], np.float64) for v in (c, r, c + 2, r - 1, 6.0)]


@pytest.mark.parametrize("s", (5, 6, 35, 36))
def test_valid_pixel_threshold_boundary(s):
    need = (s * s + 1) // 2                                       # ceil(s^2 / 2)
    for n_zero, want in ((s * s - need, 2), (s * s - need + 1, 0), (1, 2)):
        img1, img2, pts = _threshold_case(s, n_zero)
        _, st = mo.use_mcc_batch(*pts, img1, img2, s, 0.0, angles=[0])
        assert st[0] == want, (s, n_zero, st)


def test_flat_valid_template_stays_nan_and_flat_window_gives_zero():
    img1, img2, pts = _threshold_case(35, 40, flat=True)
    tab, st = mo.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[0])
    assert st[0] == 0 and np.isnan(tab[0]).all()
    tpl = template_with_zeros(np.random.default_rng(1), 35)
    flat = np.full((50, 60), 77, np.uint8)
    assert not mo.match_template_masked(flat, tpl).any()
    part = flat.copy()
    part[:, 35:] = np.random.default_rng(2).integers(0, 256, (50, 25))
    m = mo.match_template_masked(part, tpl)
    assert m[:, 0].tolist() == [0.0] * m.shape[0] and np.abs(m[:, -1]).max() > 0


def test_island_probe_recovers_the_coastal_band():
    """1000^2 speckle pair, drift (6, 4) px, an island of radius 150 px zeroed in both images; points 150 ... 185 px from
    its centre matched from the true first guess (border 20, angle 0).  The reference gives NaN wherever a template
    touches land; the masked rule recovers almost all of those with >= 50 % valid template pixels, within 1 px."""
    side, drift = 1000, (6, 4)
    big = syn.speckle_image((side + 10, side + 10), 42)
    img1 = big[1 + drift[1]:1 + drift[1] + side, 1 + drift[0]:1 + drift[0] + side].copy()
    img2 = big[1:1 + side, 1:1 + side].copy()
    yy, xx = np.mgrid[:side, :side]
    land = (xx - 500) ** 2 + (yy - 500) ** 2 < 150 ** 2
    img1[land] = 0
    img2[land] = 0
    rng = np.random.default_rng(0)
    n = 1500
    a, rad = rng.uniform(0, 2 * np.pi, n), rng.uniform(150, 185, n)
    c1, r1 = np.round(500 + rad * np.cos(a)), np.round(500 + rad * np.sin(a))
    pts = [c1, r1, c1 + drift[0], r1 + drift[1], np.full(n, 20.0)]
    plain, st = co.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[0])
    tab, st_m = mo.use_mcc_batch(*pts, img1, img2, 35, 0.0, angles=[0])
    # the template-centre convention of the reference: a true match lands at c1 + drift - 1 (odd img_size); a few valid
    # rows see land in image 2 where the ice moved towards the island
    ok = st == 1

    def error(rows):
        return np.hypot(tab[rows, 0] - (c1[rows] + drift[0] - 1), tab[rows, 1] - (r1[rows] + drift[1] - 1))
    assert ok.sum() > 100 and (error(ok) == 0).mean() >= 0.98
    touching = st == 0
    valid_frac = np.array([(co.get_template(img1, c1[i], r1[i], 0.0, 35) > 0).mean() for i in range(n)])
    eligible = touching & (valid_frac >= 0.5)
    assert touching.sum() > 0.4 * n and eligible.sum() > 0.9 * touching.sum()
    assert np.array_equal(st_m == 2, eligible)
    err = error(eligible)
    assert (err <= 1.0).mean() >= 0.97, (err <= 1.0).mean()
    assert (err > 2.0).mean() <= 0.01


def test_masked_keyword_maps_to_the_flag_and_user_matcher_is_refused():
    assert _lib.flags_from_options(dict(masked=True)) == _lib.SID_HES_NORM | _lib.SID_MASKED
    assert _lib.flags_from_options({}) == _lib.SID_HES_NORM
    img1, img2 = _land_pair(120)
    calls = []

    def matcher(*a):
        calls.append(a)
        raise AssertionError("the user matcher must not run")
    with pytest.raises(ValueError, match="masked=True"):
        pmlib.rotate_and_match(img1, 60.0, 60.0, 35, img2[20:100, 20:100], 0.0, template_matcher=matcher, masked=True)
    with pytest.raises(ValueError, match="masked=True"):
        pmlib.use_mcc_batch([60.0], [60.0], [60.0], [60.0], [10.0], img1, img2, 35, 0.0, template_matcher=matcher,
                            masked=True)
    assert not calls


# ---------------------------------------------------------------------------------------------------- GPU
def expected(img1, img2, pts, s, angles, o, subpixel=False):
    """The exact oracle's masked table and status; with ``subpixel`` c2 / r2 of valid and masked rows refined by
    peak_offsets of the oracle's map."""
    tab, st = mo.use_mcc_batch(*pts, img1, img2, s, 0.0, angles=angles, **o)
    if subpixel:
        c1, r1, c2, r2, b = pts
        for i in np.flatnonzero(st > 0):
            res = mo.rotate_and_match(img1, c1[i], r1[i], s, window(img2, s, c2[i], r2[i], b[i]), 0.0, angles=angles,
                                      **o)
            dx, dy = peak_offsets(res[5])
            tab[i, 0], tab[i, 1] = (c2[i] + res[0]) + dx, (r2[i] + res[1]) + dy
    return tab, st


def flags_of(o, subpixel=False, masked=True):
    return _lib.flags_from_kwargs(o.get("hes_norm", True), o.get("hes_smth", False), o.get("mcc_norm", False),
                                  subpixel, masked)


def assert_table(got, st_got, exp, st_exp):
    assert np.array_equal(st_got, st_exp), np.flatnonzero(st_got != st_exp)
    bad = np.flatnonzero((got.view(np.uint64) != exp.view(np.uint64)).any(axis=1))
    assert bad.size == 0, (bad, got[bad[:3]], exp[bad[:3]])


# (name, img_size, angles, border, environment, kernel name)
FAMILIES = [
    ("ws", 35, [-3, 0, 3], 16, {}, "sid::pm_ws_kernel"),
    ("tc", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "tc"}, "sid::pm_tc_kernel"),
    ("tc_fused", 35, [-3, 0, 3], 36, {}, "sid::pm_tc_kernel"),
    ("imma", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "imma"}, "sid::pm_points_kernel<imma>"),
    ("dp4a", 35, [-3, 0, 3], 24, {"SID_PM_PATH": "dp4a"}, "sid::pm_points_kernel<dp4a>"),
    ("ws_even_1angle", 36, [0], 14, {}, "sid::pm_ws_kernel"),
    ("tc_even_7angles", 36, [-9, -6, -3, 0, 3, 6, 9], 22, {"SID_PM_PATH": "tc"}, "sid::pm_tc_kernel"),
    ("dp4a_odd_7angles", 21, [-9, -6, -3, 0, 3, 6, 9], 14, {"SID_PM_PATH": "dp4a"}, "sid::pm_points_kernel<dp4a>"),
    ("imma_s50", 50, [-3, 0, 3], 20, {"SID_PM_PATH": "imma", "SID_PM_SPLIT_TAIL": "0"}, "sid::pm_points_kernel<imma>"),
]
OPTION_SETS = {
    "default": ({}, False), "subpixel": ({}, True), "hes_smth": (dict(hes_smth=True), False),
    "mcc_norm_subpixel": (dict(mcc_norm=True), True), "raw_hes_rot1": (dict(hes_norm=False, rot_order=1), False),
    "all": (dict(hes_smth=True, mcc_norm=True, rot_order=1), True),
}
CASES = [(f, o) for f in FAMILIES for o in (("default", "subpixel", "hes_smth", "mcc_norm_subpixel", "raw_hes_rot1", "all")
                                            if f[0] in ("ws", "tc", "dp4a") else ("default", "subpixel"))]


@pytest.mark.gpu
@pytest.mark.parametrize("family,option_set", CASES, ids=["%s-%s" % (f[0], o) for f, o in CASES])
def test_every_kernel_family_equals_masked_oracle(gpu_ctx, monkeypatch, family, option_set):
    name, s, angles, border, env, kernel = family
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    o, subpixel = OPTION_SETS[option_set]
    img1, img2 = _land_pair()
    pts = _land_points(img1, s, border)
    gpu_ctx.set_pair(img1, img2)
    rot = o.get("rot_order", 0)
    plain, st_plain = gpu_ctx.run(*pts, s, angles, 0.0, rot, flags_of(o, subpixel, False), want_status=True)
    n0 = gpu_ctx.launch_count
    gpu_ctx.run(*pts, s, angles, 0.0, rot, flags_of(o, subpixel, False))
    n_plain = gpu_ctx.launch_count - n0
    got, st = gpu_ctx.run(*pts, s, angles, 0.0, rot, flags_of(o, subpixel), want_status=True)
    assert gpu_ctx.last_kernel_name == kernel
    assert gpu_ctx.launch_count - n0 - n_plain == n_plain + 2          # + candidates + pm_masked_kernel
    exp, st_exp = expected(img1, img2, pts, s, angles, o, subpixel)
    assert_table(got, st, exp, st_exp)
    assert (st == 2).sum() >= 5 and (st == 1).sum() >= 10 and (st == -1).sum() >= 1
    keep = st_plain != 0                                                # rows without zeros: the call without the flag
    assert np.array_equal(st[keep], st_plain[keep]) and got[keep].tobytes() == plain[keep].tobytes()


@pytest.mark.gpu
def test_launch_count_without_the_flag(gpu_ctx):
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 16)
    gpu_ctx.set_pair(img1, img2)
    n0 = gpu_ctx.launch_count
    gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0)
    assert gpu_ctx.launch_count - n0 == 2                               # pm_ws_kernel and its split tail
    n0 = gpu_ctx.launch_count
    gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, flags=MASKED_FLAGS)
    assert gpu_ctx.launch_count - n0 == 4


@pytest.mark.gpu
@pytest.mark.parametrize("bands", ("3", "8"))
def test_run_pair_bands(gpu_ctx, monkeypatch, bands):
    monkeypatch.setenv("SID_BANDS", bands)
    img1, img2 = _land_pair(side=1400, seed=8)
    pts = _land_points(img1, 35, 20)
    other = np.ascontiguousarray(img1[::-1])                            # a stale resident pair first
    gpu_ctx.set_pair(other, other)
    got, st = gpu_ctx.run_pair(img1, img2, *pts, 35, [-3, 0, 3], 0.0, flags=MASKED_FLAGS | _lib.SID_SUBPIXEL,
                               want_status=True)
    exp, st_exp = expected(img1, img2, pts, 35, [-3, 0, 3], {}, True)
    assert_table(got, st, exp, st_exp)
    assert (st == 2).sum() >= 5


def _two_class_points(img1):
    pts = _land_points(img1, 35, 20, seed=1)
    c1, r1, c2, r2, _ = pts
    reps = 12                                                           # >= 512 points: run_device splits classes
    k = np.arange(c1.size * reps)
    brd = np.where(k % 4 == 3, 21 + k % 20, 16).astype(np.float64)
    return [np.tile(c1, reps), np.tile(r1, reps), np.tile(c2, reps), np.tile(r2, reps), brd]


@pytest.mark.gpu
def test_run_device_and_two_border_classes(gpu_ctx):
    import torch
    img1, img2 = _land_pair(side=420, seed=5)
    pts = _two_class_points(img1)
    gpu_ctx.set_pair(img1, img2)
    got, st = gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, flags=MASKED_FLAGS, want_status=True)
    big, small = gpu_ctx.last_kernel_name.split(" + ")
    assert small == "sid::pm_ws_kernel", gpu_ctx.last_kernel_name
    exp, st_exp = expected(img1, img2, pts, 35, [-3, 0, 3], {})
    assert_table(got, st, exp, st_exp)
    assert (st == 2).sum() >= 20
    dev = torch.device("cuda", gpu_ctx.device)
    n = pts[0].size
    d_pts = torch.from_numpy(np.stack(pts)).to(dev)
    for with_status in (True, False):
        d_out = torch.full((n, 5), -7.0, dtype=torch.float64, device=dev)
        d_st = torch.full((n,), 9, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        gpu_ctx.run_device(n, *[d_pts[j].data_ptr() for j in range(5)], 40, 35, [-3, 0, 3], 0.0, d_out.data_ptr(),
                           d_st.data_ptr() if with_status else 0, flags=MASKED_FLAGS)
        gpu_ctx.synchronize()
        assert d_out.cpu().numpy().tobytes() == got.tobytes()
        if with_status:
            assert np.array_equal(d_st.cpu().numpy(), st)


@pytest.mark.gpu
@pytest.mark.parametrize("option_set", ("default", "all"))
def test_run_maps_masked_maps_and_templates(gpu_ctx, option_set):
    o, subpixel = OPTION_SETS[option_set]
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 16)
    gpu_ctx.set_pair(img1, img2)
    rot = o.get("rot_order", 0)
    tab, maps, tpls, st = gpu_ctx.run_maps(*pts, 35, [-3, 0, 3], 0.0, rot, flags_of(o, subpixel), want_status=True)
    ref, st_ref = gpu_ctx.run(*pts, 35, [-3, 0, 3], 0.0, rot, flags_of(o, subpixel), want_status=True)
    assert tab.tobytes() == ref.tobytes() and np.array_equal(st, st_ref)
    c1, r1, c2, r2, b = pts
    for i in range(c1.size):
        if st[i] <= 0:
            assert maps[i] is None and not tpls[i].any()
            continue
        res = mo.rotate_and_match(img1, c1[i], r1[i], 35, window(img2, 35, c2[i], r2[i], b[i]), 0.0,
                                  angles=[-3, 0, 3], **o)
        assert maps[i].view(np.uint32).tobytes() == res[5].view(np.uint32).tobytes(), i
        assert np.array_equal(tpls[i], res[6]), i
        if (res[6] == 0).any():                             # (a masked row's winning template may have no zero)
            assert st[i] == 2
    assert (st == 2).sum() >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("option_set", ("default", "subpixel", "all"))
def test_single_call_rotate_and_match(gpu_ctx, option_set):
    o, subpixel = OPTION_SETS[option_set]
    img1, img2 = _land_pair()
    pts = _land_points(img1, 35, 16)
    c1, r1, c2, r2, b = pts
    masked = 0
    for i in range(c1.size):
        if int(r2[i] - 17 - b[i]) < 0 or int(c2[i] - 17 - b[i]) < 0:
            continue
        win = window(img2, 35, c2[i], r2[i], b[i])
        got = pmlib.rotate_and_match(img1, c1[i], r1[i], 35, win, 0.0, angles=[-3, 0, 3], masked=True,
                                     subpixel=subpixel, **o)
        res = mo.rotate_and_match(img1, c1[i], r1[i], 35, win, 0.0, angles=[-3, 0, 3], **o)
        if np.isnan(res[0]):
            assert np.isnan(got[0])
            continue
        dx, dy = peak_offsets(res[5]) if subpixel else (0.0, 0.0)
        assert got[0] == res[0] + dx and got[1] == res[1] + dy and got[2] == res[2]
        assert np.float32(got[3]).tobytes() == np.float32(res[3]).tobytes()
        assert abs(got[4] - res[4]) <= 4e-6 * (1 + abs(res[4]))
        assert got[5].tobytes() == res[5].tobytes() and np.array_equal(got[6], res[6])
        masked += bool((res[6] == 0).any())
    assert masked >= 5
    # a window of any size: 300 x 280 around a point next to the island
    i = next(k for k in range(c1.size) if 80 < c1[k] < 240 and 80 < r1[k] < 240 and
             (co.get_template(img1, c1[k], r1[k], -3.0, 35) == 0).any() and
             mo.use_mcc_batch(*[p[k:k + 1] for p in pts], img1, img2, 35, 0.0)[1][0] == 2)
    win = img2[10:310, 20:300]
    got = pmlib.rotate_and_match(img1, c1[i], r1[i], 35, win, 0.0, angles=[-3, 0, 3], masked=True)
    res = mo.rotate_and_match(img1, c1[i], r1[i], 35, win, 0.0, angles=[-3, 0, 3])
    assert got[:3] == res[:3] and got[5].tobytes() == res[5].tobytes()


def _coast_scene(side=1600, drift=(6.0, 4.0), grid=50):
    """Drop-in scene: speckle ice moving by a known drift, a coastline (land fixed in both images), no-data corners and
    feature-tracking matches on ice only."""
    img1 = syn.speckle_image((side, side), 4)
    m = syn.shift_matrix(*drift)
    img2 = syn.warp_pair(img1, m, 4)
    yy, xx = np.mgrid[:side, :side]
    land = xx > 0.7 * side + 60 * np.sin(yy / 90.0)
    img1[land | (xx + yy < 0.25 * side)] = 0
    img2[land | ((side - xx) + yy < 0.25 * side)] = 0
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    rng = np.random.default_rng(9)
    kx, ky = rng.uniform(40, side - 40, 8000), rng.uniform(40, side - 40, 8000)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    on_ice = (img1[ky.astype(int), kx.astype(int)] > 0) & (img2[np.clip(k2y, 0, side - 1).astype(int),
                                                              np.clip(k2x, 0, side - 1).astype(int)] > 0)
    kx, ky, k2x, k2y = kx[on_ice], ky[on_ice], k2x[on_ice] + rng.normal(0, 0.5, on_ice.sum()), \
        k2y[on_ice] + rng.normal(0, 0.5, on_ice.sum())
    gx, gy = np.meshgrid(np.linspace(100, side - 100, grid), np.linspace(100, side - 100, grid))
    lon, lat = n2.transform_points(gx, gy)
    return n1, n2, kx, ky, k2x, k2y, lon, lat, m


def drift_errors(res, n1, n2, lon, lat, m):
    ok = np.isfinite(res[0])
    c2, r2 = n2.transform_points(res[5][ok], res[6][ok], 1)
    c1g, r1g = n1.transform_points(lon[ok], lat[ok], 1)
    tx, ty = syn.apply_affine(m, c1g, r1g)
    out = np.full(res[0].shape, np.nan)
    out[ok] = np.hypot(c2 - (tx - 1), r2 - (ty - 1))
    return out


@pytest.mark.gpu
def test_get_drift_pm_masked_recovers_coastal_vectors(gpu_ctx):
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = _coast_scene()
    sid = SeaIceDrift(n1, n2)
    ll = (*n1.transform_points(kx, ky), *n2.transform_points(k2x, k2y))
    plain = sid.get_drift_PM(lon, lat, *ll, angles=[-3, 0, 3], img_size=35)
    got = sid.get_drift_PM(lon, lat, *ll, angles=[-3, 0, 3], img_size=35, masked=True)
    was = np.isfinite(plain[0])
    for a, b in zip(plain, got):                                    # the unmasked call's vectors, unchanged
        assert a[was].tobytes() == b[was].tobytes()
    new = np.isfinite(got[0]) & ~was
    assert new.sum() >= 40, new.sum()
    err = drift_errors(got, n1, n2, lon, lat, m)
    assert np.nanmedian(err[new]) <= 0.5 and np.mean(err[new] <= 1.5) >= 0.85, (np.nanmedian(err[new]),
                                                                              np.mean(err[new] <= 1.5))
    assert np.nanmedian(err[was]) <= 0.8
