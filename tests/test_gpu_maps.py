"""Winning correlation maps and templates from one batched call (sid_map_layout / sid_run_maps, Context.run_maps,
pmlib.use_mcc_batch(return_maps=True)).

For every valid row the map must be what the exact oracle's ``rotate_and_match(...)[5]`` returns for the point's
search window as ``use_mcc`` slices it, and the template its ``[6]``, bit for bit; the table and status must be
``run``'s bit for bit.  Every kernel family runs, with split and fused tails, shared-memory and global scratch, and the
kernel that ran is checked by name.  The CPU test pins the layout rule against NumPy slicing; the others need a GPU."""
import ctypes as C
import functools

import numpy as np
import pytest

from sea_ice_drift_b200 import _lib, pmlib
from sea_ice_drift_b200 import synthetic as syn
from oracle import c_oracle as co
from tests import test_degenerate_content as dg

SIDE = 360
ANGLES = [0, 3, -3]                 # img2 is img1 rotated by 3 degrees: the winner is mostly not index 0
ZERO_PIXEL = (150, 200)             # (row, col) of the 0 pixel in img1: the point centred there gives a NaN row
FLAG_SETS = {"default": {}, "hes_smth": dict(hes_smth=True), "mcc_norm": dict(mcc_norm=True),
             "raw_hes": dict(hes_norm=False), "rot_order1": dict(rot_order=1)}


def opts_of(flag_set):
    o = dict(rot_order=0, hes_norm=True, hes_smth=False, mcc_norm=False)
    o.update(FLAG_SETS[flag_set])
    return o


def flags_of(o):
    return _lib.flags_from_kwargs(o["hes_norm"], o["hes_smth"], o["mcc_norm"])


@functools.lru_cache(maxsize=None)
def speckle_pair():
    img1 = syn.speckle_image((SIDE, SIDE), seed=11)
    img2 = syn.warp_pair(img1, syn.rotation_matrix((SIDE, SIDE), 3.0), seed=11)
    img1 = img1.copy()
    img1[ZERO_PIXEL] = 0
    return img1, img2


def speckle_points(s, lo, hi, n_grid=5):
    """A grid of points with first guesses from the known rotation, plus one row of each special kind: a NaN row (0
    pixel in the template), two rejected rows (window starting left of image 2, NaN coordinate), windows clipped at the
    far edge (non-square maps) and fractional first guesses / borders."""
    hws = int(s / 2.)
    m = syn.rotation_matrix((SIDE, SIDE), 3.0)
    inset = hws + hi + 12
    gx, gy = syn.grid_points((SIDE, SIDE), n_grid, inset)
    c2, r2 = syn.apply_affine(m, gx, gy)
    c1, r1, c2, r2 = list(gx), list(gy), list(np.round(c2)), list(np.round(r2))
    brd = list(lo + np.arange(len(c1)) % (hi - lo + 1))

    def add(a, b, c, d, e):
        c1.append(a), r1.append(b), c2.append(c), r2.append(d), brd.append(e)
    add(ZERO_PIXEL[1], ZERO_PIXEL[0], ZERO_PIXEL[1], ZERO_PIXEL[0], lo)               # NaN row
    add(100.0, 100.0, float(hws + lo - 3), 100.0, lo)                                   # rejected: x0 < 0
    add(np.nan, 100.0, 100.0, 100.0, lo)                                                # rejected: NaN c1
    far = SIDE - hws - lo // 2                                                          # x1 / y1 clipped by the image
    add(float(far), 180.0, float(far), 180.0, lo)
    add(180.0, float(far), 180.0, float(far), lo)
    add(float(far), float(far), float(far), float(far), lo)
    add(170.0, 190.0, 170.5, 189.75, hi - 0.5)                                          # fractional first guess / border
    add(190.0, 170.0, 189.25, 170.5, lo + 0.25)
    return [np.asarray(v, dtype=np.float64) for v in (c1, r1, c2, r2, brd)]


def window(img2, s, c2, r2, b):
    """The search window exactly as use_mcc slices it (reference pmlib.py:200-202)."""
    hws = int(s / 2.)
    return img2[int(r2 - hws - b):int(r2 + hws + b + 1), int(c2 - hws - b):int(c2 + hws + b + 1)]


def window_rule(img2, s, c1, r1, c2, r2, b):
    """The kernels' acceptance rule for a search window, in NumPy terms: finite inputs, window starting inside image 2,
    at least one displacement more than the template in each direction after the far-edge clipping."""
    if not np.all(np.isfinite([c1, r1, c2, r2, b])):
        return None
    hws = int(s / 2.)
    y0, x0 = int(r2 - hws - b), int(c2 - hws - b)
    if y0 < 0 or x0 < 0:
        return None
    h, w = window(img2, s, c2, r2, b).shape
    return (h - s + 1, w - s + 1) if h >= s + 1 and w >= s + 1 else None


def layout(ctx, pts, s):
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in pts]
    shape = np.zeros((arrs[0].size, 2), np.int32)
    total = C.c_int64(0)
    ctx._check(ctx._lib.sid_map_layout(ctx.handle, arrs[0].size, *[a.ctypes.data for a in arrs], int(s),
                                       shape.ctypes.data, C.byref(total)))
    return shape, int(total.value)


def raw_run_maps(ctx, pts, s, angles, o, capacity=None, want_templates=True, alpha0=0.0):
    """sid_run_maps through ctypes with an explicit capacity: (table, status, packed maps, templates or None)."""
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in pts]
    n = arrs[0].size
    _, total = layout(ctx, pts, s)
    cap = total if capacity is None else capacity
    buf = np.full(max(cap, 1), 7.0, np.float32)
    tpl = np.full((n, s, s), 7, np.uint8) if want_templates else None
    ang = np.asarray(angles, dtype=np.float64)
    tab = _lib.angle_table(angles, alpha0, s)
    out = np.zeros((n, 5))
    st = np.zeros(n, np.int32)
    ctx._check(ctx._lib.sid_run_maps(
        ctx.handle, n, *[a.ctypes.data for a in arrs], int(s), len(angles), ang.ctypes.data, tab.ctypes.data,
        int(o["rot_order"]), int(flags_of(o)), 5, out.ctypes.data, st.ctypes.data, cap, buf.ctypes.data,
        None if tpl is None else tpl.ctypes.data))
    return out, st, buf[:total], tpl


def check_maps(ctx, img1, img2, pts, s, angles, o, kernel=None, alpha0=0.0):
    """run_maps against run (table, status), the exact oracle (maps, templates) and the layout; returns (table, maps,
    templates, status)."""
    ctx.set_pair(img1, img2)
    flags = flags_of(o)
    ref, st_ref = ctx.run(*pts, s, angles, alpha0, o["rot_order"], flags, want_status=True)
    ran = ctx.last_kernel_name
    if kernel is not None:
        assert ran == kernel, ran
    tab, maps, tpls, st = ctx.run_maps(*pts, s, angles, alpha0, o["rot_order"], flags, want_status=True)
    assert ctx.last_kernel_name == ran
    assert tab.tobytes() == ref.tobytes()
    assert np.array_equal(st, st_ref)
    shape, total = layout(ctx, pts, s)
    c1, r1, c2, r2, b = pts
    n_valid = 0
    for i in range(c1.size):
        rule = window_rule(img2, s, c1[i], r1[i], c2[i], r2[i], b[i])
        assert tuple(shape[i]) == (rule if rule is not None else (0, 0)), (i, shape[i], rule)
        if rule is None:
            assert st[i] == -1
        if st[i] != 1:
            assert maps[i] is None and not tpls[i].any()
            continue
        n_valid += 1
        res = co.rotate_and_match(img1, c1[i], r1[i], s, window(img2, s, c2[i], r2[i], b[i]), alpha0, angles=angles, **o)
        assert res[2] == tab[i, 2]
        assert maps[i].dtype == np.float32 and maps[i].shape == res[5].shape == tuple(shape[i])
        assert np.array_equal(maps[i].view(np.uint32), res[5].view(np.uint32)), i
        assert np.array_equal(tpls[i], res[6]), i
    assert n_valid > 0
    # the packed buffer: valid segments in point order, NaN everywhere else; templates 0 for rows that are not valid
    tab2, st2, buf, tpl2 = raw_run_maps(ctx, pts, s, angles, o, alpha0=alpha0)
    assert tab2.tobytes() == ref.tobytes() and np.array_equal(st2, st)
    assert buf.size == total
    off = np.concatenate([[0], np.cumsum(shape[:, 0].astype(np.int64) * shape[:, 1])])
    for i in range(c1.size):
        seg = buf[off[i]:off[i + 1]]
        if st[i] == 1:
            assert np.array_equal(seg.view(np.uint32), maps[i].ravel().view(np.uint32))
        else:
            assert np.isnan(seg).all()
    assert np.array_equal(tpl2, tpls)
    return tab, maps, tpls, st


# ---------------------------------------------------------------------------------------------------- CPU
def test_window_rule_shapes_match_numpy_slicing():
    """The layout rule used by the tests is NumPy's slicing: clipped far edges and fractional inputs give non-square
    maps, and the shape of a valid window is exactly the oracle's map shape."""
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    shapes = [window_rule(img2, 35, *[p[i] for p in pts]) for i in range(pts[0].size)]
    assert any(sh is not None and sh[0] != sh[1] for sh in shapes)
    assert sum(sh is None for sh in shapes) == 2
    i = next(k for k, sh in enumerate(shapes) if sh is not None and sh[0] != sh[1])
    c1, r1, c2, r2, b = [p[i] for p in pts]
    res = co.rotate_and_match(img1, c1, r1, 35, window(img2, 35, c2, r2, b), 0.0, angles=ANGLES)
    assert res[5].shape == shapes[i]


# ---------------------------------------------------------------------------------------------------- GPU
# (name, img_size, angles, border range, environment, kernel name or None)
FAMILIES = [
    ("ws", 35, ANGLES, (16, 20), {}, "sid::pm_ws_kernel"),
    ("tc_split", 35, ANGLES, (20, 26), {"SID_PM_PATH": "tc"}, "sid::pm_tc_kernel"),
    ("tc_fused", 35, ANGLES, (30, 40), {}, "sid::pm_tc_kernel"),
    ("tc_fused_global", 35, ANGLES, (30, 40), {"SID_PM_PATH": "tc", "SID_PM_GLOBAL_SCRATCH": "1"}, "sid::pm_tc_kernel"),
    ("imma_split", 35, ANGLES, (20, 30), {"SID_PM_PATH": "imma"}, "sid::pm_points_kernel<imma>"),
    ("imma_fused", 35, ANGLES, (20, 30), {"SID_PM_PATH": "imma", "SID_PM_SPLIT_TAIL": "0"}, "sid::pm_points_kernel<imma>"),
    ("imma_fused_global", 35, ANGLES, (20, 30), {"SID_PM_PATH": "imma", "SID_PM_SPLIT_TAIL": "0",
                                                 "SID_PM_GLOBAL_SCRATCH": "1"}, "sid::pm_points_kernel<imma>"),
    ("dp4a_s35_split", 35, ANGLES, (20, 30), {"SID_PM_PATH": "dp4a"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s35_fused", 35, ANGLES, (20, 30), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s35_fused_global", 35, ANGLES, (20, 30), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0",
                                                     "SID_PM_GLOBAL_SCRATCH": "1"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s50_fused", 50, ANGLES, (15, 25), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s50_fused_global", 50, ANGLES, (15, 25), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0",
                                                     "SID_PM_GLOBAL_SCRATCH": "1"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s21_fused", 21, ANGLES, (10, 16), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0"}, "sid::pm_points_kernel<dp4a>"),
    ("dp4a_s21_fused_global", 21, ANGLES, (10, 16), {"SID_PM_PATH": "dp4a", "SID_PM_SPLIT_TAIL": "0",
                                                     "SID_PM_GLOBAL_SCRATCH": "1"}, "sid::pm_points_kernel<dp4a>"),
    ("default_s21", 21, ANGLES, (10, 16), {}, None),
    ("default_s50_7angles", 50, [-9, -6, -3, 0, 3, 6, 9], (15, 20), {}, None),
    ("repeated_angle", 35, [2, 2, 2], (16, 20), {}, "sid::pm_ws_kernel"),
]
FAMILY_FLAGS = {"ws": FLAG_SETS, "tc_fused": FLAG_SETS, "imma_split": FLAG_SETS, "tc_split": ("default", "hes_smth"),
                "dp4a_s35_split": ("default", "hes_smth")}
CASES = [(f, fs) for f in FAMILIES for fs in FAMILY_FLAGS.get(f[0], ("default",))]


def _setenv(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("family,flag_set", CASES, ids=["%s-%s" % (f[0], fs) for f, fs in CASES])
def test_maps_equal_exact_oracle(gpu_ctx, monkeypatch, family, flag_set):
    name, s, angles, (lo, hi), env, kernel = family
    _setenv(monkeypatch, env)
    img1, img2 = speckle_pair()
    pts = speckle_points(s, lo, hi)
    tab, maps, tpls, st = check_maps(gpu_ctx, img1, img2, pts, s, angles, opts_of(flag_set), kernel)
    assert (st == 0).sum() >= 1 and (st == -1).sum() == 2
    assert any(m is not None and m.shape[0] != m.shape[1] for m in maps)
    if len(set(angles)) > 1:
        assert any(st[i] == 1 and tab[i, 2] != angles[0] for i in range(st.size))


DEGENERATE = [f for f in FAMILIES if f[0] in ("ws", "tc_fused", "imma_split", "imma_fused", "dp4a_s35_fused",
                                                 "repeated_angle")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ("plateaus", "periodic"))
@pytest.mark.parametrize("family", DEGENERATE, ids=[f[0] for f in DEGENERATE])
def test_maps_on_degenerate_content(gpu_ctx, monkeypatch, family, kind):
    """Flat templates (all-1.0 maps) and exact position / angle ties (first index wins)."""
    name, s, angles, (lo, hi), env, kernel = family
    _setenv(monkeypatch, env)
    img1, img2 = dg.images(kind)
    n = dg.n_points(kind)
    pts = dg.points(kind, s, (lo + np.arange(n) % (hi - lo + 1)).astype(np.float64))
    tab, maps, tpls, st = check_maps(gpu_ctx, img1, img2, pts, s, angles, opts_of("default"), kernel)
    if kind == "plateaus":
        assert any(m is not None and (m == 1.0).all() for m in maps)


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", ("default", "hes_smth"))
def test_maps_with_two_border_classes(gpu_ctx, flag_set):
    """Borders 20 and 21 ... 50 in one call: the larger class and the pm_ws_kernel class write one buffer."""
    img1, img2 = speckle_pair()
    c1, r1, c2, r2, _ = speckle_points(35, 20, 50, n_grid=19)
    k = np.arange(c1.size)
    brd = np.where(k % 4 == 3, 21 + k % 30, 20).astype(np.float64)
    brd[-8:] = 20.0
    assert (brd == 20).sum() >= 256 and brd.max() == 50
    pts = [c1, r1, c2, r2, brd]
    check_maps(gpu_ctx, img1, img2, pts, 35, ANGLES, opts_of(flag_set))
    assert gpu_ctx.last_kernel_name.endswith(" + sid::pm_ws_kernel"), gpu_ctx.last_kernel_name


@pytest.mark.gpu
def test_maps_s51_border60_fused_tail(gpu_ctx):
    img1, img2 = speckle_pair()
    pts = speckle_points(51, 60, 60, n_grid=3)
    check_maps(gpu_ctx, img1, img2, pts, 51, ANGLES, opts_of("default"))
    assert "pm_ws_kernel" not in gpu_ctx.last_kernel_name


@pytest.mark.gpu
def test_capacity_below_total_is_refused_before_any_launch(gpu_ctx):
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    gpu_ctx.set_pair(img1, img2)
    _, total = layout(gpu_ctx, pts, 35)
    launches = gpu_ctx.launch_count
    with pytest.raises(ValueError):
        raw_run_maps(gpu_ctx, pts, 35, ANGLES, opts_of("default"), capacity=total - 1)
    assert gpu_ctx.launch_count == launches
    tab, st, buf, _ = raw_run_maps(gpu_ctx, pts, 35, ANGLES, opts_of("default"), capacity=total)
    assert gpu_ctx.launch_count > launches and (st == 1).any()


@pytest.mark.gpu
def test_templates_may_be_null(gpu_ctx):
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    gpu_ctx.set_pair(img1, img2)
    o = opts_of("default")
    tab, st, buf, tpl = raw_run_maps(gpu_ctx, pts, 35, ANGLES, o)
    tab0, st0, buf0, tpl0 = raw_run_maps(gpu_ctx, pts, 35, ANGLES, o, want_templates=False)
    assert tpl0 is None and tab0.tobytes() == tab.tobytes() and np.array_equal(st0, st)
    assert buf0.tobytes() == buf.tobytes()


@pytest.mark.gpu
def test_use_mcc_batch_return_maps(gpu_ctx):
    img1, img2 = speckle_pair()
    c1, r1, c2, r2, b = speckle_points(35, 16, 20)
    kw = dict(angles=ANGLES, hes_smth=True)
    ref, st = gpu_ctx.set_pair(img1, img2).run(c1, r1, c2, r2, b, 35, ANGLES, 0.0, 0, flags_of(opts_of("hes_smth")),
                                               want_status=True)
    _, maps_ref, tpls_ref = gpu_ctx.run_maps(c1, r1, c2, r2, b, 35, ANGLES, 0.0, 0, flags_of(opts_of("hes_smth")))
    plain = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, **kw)
    assert isinstance(plain, np.ndarray) and plain.tobytes() == ref.tobytes()
    for resident in (False, True):
        tab, maps, tpls = pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, return_maps=True,
                                              resident=resident, **kw)
        assert tab.tobytes() == ref.tobytes() and np.array_equal(tpls, tpls_ref)
        for m, mr in zip(maps, maps_ref):
            assert (m is None and mr is None) or m.tobytes() == mr.tobytes()
    # a user-supplied matcher cannot return maps from the batched kernels
    with pytest.raises(ValueError):
        pmlib.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, return_maps=True,
                            template_matcher=lambda im, tp, m: pmlib.match_template(im, tp, m), **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", ("default", "mcc_norm"))
def test_maps_agree_with_per_point_rotate_and_match(gpu_ctx, flag_set):
    """A sample of points against the public single-point call, which uploads its own window."""
    img1, img2 = speckle_pair()
    pts = speckle_points(35, 16, 20)
    o = opts_of(flag_set)
    gpu_ctx.set_pair(img1, img2)
    tab, maps, tpls, st = gpu_ctx.run_maps(*pts, 35, ANGLES, 0.0, o["rot_order"], flags_of(o), want_status=True)
    checked = 0
    for i in np.flatnonzero(st == 1)[::3]:
        c1, r1, c2, r2, b = [p[i] for p in pts]
        res = pmlib.rotate_and_match(img1, c1, r1, 35, window(img2, 35, c2, r2, b), 0.0, angles=ANGLES,
                                     template_matcher=None, mcc_norm=o["mcc_norm"])
        assert res[2] == tab[i, 2]
        assert res[5].tobytes() == maps[i].tobytes() and np.array_equal(res[6], tpls[i])
        checked += 1
    assert checked >= 5
