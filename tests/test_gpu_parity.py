"""Parity tests proper: the CUDA path, called through the C ABI, against (a) the golden
vectors of the live reference, (b) the exact CPU oracle on seeded inputs, and (c)
size-independent properties at BASELINE.json's full sizes.  Needs a B200 (-m gpu)."""
import contextlib
import io
import os

import numpy as np
import pytest

import sea_ice_drift_b200 as sid
from sea_ice_drift_b200 import _lib, synthetic as syn, sharding
from oracle import c_oracle as co
from tests.helpers import variant_inputs, classify, make_exact_lookup, assert_parity, assert_equals_exact_oracle

pytestmark = pytest.mark.gpu

VARIANTS = ["default", "one_angle", "rot_order1", "hes_smth", "raw_hes_mcc_norm", "even50_7angles",
            "s51_b60", "s21_b9"]


def flags(opts):
    return _lib.flags_from_kwargs(opts["hes_norm"], opts["hes_smth"], opts["mcc_norm"])


@pytest.mark.parametrize("name", VARIANTS)
def test_golden_reference_tables(gpu_ctx, golden_points, name):
    g = golden_points
    pts, s, alpha0, angles, opts, ref = variant_inputs(g, name)
    gpu_ctx.set_pair(g["img1"], g["img2"])
    got, status = gpu_ctx.run(*pts, s, angles, alpha0, opts["rot_order"], flags(opts), want_status=True)
    stats = classify(got, ref, make_exact_lookup(co, pts, g["img1"], g["img2"], s, alpha0, angles, opts))
    assert_parity(stats)
    exact, st2 = co.use_mcc_batch(*pts, g["img1"], g["img2"], s, alpha0, angles=angles, **opts)
    assert_equals_exact_oracle(got, exact, status, st2)


def test_golden_stage_vectors(gpu_ctx, golden_points, golden_stages):
    g = golden_stages
    for k, (c, r, ang, s, order) in enumerate(g["tpl_cases"]):
        got = gpu_ctx.get_template(g["img"], c, r, ang, int(s), int(order))
        assert np.array_equal(got, g["tpl_%d" % k]), "template case %d" % k
    for k in range(4):
        win, tpl, ref = g["mt_win_%d" % k], g["mt_tpl_%d" % k], g["mt_out_%d" % k]
        got = gpu_ctx.match_template(win, tpl)
        assert got.shape == ref.shape and got.dtype == np.float32
        assert np.abs(got - ref).max() < 1e-5                      # cv2's own float32 noise
        assert np.array_equal(got, co.match_template(win, tpl))    # exact oracle: bit-exact
        for hn, hs in ((1, 0), (0, 0), (1, 1), (0, 1)):
            h = gpu_ctx.get_hessian(ref, _lib.flags_from_kwargs(bool(hn), bool(hs), False))
            href = g["hes_%d_%d%d" % (k, hn, hs)]
            assert np.abs(h - href).max() <= 2e-6 * (1 + np.abs(href).max())
    p = golden_points
    angles = [-3, -2, -1, 0, 1, 2, 3]
    dc, dr, a, r, h, ccm, tpl = sid.rotate_and_match(p["img1"], 210.3, 120.6, 50, p["img2"][40:190, 130:300], -3.85,
                                                    angles=angles)
    ref = g["ram_scalars"]
    assert (dc, dr, a) == (ref[0], ref[1], ref[2])
    assert abs(r - ref[3]) < 1e-4 and abs(h - ref[4]) < 1e-4
    assert np.array_equal(tpl, g["ram_template"]) and np.abs(ccm - g["ram_result"]).max() < 1e-5


CASES = [
    dict(s=35, angles=[-3, 0, 3], border=(20, 50)),
    dict(s=35, angles=[0], border=(20, 20)),
    dict(s=35, angles=list(range(-10, 11)), border=(20, 24), n=150),
    dict(s=35, angles=[-3, 0, 3], border=(20, 28), rot_order=1, hes_smth=True),
    dict(s=35, angles=[-3, 3], border=(20, 22), hes_norm=False, mcc_norm=True),
    dict(s=50, angles=[-3, 0, 3], border=(20, 30)),
    dict(s=34, angles=[-2, 2], border=(23, 23), mcc_norm=True),
    dict(s=51, angles=[-3, 0, 3], border=(100, 100), n=120),
    dict(s=21, angles=[-3, 0, 3], border=(8, 14)),
    dict(s=64, angles=[0, 5], border=(30, 40), n=200),
    dict(s=9, angles=[0], border=(3, 6)),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "s%d_a%d_b%d-%d" % (c["s"], len(c["angles"]), c["border"][0], c["border"][1]))
def test_seeded_batches_equal_exact_oracle(gpu_ctx, case):
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=2, side=1500, grid=26)
    img1 = img1.copy()
    img1[690:770, 690:770] = 0                                      # NaN points
    rng = np.random.default_rng(9)
    n = min(case.get("n", len(c1)), len(c1))
    brd = np.floor(rng.uniform(case["border"][0], case["border"][1] + 1, len(c1)))[:n]
    pts = [x[:n] for x in (c1, r1, c2, r2)] + [brd]
    pts[2][:3] = [5.0, 1490.0, 700.0]                               # windows off the left / right edge
    opts = dict(rot_order=case.get("rot_order", 0), hes_norm=case.get("hes_norm", True),
                hes_smth=case.get("hes_smth", False), mcc_norm=case.get("mcc_norm", False))
    gpu_ctx.set_pair(img1, img2)
    got, st = gpu_ctx.run(*pts, case["s"], case["angles"], 1.5, opts["rot_order"], flags(opts), want_status=True)
    ref, st2 = co.use_mcc_batch(*pts, img1, img2, case["s"], 1.5, angles=case["angles"], **opts)
    assert_equals_exact_oracle(got, ref, st, st2)
    assert (st == -1).sum() >= 1 and (st == 1).sum() > n // 2


def test_known_answer_identical_images(gpu_ctx):
    """img2 == img1: every vector must sit at the reference's -1 px template-centre bias
    (pmlib.py:105) with r == 1 exactly and angle 0."""
    img = syn.speckle_image((900, 900), seed=4)
    c, r = np.meshgrid(np.arange(100.0, 800.0, 50.0), np.arange(100.0, 800.0, 50.0))
    c, r = c.ravel(), r.ravel()
    gpu_ctx.set_pair(img, img)
    out = gpu_ctx.run(c, r, c, r, np.full(c.size, 20.0), 35, [-3, 0, 3], 0.0)
    assert np.array_equal(out[:, 0], c - 1) and np.array_equal(out[:, 1], r - 1)
    assert np.all(out[:, 2] == 0) and np.all(out[:, 3] == 1.0) and np.all(out[:, 4] > 5)


def test_full_size_config2_properties_and_sample(gpu_ctx):
    """BASELINE configs[1] at full size (10400 x 10400, 200 x 200 grid, 3 angles)."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    assert img1.shape == (10400, 10400) and len(c1) > 39000
    gpu_ctx.set_pair(img1, img2)
    out = gpu_ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
    # determinism + independence of the processing order
    perm = np.random.default_rng(0).permutation(len(c1))
    out_p = gpu_ctx.run(c1[perm], r1[perm], c2[perm], r2[perm], b[perm], 35, cfg["angles"], 0.0)
    assert np.array_equal(out[perm], out_p, equal_nan=True)
    ok = ~np.isnan(out[:, 0])
    assert ok.mean() > 0.99
    assert np.all(np.abs(out[ok, 3]) <= 1.0) and np.all(np.isin(out[ok, 2], cfg["angles"]))
    assert np.all(np.abs(out[ok, 0] - c2[ok]) <= b[ok]) and np.all(np.abs(out[ok, 1] - r2[ok]) <= b[ok])
    tx, ty = syn.apply_affine(cfg["matrix"], c1, r1)           # known drift field, minus the -1 px bias
    assert np.median(np.abs(out[ok, 0] - (tx[ok] - 1))) < 0.6 and np.median(np.abs(out[ok, 1] - (ty[ok] - 1))) < 0.6
    assert np.median(out[ok, 3]) > 0.8
    # seeded sample against the exact oracle
    sel = np.random.default_rng(1).choice(len(c1), 1500, replace=False)
    ref, _ = co.use_mcc_batch(c1[sel], r1[sel], c2[sel], r2[sel], b[sel], img1, img2, 35, 0.0, angles=cfg["angles"])
    assert_equals_exact_oracle(out[sel], ref)


def test_full_size_config4_sample(gpu_ctx):
    """BASELINE configs[3]: img_size 51, search radius 100 (shared-memory window staging stress)."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg4", seed=0, side=4000, grid=40)
    gpu_ctx.set_pair(img1, img2)
    out = gpu_ctx.run(c1, r1, c2, r2, b, 51, cfg["angles"], 0.0)
    sel = np.random.default_rng(2).choice(len(c1), 60, replace=False)
    ref, _ = co.use_mcc_batch(c1[sel], r1[sel], c2[sel], r2[sel], b[sel], img1, img2, 51, 0.0, angles=cfg["angles"])
    assert_equals_exact_oracle(out[sel], ref)


def test_edge_cases_and_errors(gpu_ctx, golden_points):
    g = golden_points
    gpu_ctx.set_pair(g["img1"], g["img2"])
    out = gpu_ctx.run([], [], [], [], [], 35, [0], 0.0)
    assert out.shape == (0, 5)
    before = gpu_ctx.launch_count
    gpu_ctx.run([100.0], [100.0], [100.0], [100.0], [20.0], 35, [0], 0.0)
    assert gpu_ctx.launch_count > before and 0.0 < gpu_ctx.last_kernel_ms < 1000.0
    out, st = gpu_ctx.run([245.0, 100.0, 100.0, np.nan], [160.0, 100.0, 100.0, 100.0], [245.0, 10.0, 100.0, 100.0],
                          [160.0, 100.0, 100.0, 100.0], [20.0, 20.0, 20.0, 20.0], 35, [-3, 0, 3], 0.0, want_status=True)
    assert st.tolist() == [0, -1, 1, -1]
    assert np.isnan(out[[0, 1, 3]]).all() and not np.isnan(out[2]).any()
    with pytest.raises(ValueError):
        gpu_ctx.run([100.], [100.], [100.], [100.], [20.], 35, [0], 0.0, rot_order=3)
    with pytest.raises(ValueError):
        gpu_ctx.run([100.], [100.], [100.], [100.], [20.], 35, [0], 0.0, mtype=3)
    with pytest.raises(ValueError):
        gpu_ctx.run([100.], [100.], [100.], [100.], [20.], 300, [0], 0.0)
    fresh = _lib.Context(0)
    with pytest.raises(_lib.SidError):
        fresh.run([100.], [100.], [100.], [100.], [20.], 35, [0], 0.0)      # no pair yet
    fresh.close()
    with pytest.raises(ValueError):
        gpu_ctx.match_template(g["img1"][:20, :20], g["img1"][:30, :30])
    # pitched (non-contiguous rows) input views are accepted as they are
    view = g["img2"][40:190, 130:300]
    assert np.array_equal(gpu_ctx.match_template(view, view[20:70, 30:80]),
                          co.match_template(np.ascontiguousarray(view), np.ascontiguousarray(view[20:70, 30:80])))


def test_template_matcher_plugin(golden_points):
    import cv2
    g = golden_points
    win = g["img2"][100:175, 100:175]
    base = sid.rotate_and_match(g["img1"], 140.2, 139.7, 35, win, 0.0)
    same = sid.rotate_and_match(g["img1"], 140.2, 139.7, 35, win, 0.0, template_matcher=cv2.matchTemplate)
    gpu = sid.rotate_and_match(g["img1"], 140.2, 139.7, 35, win, 0.0, template_matcher=sid.match_template)
    calls = []

    def custom(image, templ, method):
        calls.append(templ.shape)
        return cv2.matchTemplate(image, templ, method)
    user = sid.rotate_and_match(g["img1"], 140.2, 139.7, 35, win, 0.0, template_matcher=custom)
    assert len(calls) == 3
    for other in (same, gpu, user):
        assert other[:3] == base[:3] and abs(other[3] - base[3]) < 1e-5 and abs(other[4] - base[4]) < 1e-3
    assert np.isnan(sid.rotate_and_match(g["img1"], 245.0, 160.0, 35, win, 0.0)[0])    # zero patch
    one = sid.use_mcc(140.2, 139.7, 138.0, 137.0, 20, g["img1"], g["img2"], 35, 0.0)
    ref = co.use_mcc_batch([140.2], [139.7], [138.0], [137.0], [20.0], g["img1"], g["img2"], 35, 0.0)[0][0]
    assert one[:3] == tuple(ref[:3]) and one[2] in (-3, 0, 3)


def test_pattern_matching_drop_in_end_to_end(monkeypatch):
    from tests.test_host_api import _scene, oracle_compute
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = _scene()
    with contextlib.redirect_stdout(io.StringIO()):
        gpu = sid.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, threads=5, angles=[-3, 0, 3])
    monkeypatch.setattr(sharding, "use_mcc_batch_sharded",
                        lambda *a, **k: oracle_compute(*a, **{kk: vv for kk, vv in k.items() if kk != "compute"}))
    with contextlib.redirect_stdout(io.StringIO()):
        cpu = sid.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, threads=5, angles=[-3, 0, 3])
    for a, b in zip(gpu, cpu):
        assert np.array_equal(np.isnan(a), np.isnan(b))
        assert np.nanmax(np.abs(a - b)) <= 1e-4
    drift = sid.SeaIceDrift(n1, n2)
    lon1, lat1 = n1.transform_points(kx, ky)
    lon2, lat2 = n2.transform_points(k2x, k2y)
    with contextlib.redirect_stdout(io.StringIO()):
        u = drift.get_drift_PM(lon, lat, lon1, lat1, lon2, lat2, angles=[-3, 0, 3])[0]
    assert np.array_equal(u, gpu[0], equal_nan=True)


def test_run_pair_overlapped_upload_equals_set_pair_then_run(gpu_ctx):
    """sid_run_pair (banded upload overlapped with compute) == sid_set_pair + sid_run, bit for bit."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=7, side=5200, grid=70)
    b = np.floor(np.random.default_rng(3).uniform(20, 41, b.size))
    gpu_ctx.set_pair(img1, img2)
    ref, st_ref = gpu_ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, want_status=True)
    other = np.ascontiguousarray(img1[::-1])                       # make the resident pair stale first
    gpu_ctx.set_pair(other, other)
    got, st = gpu_ctx.run_pair(img1, img2, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, want_status=True)
    assert np.array_equal(got, ref, equal_nan=True) and np.array_equal(st, st_ref)
    again = gpu_ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)       # the pair stays resident
    assert np.array_equal(again, ref, equal_nan=True)
    # pitched views of larger arrays are uploaded as they are
    big1 = np.zeros((5300, 5400), np.uint8); big1[50:5250, 100:5300] = img1
    big2 = np.zeros((5300, 5400), np.uint8); big2[50:5250, 100:5300] = img2
    got2 = gpu_ctx.run_pair(big1[50:5250, 100:5300], big2[50:5250, 100:5300], c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
    assert np.array_equal(got2, ref, equal_nan=True)
    empty = gpu_ctx.run_pair(img1, img2, [], [], [], [], [], 35, cfg["angles"], 0.0)
    assert empty.shape == (0, 5)


def test_run_pair_images_of_different_shapes_pinned_and_pageable(gpu_ctx):
    """Image 2 larger than image 1, image 1 cut short (its bottom grid points lose their template -> NaN rows), several
    upload bands with unequal row counts per image: the pageable path (NumPy memory, staged through the pinned
    double buffer by host threads) and the pinned path (direct DMA) both equal the exact oracle."""
    import torch
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=9, side=2300, grid=40)
    img2b = np.zeros((2600, 2450), np.uint8)
    img2b[:2300, :2300] = img2
    img1s = np.ascontiguousarray(img1[:2100])
    ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1s, img2b, 35, 0.0, angles=cfg["angles"])
    assert np.isnan(ref[:, 0]).any() and not np.isnan(ref[:, 0]).all()
    got_pageable = gpu_ctx.run_pair(img1s, img2b, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
    assert_equals_exact_oracle(got_pageable, ref)
    p1 = torch.from_numpy(img1s).pin_memory().numpy()
    p2 = torch.from_numpy(img2b).pin_memory().numpy()
    got_pinned = gpu_ctx.run_pair(p1, p2, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
    assert np.array_equal(got_pinned, got_pageable, equal_nan=True)
    for forced in ("1", "0"):                      # either upload path on either kind of memory
        os.environ["SID_STAGED_UPLOAD"] = forced
        try:
            a = gpu_ctx.run_pair(p1, p2, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
            bb = gpu_ctx.run_pair(img1s, img2b, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
        finally:
            del os.environ["SID_STAGED_UPLOAD"]
        assert np.array_equal(a, got_pageable, equal_nan=True) and np.array_equal(bb, got_pageable, equal_nan=True)


def test_sharded_pattern_matching_over_nccl_two_gpus():
    """Strong scaling path on real GPUs: 2 ranks, NCCL all-gather (skipped on a 1-GPU box)."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29577", os.path.join(root, "tests", "multi_gpu_sharded.py")]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:]
    assert "ranks) == single GPU: True" in res.stdout and "series(2 ranks) == single GPU: True" in res.stdout


def test_time_series_of_pairs_through_one_context(gpu_ctx):
    """BASELINE configs[4] in miniature: several pairs in sequence through one context (the pair buffers
    are reused); every pair must equal the exact oracle."""
    for seed in (11, 12, 13):
        img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=seed, side=900 + 64 * (seed - 11), grid=14)
        got = gpu_ctx.run_pair(img1, img2, c1, r1, c2, r2, b, 35, cfg["angles"], 0.0)
        ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=cfg["angles"])
        assert_equals_exact_oracle(got, ref)


def test_series_driver_two_contexts_equal_exact_oracle():
    """sharding.use_mcc_series on one GPU: pairs of different shapes and grid sizes worked through by two
    contexts concurrently (threads), one of them loaded lazily -- every table equals the exact oracle."""
    from sea_ice_drift_b200.sharding import use_mcc_series
    items = []
    for k in range(5):
        img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=30 + k, side=600 + 48 * k, grid=10 + 3 * k)
        items.append((img1, img2, c1, r1, c2, r2, b))
    pairs = list(items)
    pairs[3] = lambda: items[3]
    for n_contexts in (1, 2):
        tables = use_mcc_series(pairs, 35, 0.0, n_contexts=n_contexts, angles=[-3, 0, 3])
        assert len(tables) == 5
        for (img1, img2, c1, r1, c2, r2, b), got in zip(items, tables):
            ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=[-3, 0, 3])
            assert_equals_exact_oracle(got, ref)


@pytest.mark.parametrize("seed", range(10))
def test_randomised_configurations_equal_exact_oracle(gpu_ctx, seed):
    """Random image shapes (not multiples of 16), template sizes, per-point borders, angle lists, alpha0 and
    option flags, with points pushed against every image edge (far-edge windows are clipped like NumPy
    slices, near-edge ones rejected) -- everything must equal the exact CPU oracle."""
    rng = np.random.default_rng(1000 + seed)
    rows, cols = int(rng.integers(300, 700)), int(rng.integers(300, 700))
    img1 = syn.speckle_image((rows, cols), seed=seed)
    m = syn.rotation_matrix((rows, cols), float(rng.uniform(-3, 3)))
    m[0, 2] += rng.uniform(-6, 6)
    m[1, 2] += rng.uniform(-6, 6)
    img2 = syn.warp_pair(img1, m, seed=seed)
    if seed % 3 == 0:
        img1 = img1.copy()
        img1[rows // 3: rows // 3 + 25, cols // 2: cols // 2 + 30] = 0
    s = int(rng.choice([5, 8, 17, 24, 33, 35, 36, 41, 50, 51, 64]))
    n = 60
    bmax = int(rng.integers(3, 45))
    brd = np.floor(rng.uniform(max(1, bmax // 3), bmax + 1, n))
    c1 = rng.uniform(0, cols, n)
    r1 = rng.uniform(0, rows, n)
    tx, ty = syn.apply_affine(m, c1, r1)
    c2 = np.round(tx + rng.normal(0, 2, n))
    r2 = np.round(ty + rng.normal(0, 2, n))
    c2[:6] = [3, cols - 3, cols // 2, cols // 2, cols - s // 2 - 2, s]           # hug the edges
    r2[:6] = [rows // 2, rows // 2, 2, rows - 2, rows - s // 2 - 2, rows - s]
    angles = sorted(set(np.round(rng.uniform(-12, 12, int(rng.integers(1, 8))), 1).tolist()))
    alpha0 = float(rng.uniform(-5, 5))
    opts = dict(rot_order=int(rng.integers(0, 2)), hes_norm=bool(rng.integers(0, 2)),
                hes_smth=bool(rng.integers(0, 2)), mcc_norm=bool(rng.integers(0, 2)))
    pts = [c1, r1, c2, r2, brd]
    got, st = gpu_ctx.run_pair(img1, img2, *pts, s, angles, alpha0, opts["rot_order"], flags(opts), want_status=True)
    ref, st2 = co.use_mcc_batch(*pts, img1, img2, s, alpha0, angles=angles, **opts)
    assert_equals_exact_oracle(got, ref, st, st2)
    assert (st == 1).sum() >= 5


@pytest.mark.parametrize("seed", range(6))
def test_randomised_single_call_api_equals_exact_oracle(gpu_ctx, seed):
    rng = np.random.default_rng(2000 + seed)
    img = syn.speckle_image((int(rng.integers(120, 400)), int(rng.integers(120, 400))), seed=50 + seed)
    # template_matcher plug-in: non-square templates, image sizes not multiples of the tile
    th, tw = int(rng.integers(3, 70)), int(rng.integers(3, 70))
    H, W = int(rng.integers(th, img.shape[0] + 1)), int(rng.integers(tw, img.shape[1] + 1))
    y, x = int(rng.integers(0, img.shape[0] - H + 1)), int(rng.integers(0, img.shape[1] - W + 1))
    win = img[y:y + H, x:x + W]
    ty, tx = int(rng.integers(0, img.shape[0] - th + 1)), int(rng.integers(0, img.shape[1] - tw + 1))
    tpl = img[ty:ty + th, tx:tx + tw]
    assert np.array_equal(gpu_ctx.match_template(win, tpl),
                          co.match_template(np.ascontiguousarray(win), np.ascontiguousarray(tpl)))
    # get_hessian on maps of any shape >= 2 x 2
    rows, cols = int(rng.integers(2, 90)), int(rng.integers(2, 90))
    ccm = rng.normal(0, 0.3, (rows, cols)).astype(np.float32)
    for hn in (False, True):
        for hs in (False, True):
            got = gpu_ctx.get_hessian(ccm, _lib.flags_from_kwargs(hn, hs, False))
            ref = co.get_hessian(ccm, hes_norm=hn, hes_smth=hs)
            assert np.all(np.abs(got - ref) <= 4e-6 * (1 + np.abs(ref))), (rows, cols, hn, hs)
    # get_template anywhere, including partly outside the image
    for order in (0, 1):
        c, r, ang, s = rng.uniform(-10, img.shape[1] + 10), rng.uniform(-10, img.shape[0] + 10), rng.uniform(-180, 180), int(rng.integers(3, 80))
        assert np.array_equal(gpu_ctx.get_template(img, c, r, ang, s, order), co.get_template(img, c, r, ang, s, rot_order=order))
    # rotate_and_match against an explicit, non-square window
    s = int(rng.integers(5, 60))
    Hh, Ww = int(rng.integers(s + 2, s + 60)), int(rng.integers(s + 2, s + 60))
    img2 = syn.speckle_image((Hh, Ww), seed=90 + seed)
    angles = sorted(set(np.round(rng.uniform(-10, 10, int(rng.integers(1, 6))), 1).tolist()))
    c, r = rng.uniform(s, img.shape[1] - s), rng.uniform(s, img.shape[0] - s)
    kw = dict(rot_order=int(rng.integers(0, 2)), hes_norm=bool(rng.integers(0, 2)), hes_smth=bool(rng.integers(0, 2)))
    mcc = bool(rng.integers(0, 2))
    got = sid.rotate_and_match(img, c, r, s, img2, 1.1, angles=angles, mcc_norm=mcc, **kw)
    ref = co.rotate_and_match(img, c, r, s, img2, 1.1, angles=angles, mcc_norm=mcc, **kw)
    assert got[:3] == ref[:3]
    assert abs(got[3] - ref[3]) <= 4e-6 * (1 + abs(ref[3])) and abs(got[4] - ref[4]) <= 4e-6 * (1 + abs(ref[4]))
    assert np.array_equal(got[5], ref[5]) and np.array_equal(got[6], ref[6])


def test_image_narrower_than_tma_box_and_corner_windows(gpu_ctx):
    """The TMA box (window width rounded up + 15 bytes) can be wider than the whole image and can hang over the
    right / bottom edges: out-of-image bytes must read as zeros and never fault."""
    img1 = syn.speckle_image((88, 85), seed=3)
    img2 = syn.warp_pair(img1, syn.shift_matrix(1.0, -1.0), seed=3)
    c = np.array([42.0, 45.0, 46.3]); r = np.array([44.0, 47.0, 48.6])
    c2 = np.array([42.0, 46.0, 47.0]); r2 = np.array([44.0, 49.0, 50.0])
    b = np.array([20.0, 20.0, 20.0])
    got, st = gpu_ctx.run_pair(img1, img2, c, r, c2, r2, b, 35, [-3, 0, 3], 0.0, want_status=True)
    ref, st2 = co.use_mcc_batch(c, r, c2, r2, b, img1, img2, 35, 0.0, angles=[-3, 0, 3])
    assert_equals_exact_oracle(got, ref, st, st2)
    assert (st == 1).sum() >= 1


def test_series_honours_the_reference_defaults_and_flag_kwargs():
    """use_mcc_series without kwargs uses the reference's defaults (hes_norm=True, pmlib.py:36) and forwards
    hes_norm / hes_smth / mcc_norm / rot_order like use_mcc_batch does (round-1 advisor finding)."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=31, side=900, grid=12)
    pairs = [(img1, img2, c1, r1, c2, r2, b)]
    for kw in ({}, dict(hes_norm=False), dict(hes_smth=True), dict(mcc_norm=True, angles=[-3, 3]),
               dict(rot_order=1, hes_smth=True, mcc_norm=True)):
        table = sharding.use_mcc_series(pairs, 35, 0.0, **kw)[0]
        batch = sid.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, **kw)
        assert np.array_equal(table, batch, equal_nan=True), kw
        opts = dict(rot_order=kw.get("rot_order", 0), hes_norm=kw.get("hes_norm", True), hes_smth=kw.get("hes_smth", False),
                    mcc_norm=kw.get("mcc_norm", False))
        ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=kw.get("angles", [-3, 0, 3]), **opts)
        assert_equals_exact_oracle(table, ref)


def test_pair_is_uploaded_on_every_call_unless_resident_is_requested():
    """No identity guessing: an in-place edit of the image (masking, the usual step between two calls) is seen by the
    next call; resident=True is the explicit way to skip the upload."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=33, side=1024, grid=10)   # 1024 rows: the old sampled
    first = sid.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0)                            # checksum hit column 0 only
    img1 = img1.copy()
    img1[400:600, 400:600] = 0                                        # in-place style edit, same shape / dtype
    second = sid.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0)
    ref, _ = co.use_mcc_batch(c1, r1, c2, r2, b, img1, img2, 35, 0.0, angles=[-3, 0, 3])
    assert_equals_exact_oracle(second, ref)
    assert np.isnan(second[:, 0]).sum() > np.isnan(first[:, 0]).sum()
    again = sid.use_mcc_batch(c1, r1, c2, r2, b, None, None, 35, 0.0, resident=True)     # images not even passed
    assert np.array_equal(again, second, equal_nan=True)


def test_tcgen05_path_equals_legacy_paths_bit_for_bit(gpu_ctx):
    """The three correlation paths -- tcgen05.mma kind::i8 (default), mma.sync (SID_PM_PATH=imma) and the integer pipe
    (SID_PM_PATH=dp4a) -- must agree bit for bit, including x-tiled result maps, even sizes and 21-angle batches."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=35, side=1500, grid=22)
    rng = np.random.default_rng(2)
    gpu_ctx.set_pair(img1, img2)
    for s, angles, lo, hi in ((35, [-3, 0, 3], 20, 50), (50, [-2, 2], 20, 30), (35, list(range(-10, 11)), 20, 22), (51, [0], 60, 100)):
        brd = np.floor(rng.uniform(lo, hi + 1, len(c1)))
        tables = {}
        for path in ("tc", "imma", "dp4a"):
            os.environ["SID_PM_PATH"] = path
            try:
                tables[path] = gpu_ctx.run(c1, r1, c2, r2, brd, s, angles, 0.5)
            finally:
                del os.environ["SID_PM_PATH"]
        assert np.array_equal(tables["tc"], tables["imma"], equal_nan=True), (s, len(angles))
        assert np.array_equal(tables["tc"], tables["dp4a"], equal_nan=True), (s, len(angles))


def test_warp_specialised_path_equals_legacy_paths_bit_for_bit(gpu_ctx):
    """The warp-specialised pipeline kernel (pm_ws_kernel, the default for search radii <= 22 at img_size 35) against the mma.sync and
    tcgen05 row-loop kernels: every column of every row bit for bit, NaN rows and status included -- 1, 2, 3, 7 and 21
    angles (the screening of the angles must pick the reference's winner), even / odd / wide templates, mixed borders,
    a masked block (zero pixels -> NaN rows), bilinear sampling, raw Hessian and mcc_norm."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=36, side=1500, grid=24)
    img1 = img1.copy()
    img1[640:760, 700:820] = 0
    rng = np.random.default_rng(4)
    gpu_ctx.set_pair(img1, img2)
    # largest border the kernel's shared-memory layout takes with three sets of window statistics: 20 at (s 35, 3 angles per
    # batch), 22 at two angles, 24 at one, 14 at s 50, 13 at s 64; with two sets 22 / 24 / 24 / 15 / 14 -- every case below must
    # really run on pm_ws_kernel (asserted through sid_last_kernel_name)
    cases = ((35, [-3, 0, 3], 20, 20, {}), (35, [0], 8, 24, {}), (35, [-3, 3], 20, 22, dict(hes_norm=False, mcc_norm=True)),
             (35, list(range(-10, 11)), 14, 20, {}), (35, [-9, -6, -3, 0, 3, 6, 9], 10, 20, {}), (50, [-3, 0, 3], 8, 14, {}),
             (34, [-2, 2], 21, 21, dict(mcc_norm=True)), (21, [-3, 0, 3], 8, 14, {}), (64, [0, 5], 8, 13, {}), (9, [0], 3, 6, {}),
             (35, [-3, 0, 3], 16, 20, dict(rot_order=1, hes_smth=True)), (35, [2, 2, 2], 20, 20, {}),
             # two sets of window statistics instead of three (the layout for radius 21 ... 22 at img_size 35, 15 at 50)
             (35, [-3, 0, 3], 21, 22, {}), (35, list(range(-6, 7)), 19, 22, {}), (50, [-3, 0, 3], 15, 15, {}))
    for s, angles, lo, hi, kw in cases:
        brd = np.floor(rng.uniform(lo, hi + 1, len(c1)))
        flags = _lib.flags_from_kwargs(kw.get("hes_norm", True), kw.get("hes_smth", False), kw.get("mcc_norm", False))
        tables = {}
        for path in ("ws", "imma", "tc"):
            os.environ["SID_PM_PATH"] = path
            try:
                tables[path] = gpu_ctx.run(c1, r1, c2, r2, brd, s, angles, 0.5, kw.get("rot_order", 0), flags, want_status=True)
                if path == "ws":
                    assert gpu_ctx.last_kernel_name == "sid::pm_ws_kernel", (s, len(angles), hi, gpu_ctx.last_kernel_name)
            finally:
                del os.environ["SID_PM_PATH"]
        for other in ("imma", "tc"):
            assert np.array_equal(tables["ws"][0], tables[other][0], equal_nan=True), (s, len(angles), other)
            assert np.array_equal(tables["ws"][1], tables[other][1]), (s, len(angles), other)
        assert np.isnan(tables["ws"][0][:, 0]).any() and np.isfinite(tables["ws"][0][:, 0]).sum() > 400


def test_warp_specialised_kernel_is_the_default_for_small_search_radii(gpu_ctx):
    """Default dispatch: pm_ws_kernel where its geometry and shared-memory layout fit (radius <= 22 at img_size 35), the tcgen05 row-loop kernel or the mma.sync
    kernel otherwise -- all with the same table."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=37, side=1200, grid=16)
    gpu_ctx.set_pair(img1, img2)
    for border in (20.0, 40.0):
        brd = np.full(len(c1), border)
        default = gpu_ctx.run(c1, r1, c2, r2, brd, 35, [-3, 0, 3], 0.5)
        assert gpu_ctx.last_kernel_name == ("sid::pm_ws_kernel" if border == 20.0 else "sid::pm_tc_kernel")
        os.environ["SID_PM_PATH"] = "imma"
        try:
            legacy = gpu_ctx.run(c1, r1, c2, r2, brd, 35, [-3, 0, 3], 0.5)
        finally:
            del os.environ["SID_PM_PATH"]
        assert np.array_equal(default, legacy, equal_nan=True), border


def test_border_classes_send_small_maps_to_the_pipeline_kernel(gpu_ctx):
    """Borders as prepare_first_guess produces them (most points at the minimum of 20, a tail up to 45): the call is split
    into two launches per band -- the larger maps on the row-loop / mma.sync kernels, the rest on pm_ws_kernel -- and the
    table is bit for bit the single-launch one (SID_PM_CLASSES=0), resident and through the banded upload."""
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=41, side=2600, grid=40)
    rng = np.random.default_rng(8)
    brd = np.where(rng.random(len(c1)) < 0.86, 20.0, np.floor(rng.uniform(21, 46, len(c1))))
    brd[::97] = 20.5                                     # fractional borders: ceil() decides the class, the kernel the window
    assert (brd == 20).sum() > 1000 and brd.max() >= 44
    gpu_ctx.set_pair(img1, img2)
    for angles in ([-3, 0, 3], [0]):
        split, st_split = gpu_ctx.run(c1, r1, c2, r2, brd, 35, angles, 0.5, want_status=True)
        assert gpu_ctx.last_kernel_name.endswith("+ sid::pm_ws_kernel"), gpu_ctx.last_kernel_name
        os.environ["SID_PM_CLASSES"] = "0"
        try:
            single, st_single = gpu_ctx.run(c1, r1, c2, r2, brd, 35, angles, 0.5, want_status=True)
            assert "pm_ws_kernel" not in gpu_ctx.last_kernel_name
        finally:
            del os.environ["SID_PM_CLASSES"]
        assert np.array_equal(split, single, equal_nan=True) and np.array_equal(st_split, st_single)
        assert np.isfinite(split[:, 0]).sum() > 1400
    banded = gpu_ctx.run_pair(img1, img2, c1, r1, c2, r2, brd, 35, [0], 0.5)
    assert np.array_equal(banded, single, equal_nan=True)
    # device-resident point arrays (sid_run_device): the indices are split on the device
    import torch
    dev = torch.device("cuda", gpu_ctx.device)
    d_pts = torch.from_numpy(np.stack([c1, r1, c2, r2, brd])).to(dev)
    d_out = torch.full((len(c1), 5), -7.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    gpu_ctx.run_device(len(c1), *[d_pts[k].data_ptr() for k in range(5)], int(brd.max()), 35, [0], 0.5, d_out.data_ptr())
    assert gpu_ctx.last_kernel_name.endswith("+ sid::pm_ws_kernel"), gpu_ctx.last_kernel_name
    gpu_ctx.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), single, equal_nan=True)
    # too few small-map points for a launch of their own: one class
    few = np.where(np.arange(len(c1)) < 100, 20.0, 30.0)
    gpu_ctx.run(c1, r1, c2, r2, few, 35, [0], 0.5)
    assert "+" not in gpu_ctx.last_kernel_name


def test_device_epilogue_equals_host_post_processing():
    """SURVEY 8f rank 2: remainder add, pixel -> x/y / lon/lat, u/v differences and the _fill_gpi scatter on the device
    (sid_pm_epilogue_affine, table kept on the device) give the same seven grids, bit for bit, as the host lines that
    restate reference pmlib.py:462-497."""
    side = 900
    img1 = syn.speckle_image((side, side), seed=41)
    m = syn.rotation_matrix((side, side), 1.0)
    m[0, 2] += 3.3
    img2 = syn.warp_pair(img1, m, seed=41)
    n1 = syn.ArrayDomain(img1, lon0=5.0, lat0=81.0, rot_deg=7.0)
    n2 = syn.ArrayDomain(img2, lon0=5.0, lat0=81.0, rot_deg=7.0)
    rng = np.random.default_rng(8)
    kx, ky = rng.uniform(30, side - 30, 500), rng.uniform(30, side - 30, 500)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    gx, gy = np.meshgrid(np.linspace(-20, side + 20, 23) + 0.37, np.linspace(-20, side + 20, 21) + 0.21)   # some points outside
    lon, lat = n2.transform_points(gx, gy)
    with contextlib.redirect_stdout(io.StringIO()):
        dev = sid.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, angles=[-3, 0, 3])
        host = sid.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, angles=[-3, 0, 3], device_epilogue=False)
    assert np.isfinite(dev[0]).sum() > 100 and np.isnan(dev[0]).any()
    for name, a, b in zip("u v a r h lon2 lat2".split(), dev, host):
        assert a.shape == lon.shape and np.array_equal(a, b, equal_nan=True), name
    # the C entry point also accepts a host table
    ctx = _lib.default_context()
    gpi = np.isfinite(host[2]).ravel()
    c2pm1, r2pm1 = n2.transform_points(lon.ravel(), lat.ravel(), 1)
    table = np.column_stack([np.arange(gpi.sum(), dtype=np.float64)] * 5)
    grids = ctx.pm_epilogue_affine(gpi, c2pm1, r2pm1, *n2.affine_maps(), results=table)
    assert np.array_equal(grids[2][gpi], table[:, 2]) and np.isnan(grids[2][~gpi]).all()


def _fg_case(side, n_kp, grid, seed, integer_keypoints=False):
    rng = np.random.default_rng(seed)
    img = np.zeros((side, side), np.uint8)
    n1, n2 = syn.ArrayDomain(img), syn.ArrayDomain(img)
    m = syn.rotation_matrix((side, side), 1.5)
    m[0, 2] += 7.0
    kx, ky = rng.uniform(40, side - 40, n_kp), rng.uniform(40, side - 40, n_kp)
    if integer_keypoints:
        kx, ky = np.round(kx), np.round(ky)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    k2x, k2y = k2x + rng.normal(0, 0.8, n_kp), k2y + rng.normal(0, 0.8, n_kp)
    gx, gy = np.meshgrid(np.linspace(-30, side + 30, grid), np.linspace(-30, side + 30, grid))   # some points outside the hull / image
    return n1, n2, kx, ky, k2x, k2y, np.round(gx.ravel()), np.round(gy.ravel())


@pytest.mark.parametrize("old_border", [True, False])
def test_first_guess_on_device_equals_host_path(old_border):
    """SURVEY 8f rank 1: sid_first_guess (Delaunay-free local interpolation + exact nearest-keypoint distance) gives the
    same c2fg, r2fg, border as the SciPy path (Qhull triangulation + KD-tree) that equals the reference."""
    for side, n_kp, grid, seed in ((700, 400, 30, 1), (3000, 6000, 70, 2)):
        n1, n2, kx, ky, k2x, k2y, gx, gy = _fg_case(side, n_kp, grid, seed)
        dev = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, old_border=old_border, first_guess='device')
        host = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, old_border=old_border, first_guess='host')
        for name, a, b in zip(("c2fg", "r2fg", "border"), dev, host):
            assert np.array_equal(a, b, equal_nan=True), (name, side, int((a != b).sum()))


def test_first_guess_on_device_ew_size_and_interpolant_values():
    """EW size (10400 x 10400, 50 000 keypoints, 200 x 200 grid): identical outputs, and the raw interpolant agrees with
    scipy's LinearNDInterpolator to rounding error; timing printed for the record."""
    import time
    from scipy.interpolate import LinearNDInterpolator
    n1, n2, kx, ky, k2x, k2y, gx, gy = _fg_case(10400, 50000, 200, 3)
    sid.prepare_first_guess(gx[:10], gy[:10], n1, kx, ky, n2, k2x, k2y, 35, first_guess='device')       # warm-up
    t0 = time.perf_counter()
    dev = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, first_guess='device')
    t_dev = time.perf_counter() - t0
    t0 = time.perf_counter()
    host = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, first_guess='host')
    t_host = time.perf_counter() - t0
    print("prepare_first_guess EW size: device %.1f ms, host %.1f ms" % (1e3 * t_dev, 1e3 * t_host))
    for name, a, b in zip(("c2fg", "r2fg", "border"), dev, host):
        assert np.array_equal(a, b, equal_nan=True), (name, int((a != b).sum()))
    ctx = _lib.default_context()
    vx, vy, dist, flag = ctx.first_guess(kx, ky, k2x, k2y, np.uint16(k2x), np.uint16(k2y), gx, gy)
    ref = LinearNDInterpolator(np.column_stack([ky, kx]), np.column_stack([k2x, k2y]))(np.column_stack([gy, gx]))
    inside = ~np.isnan(ref[:, 0])
    assert np.array_equal(flag == 1, ~inside) and not np.any(flag >= 2)             # resolved and unique
    assert np.abs(vx[inside] - ref[inside, 0]).max() < 1e-7 and np.abs(vy[inside] - ref[inside, 1]).max() < 1e-7
    # timing is printed for the record only (typically 13 ms vs 380 ms): a first-time cudaMalloc of the larger staging block
    # inside the device call can take hundreds of milliseconds on a context that holds gigabytes from earlier tests


def test_first_guess_integer_keypoints_cocircular_degeneracies():
    """ORB keypoints of pyramid level 0 sit on integer pixels, so four of them can be cocircular and the Delaunay
    triangulation is then not unique (Qhull's choice is arbitrary too): the device result must still be a valid
    Delaunay interpolant -- the lifted-paraboloid check of tests/test_first_guess_geometry.py, whose expected value is
    the same over every valid triangulation of a cocircular cell."""
    from tests import test_first_guess_geometry as fgg
    n1, n2, kx, ky, k2x, k2y, gx, gy = _fg_case(1200, 3000, 60, 4, integer_keypoints=True)
    dev = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, first_guess='device')
    host = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35, first_guess='host')
    auto = sid.prepare_first_guess(gx, gy, n1, kx, ky, n2, k2x, k2y, 35)       # default: detects the ambiguity, SciPy decides
    for a, b in zip(auto, host):
        assert np.array_equal(a, b, equal_nan=True)
    flag = _lib.default_context().first_guess(kx, ky, k2x, k2y, kx, ky, gx, gy)[3]
    assert (flag == 3).any() and not (flag == 2).any()
    assert np.array_equal(dev[2], host[2])                                   # distances are exact either way
    fgg.add_layout("integer_keypoints", kx, ky, k2x, k2y, gx, gy)
    census = fgg.check_device(_lib.default_context(), "integer_keypoints", generic=False)
    assert census[3] > 0 and census[2] == 0
