"""Drift without feature tracking: ``sid_downsample_pair`` and ``pmlib.coarse_tracking``.

The downsampling rule is restated here in NumPy integers (``downsample_ref``); the "oracle composition" is that
restatement, the exact C oracle's ``use_mcc_batch`` on the lattice of ``pmlib.coarse_inputs`` and the selection and
full-resolution mapping restated below (``select_and_map``).  The CPU tests pin the restatement, the mapping (exact on
pairs shifted by multiples of the factor, for odd and even template sizes) and the accuracy on the scenes of DESIGN
section 8; the GPU tests hold the kernel byte for byte and ``coarse_tracking`` bit for bit to them."""
import numpy as np
import pytest

from sea_ice_drift_b200 import pmlib, synthetic as syn
from sea_ice_drift_b200.seaicedrift import SeaIceDrift


def downsample_ref(img, k):
    """k x k box downsampling: 0 if any source pixel of the block is 0, else (2 * sum + k*k) // (2 * k*k)."""
    img = np.asarray(img)
    h, w = img.shape[0] // k, img.shape[1] // k
    blk = img[:h * k, :w * k].reshape(h, k, w, k).astype(np.int64)
    total = blk.sum(axis=(1, 3))
    out = (2 * total + k * k) // (2 * k * k)
    out[(blk == 0).any(axis=(1, 3))] = 0
    return out.astype(np.uint8)


def select_and_map(table, status, c1, r1, k, img_size, min_quality):
    keep = (status == 1) & np.isfinite(table).all(axis=1)
    keep[keep] = table[keep, 3] * table[keep, 4] > min_quality
    delta = 1.0 if img_size % 2 else 1.5
    off = (k - 1) / 2.
    return (k * c1[keep] + off, k * r1[keep] + off, k * (table[keep, 0] + delta) + off,
            k * (table[keep, 1] + delta) + off)


def oracle_coarse(img1, img2, n1, n2, factor=4, step=16, img_size=35, max_drift=100.0, min_quality=4.0,
                  angles=(-3, 0, 3), seed=0):
    from oracle import c_oracle
    d1, d2 = downsample_ref(img1, factor), downsample_ref(img2, factor)
    c1, r1, c2fg, r2fg, border, alpha0 = pmlib.coarse_inputs(n1, n2, d1.shape, d2.shape, factor, step, img_size,
                                                             max_drift, seed)
    tab, st = c_oracle.use_mcc_batch(c1, r1, c2fg, r2fg, border, d1, d2, img_size, alpha0, angles=list(angles))
    got = select_and_map(tab, st, c1, r1, factor, img_size, min_quality)
    again = pmlib.coarse_matches(tab, st, c1, r1, factor, img_size, min_quality)
    for a, b in zip(got, again):
        assert np.array_equal(a, b)
    return got


def shifted_pair(side, k, a, b, seed=3):
    """img2 = img1 moved by exactly (k*a, k*b) px; uncovered pixels 0."""
    img1 = syn.speckle_image((side, side), seed)
    img2 = np.zeros_like(img1)
    dx, dy = k * a, k * b
    img2[max(dy, 0):side + min(dy, 0), max(dx, 0):side + min(dx, 0)] = \
        img1[max(-dy, 0):side - max(dy, 0), max(-dx, 0):side - max(dx, 0)]
    return img1, img2


PROBE = {
    "shift": syn.shift_matrix(57, -41),
    "rot2": syn.rotation_matrix((2400, 2400), 2.0),
    "rot-4": syn.rotation_matrix((2400, 2400), -4.0),
}
_probe_images = {}


def probe_pair(name, side=2400):
    if name not in _probe_images:
        img1 = syn.speckle_image((side, side), 3)
        _probe_images[name] = (img1, syn.warp_pair(img1, PROBE[name], 3))
    return _probe_images[name]


# ---------------------------------------------------------------- CPU: the rule, the mapping, the accuracy, refusals

def test_restatement_hand_cases():
    a = np.array([[1, 2, 3, 4, 9],
                  [3, 2, 5, 0, 9],
                  [7, 7, 8, 8, 9]], np.uint8)
    # blocks [[1, 2], [3, 2]] -> 8 / 4 = 2.0 -> 2; [[3, 4], [5, 0]] holds a 0 -> 0; last row and column dropped
    assert downsample_ref(a, 2).tolist() == [[2, 0]]
    assert downsample_ref(np.array([[1, 2]] * 2, np.uint8), 2).tolist() == [[2]]          # mean 1.5 rounds up
    assert downsample_ref(np.array([[1, 1], [1, 2]], np.uint8), 2).tolist() == [[1]]      # 1.25 -> 1
    assert downsample_ref(np.array([[1, 2], [2, 2]], np.uint8), 2).tolist() == [[2]]      # 1.75 -> 2
    assert downsample_ref(np.full((16, 16), 255, np.uint8), 16).tolist() == [[255]]
    assert downsample_ref(np.ones((3, 3), np.uint8), 3).tolist() == [[1]]
    assert downsample_ref(np.ones((2, 7), np.uint8), 3).shape == (0, 2)
    rng = np.random.default_rng(0)
    for k in (2, 3, 4, 8, 16):
        img = rng.integers(1, 256, (5 * k + k - 1, 7 * k + 1)).astype(np.uint8)
        img[rng.integers(0, img.shape[0], 3), rng.integers(0, img.shape[1], 3)] = 0
        got = downsample_ref(img, k)
        assert got.shape == (5, 7)
        blk = img[:5 * k, :7 * k].reshape(5, k, 7, k).astype(np.float64)
        want = np.floor(blk.mean(axis=(1, 3)) + 0.5)
        want[(blk == 0).any(axis=(1, 3))] = 0
        assert np.array_equal(got, want.astype(np.uint8)), k
        assert (got == 0).sum() >= 1


@pytest.mark.parametrize("img_size", [35, 34])
@pytest.mark.parametrize("k,a,b", [(4, 7, -5), (2, -9, 6)])
def test_exact_mapping_on_shift_by_multiple_of_factor(img_size, k, a, b):
    img1, img2 = shifted_pair(800, k, a, b)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    x1, y1, x2, y2 = oracle_coarse(img1, img2, n1, n2, factor=k, step=24, img_size=img_size, max_drift=12 * k)
    assert x1.size >= 20
    assert np.array_equal(x2 - x1, np.full(x1.size, float(k * a)))
    assert np.array_equal(y2 - y1, np.full(y1.size, float(k * b)))


@pytest.mark.parametrize("scene", ["shift", "rot2", "rot-4"])
def test_accuracy_factor4_within_factor(scene):
    img1, img2 = probe_pair(scene)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    x1, y1, x2, y2 = oracle_coarse(img1, img2, n1, n2, factor=4, step=32, img_size=25, max_drift=88)
    tx, ty = syn.apply_affine(PROBE[scene], x1, y1)
    err = np.hypot(x2 - tx, y2 - ty)
    assert x1.size >= 150
    assert err.max() <= 4.0, err.max()


def test_drift_beyond_reach_is_not_accepted():
    """factor 2, border 24 coarse px: reach 48 px, the drift (57, -41) is 70 px."""
    img1, img2 = probe_pair("shift")
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    x1, y1, x2, y2 = oracle_coarse(img1, img2, n1, n2, factor=2, step=48, img_size=25, max_drift=44)
    tx, ty = syn.apply_affine(PROBE["shift"], x1, y1)
    assert np.all(np.hypot(x2 - tx, y2 - ty) <= 2.0)


def test_lattice_and_inputs_follow_keywords():
    c, r = pmlib.coarse_lattice((300, 400), 16, 5)
    gx, gy = np.meshgrid(np.arange(8, 400, 16), np.arange(8, 300, 16))
    assert c.dtype == np.int64 and c.size == gx.size
    assert np.abs(c - gx.ravel()).max() <= 4 and np.abs(r - gy.ravel()).max() <= 4
    assert np.any(c != gx.ravel())
    c2, r2 = pmlib.coarse_lattice((300, 400), 16, 5)
    assert np.array_equal(c, c2) and np.array_equal(r, r2)            # seeded: deterministic
    assert not np.array_equal(c, pmlib.coarse_lattice((300, 400), 16, 6)[0])
    # no lattice cell is cocircular
    cc, rr = c.reshape(gx.shape), r.reshape(gx.shape)
    assert not pmlib._incircle_zero(cc[:-1, :-1], rr[:-1, :-1], cc[:-1, 1:], rr[:-1, 1:], cc[1:, 1:], rr[1:, 1:],
                                    cc[1:, :-1], rr[1:, :-1]).any()
    img = np.ones((1200, 1600), np.uint8)
    n1, n2 = syn.ArrayDomain(img), syn.ArrayDomain(img)
    for k, max_drift, s in ((4, 100.0, 35), (3, 50.0, 20), (8, 7.0, 9)):
        shape = (1200 // k, 1600 // k)
        c1, r1, c2fg, r2fg, border, alpha0 = pmlib.coarse_inputs(n1, n2, shape, shape, k, 16, s, max_drift)
        assert np.all(border == np.ceil(max_drift / k) + 2) and alpha0 == 0.0
        assert np.array_equal(c2fg, c1) and np.array_equal(r2fg, r1)  # identical geolocation: zero drift
        hws = round(s / 2) + 1
        lim = max(np.hypot(hws, hws), border[0] + hws)
        assert np.all(c1 > lim) and np.all(c1 < shape[1] - lim) and np.all(r1 > lim) and np.all(r1 < shape[0] - lim)
        lc, lr = pmlib.coarse_lattice(shape, 16, 0)
        inside = (lc > lim + 1) & (lc < shape[1] - lim - 1) & (lr > lim + 1) & (lr < shape[0] - lim - 1)
        assert c1.size >= inside.sum() > 0
    # a geolocation offset moves the first guess by the offset in coarse pixels
    n2s = syn.ArrayDomain(img, lon0=-40 * 1e-3)                       # image 2 starts 40 px further west
    c1, r1, c2fg, r2fg, _, _ = pmlib.coarse_inputs(n1, n2s, (300, 400), (300, 400), 4, 16, 35, 100.0)
    assert np.array_equal(c2fg, c1 + 10) and np.array_equal(r2fg, r1)


def test_refusals_before_any_device_work():
    img = syn.speckle_image((400, 400), 1)
    n1, n2 = syn.ArrayDomain(img), syn.ArrayDomain(img)
    for kw in (dict(factor=1), dict(factor=17), dict(factor=2.5), dict(factor=4, img_size=129),
               dict(factor=16, img_size=35), dict(factor=8, img_size=51), dict(step=2)):
        with pytest.raises(ValueError):
            pmlib.coarse_tracking(n1, n2, **kw)
    with pytest.raises(ValueError):
        SeaIceDrift(n1, n2).get_drift_coarse(factor=17)


def test_public_names():
    import sea_ice_drift_b200 as sid
    assert sid.coarse_tracking is pmlib.coarse_tracking
    assert pmlib.COARSE_DEFAULTS == dict(factor=4, step=32, img_size=35, max_drift=100.0, min_quality=4.0,
                                         angles=[-3, 0, 3], seed=0)


# ---------------------------------------------------------------- GPU

def _coarse_buffers(shapes):
    import torch
    from sea_ice_drift_b200 import _lib
    bufs = []
    for shape in shapes:
        pitch, nbytes = _lib.pair_layout(*shape)
        t = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda:0")      # the pitch padding stays 0xA5
        bufs.append((t, pitch, nbytes))
    return bufs


def _read(buf, shape):
    t, pitch, _ = buf
    return t[:pitch * shape[0]].view(shape[0], pitch).cpu().numpy()


def _pair_with_zeros(rows1, cols1, rows2, cols2, seed):
    rng = np.random.default_rng(seed)
    img1 = rng.integers(1, 256, (rows1, cols1)).astype(np.uint8)
    img2 = rng.integers(1, 256, (rows2, cols2)).astype(np.uint8)
    for img in (img1, img2):
        img[rng.integers(0, img.shape[0], 40), rng.integers(0, img.shape[1], 40)] = 0
        img[:, : img.shape[1] // 7] = np.where(rng.random((img.shape[0], img.shape[1] // 7)) < 0.02, 0,
                                               img[:, : img.shape[1] // 7])
    return img1, img2


def _check_downsample(ctx, img1, img2, k):
    shapes = [(img1.shape[0] // k, img1.shape[1] // k), (img2.shape[0] // k, img2.shape[1] // k)]
    bufs = _coarse_buffers(shapes)
    ctx.downsample_pair(k, *[(t.data_ptr(), p, n) for t, p, n in bufs])
    ctx.synchronize()
    for buf, shape, img in zip(bufs, shapes, (img1, img2)):
        got = _read(buf, shape)
        assert np.array_equal(got[:, :shape[1]], downsample_ref(img, k)), (k, shape)
        assert np.all(got[:, shape[1]:] == 0xA5)                         # nothing written past the columns
        assert np.all(buf[0][buf[1] * shape[0]:].cpu().numpy() == 0xA5)  # nor into the tail slack


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 4, 8])
def test_gpu_downsample_set_pair(k):
    from sea_ice_drift_b200 import _lib
    ctx = _lib.Context(0)
    for dims, seed in (((1037, 2203, 611, 1500), 1), ((8 * k + k - 1, 4099, 3 * k, 17 * k + 1), 2)):
        img1, img2 = _pair_with_zeros(*dims, seed)
        ctx.set_pair(img1, img2)
        _check_downsample(ctx, img1, img2, k)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 4, 8])
def test_gpu_downsample_run_pair_and_adopted(k):
    import torch
    from sea_ice_drift_b200 import _lib
    img1, img2 = _pair_with_zeros(2100, 1333, 1999, 2047, 10 + k)
    ctx = _lib.Context(0)
    ctx.run_pair(img1, img2, [600.], [600.], [600.], [600.], [20.], 35, [0.], 0.0)       # several upload bands
    _check_downsample(ctx, img1, img2, k)
    # adopted caller-owned buffers
    bufs = []
    for img in (img1, img2):
        pitch, nbytes = _lib.pair_layout(*img.shape)
        t = torch.zeros(nbytes, dtype=torch.uint8, device="cuda:0")
        t[:pitch * img.shape[0]].view(img.shape[0], pitch)[:, :img.shape[1]] = torch.from_numpy(img).cuda()
        bufs.append((t, pitch, nbytes))
    torch.cuda.synchronize()
    other = _lib.Context(0)
    (t1, p1, b1), (t2, p2, b2) = bufs
    other.adopt_pair_device(t1.data_ptr(), img1.shape, p1, b1, t2.data_ptr(), img2.shape, p2, b2)
    _check_downsample(other, img1, img2, k)
    other.close()
    ctx.close()


@pytest.mark.gpu
def test_gpu_downsample_refusals_leave_context_usable():
    from sea_ice_drift_b200 import _lib
    img1, img2 = _pair_with_zeros(401, 523, 390, 600, 3)
    ctx = _lib.Context(0)
    shapes = [(100, 130), (97, 150)]
    bufs = _coarse_buffers(shapes)
    ok = [(t.data_ptr(), p, n) for t, p, n in bufs]
    with pytest.raises(_lib.SidError, match=r"code -5"):
        ctx.downsample_pair(4, *ok)                                       # no pair resident
    ctx.set_pair(img1, img2)
    pts = ([150., 260., 330.], [120., 200., 280.], [152., 259., 331.], [121., 198., 282.], [20., 20., 20.])
    before = ctx.run(*pts, 35, [0.], 0.0)
    for k in (1, 17, 0, -4):
        with pytest.raises(ValueError, match=r"code -1"):
            ctx.downsample_pair(k, *ok)
    (p1, pitch1, n1), (p2, pitch2, n2) = ok
    for bad in (((p1, pitch1, n1 - 1), ok[1]), (ok[0], (p2, pitch2, n2 - 1)), ((p1, pitch1 - 16, n1), ok[1]),
                ((p1, pitch1 + 8, n1 + 4096), ok[1]), ((0, pitch1, n1), ok[1])):
        with pytest.raises(ValueError, match=r"code -1"):
            ctx.downsample_pair(4, *bad)
    small = _lib.Context(0)
    small.set_pair(np.ones((3, 40), np.uint8), np.ones((40, 40), np.uint8))
    with pytest.raises(ValueError, match=r"code -1"):
        small.downsample_pair(4, *ok)                                     # image 1 would be 0 x 10
    small.close()
    launches = ctx.launch_count
    _check_downsample(ctx, img1, img2, 4)
    assert ctx.launch_count == launches + 1
    # the resident pair is unchanged: the same points give the same rows as before the refusals
    after = ctx.run(*pts, 35, [0.], 0.0)
    assert np.array_equal(after, before, equal_nan=True)
    assert np.isfinite(before).any()
    ctx.close()


GPU_SCENES = [("shift", 4, 35), ("shift", 2, 34), ("rot-4", 4, 34), ("rot-4", 2, 35)]


@pytest.mark.gpu
@pytest.mark.parametrize("scene,k,img_size", GPU_SCENES)
def test_gpu_coarse_tracking_equals_oracle_composition(scene, k, img_size):
    img1, img2 = probe_pair(scene)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    kw = dict(factor=k, step=20 if k == 4 else 40, img_size=img_size, max_drift=120 if k == 4 else 60)
    got = pmlib.coarse_tracking(n1, n2, **kw)
    want = oracle_coarse(img1, img2, n1, n2, **kw)
    assert want[0].size >= 50
    for g, w in zip(got, want):
        assert g.dtype == np.float64 and np.array_equal(g, w)
    # cached buffers and the private context: a second call gives the same arrays
    again = pmlib.coarse_tracking(n1, n2, **kw)
    for g, w in zip(again, want):
        assert np.array_equal(g, w)


@pytest.mark.gpu
def test_gpu_coarse_tracking_ordered_after_torch_stream():
    """The coarse buffers are zero-filled on torch's current stream and written on the context's own stream: with work
    still queued on torch's stream when the buffers are allocated, the result must be the same."""
    import torch
    img1, img2 = probe_pair("shift")
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    kw = dict(factor=4, step=20, img_size=35, max_drift=120)
    want = oracle_coarse(img1, img2, n1, n2, **kw)
    pmlib._coarse_buffers.clear()
    torch.cuda._sleep(200_000_000)                  # keeps torch's stream busy for ~0.1 s
    got = pmlib.coarse_tracking(n1, n2, **kw)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


@pytest.mark.gpu
def test_gpu_drop_in_scene_coarse_route_vs_orb_route(monkeypatch):
    """cfg1 drop-in scene (2000 x 2000, drift (12, 12) px, 50 x 50 grid, angles [0], img_size 35): get_drift_PM fed by
    get_drift_coarse runs the device first guess and is at least as good as the ORB route against the known drift."""
    img1, img2, _, _, _, _, _, cfg = syn.make_config("cfg1", seed=0, side=2000)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(100, 1900, 50), np.linspace(100, 1900, 50))
    lon, lat = n2.transform_points(gx, gy)
    sid = SeaIceDrift(n1, n2)

    def errors(res):
        ok = np.isfinite(res[0])
        c2, r2 = n2.transform_points(res[5][ok], res[6][ok], 1)
        c1g, r1g = n1.transform_points(lon[ok], lat[ok], 1)
        tx, ty = syn.apply_affine(cfg["matrix"], c1g, r1g)
        return int(ok.sum()), np.hypot(c2 - (tx - 1), r2 - (ty - 1))

    x1, y1, x2, y2 = syn.orb_matches(img1, img2)
    orb = sid.get_drift_PM(lon, lat, *n1.transform_points(x1, y1), *n2.transform_points(x2, y2),
                           angles=[0], img_size=35)
    coarse_ll = sid.get_drift_coarse()
    assert coarse_ll[0].size >= 100

    def no_host_path(*a, **k):
        raise AssertionError("prepare_first_guess took the Qhull path")
    monkeypatch.setattr(pmlib, "interpolation_near", no_host_path)
    coarse = sid.get_drift_PM(lon, lat, *coarse_ll, angles=[0], img_size=35)
    n_orb, e_orb = errors(orb)
    n_coarse, e_coarse = errors(coarse)
    assert n_coarse >= n_orb
    assert np.median(e_coarse) <= np.median(e_orb)
