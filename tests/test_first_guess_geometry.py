"""The device first guess (``first_guess_kernel``, ``sid_first_guess``) against exact geometry.

The kernel finds every query's Delaunay triangle by pivoting, without a triangulation, and returns the interpolated
values, the distance to the nearest integer keypoint and a flag (0 ok, 1 outside the hull, 2 undecided, 3 ok but the
triangulation is not unique there).  ``prepare_first_guess(first_guess='auto')`` trusts that flag to choose between the
device result and SciPy.  Uniformly random keypoints (the content of the other first-guess tests) never reach most of
its branches, so the layouts here are built to: clustered keypoints with voids between them (starts from the hull fan),
far outliers (hundreds of keypoints in one hash cell), integer lattices (every cell cocircular, collinear hull sides),
a ring (huge, nearly cocircular circumcircles: the pivot cap), a 20000 x 3 px strip (the 2048-column cap of the hash
grid), duplicates, collinear and too few sources, ORB keypoints on an image with a large flat region, and queries on
source points, hull vertices, hull edges, circumcentres and just outside the hull, inside SciPy's tolerance band.
``test_layouts_reach_their_cases`` checks that the content still reaches those cases.

References, all independent of the code under test:
* the lifted paraboloid: with values f = |s - c|^2 the linear interpolant over any triangle that contains q is at least
  the lower convex hull of the lifted points, with equality exactly on Delaunay triangles, and every valid triangulation
  of a cocircular cell gives the same value.  So the expected value at q is unique even where the triangulation is not
  (flag 3, ``first_guess='device'``); it is computed in exact rational arithmetic over SciPy's simplex, after the
  triangulation itself has been verified to be Delaunay with exact in-circle determinants;
* linear precision: values equal to the coordinates must reproduce q;
* exact rational interpolation and the host path's ``LinearNDInterpolator`` at flag-0 queries with real value sets;
* brute-force int64 nearest-keypoint distances, compared bit for bit."""
import functools
import time
from fractions import Fraction

import numpy as np
import pytest
from scipy.interpolate import LinearNDInterpolator
from scipy.spatial import Delaunay, QhullError

import sea_ice_drift_b200 as sid
from sea_ice_drift_b200 import lib, pmlib, synthetic as syn

EPS = float(np.finfo(np.float64).eps)
SCIPY_EPS = 100 * EPS                      # scipy/spatial/_qhull.pyx: the barycentric tolerance of find_simplex
HULL_BAND_EPS = 2048 * EPS                 # csrc/sid_fg_kernel.cuh FG_HULL_BAND_EPS
ON_CIRCLE_TOL = 4e-14                      # csrc/sid_fg_kernel.cuh: |incircle| <= 4e-14 * (sa + sb + sc)^2 is "on the circle"


# ---------------------------------------------------------------------------------------------------- exact arithmetic
def exact_ints(*arrays):
    """Exact integer images of float arrays under one common power-of-two scale: (object arrays of Python ints, k) with
    every value multiplied by 2^k."""
    flat = np.concatenate([np.ravel(np.asarray(a, dtype=np.float64)) for a in arrays])
    nz = flat[flat != 0]
    k = int(max(0, (53 - np.frexp(nz)[1]).max())) if nz.size else 0
    out = []
    for a in arrays:
        o = np.empty(np.size(a), dtype=object)
        o[:] = [int(v) for v in np.ldexp(np.ravel(np.asarray(a, dtype=np.float64)), k)]
        out.append(o)
    return out, k


def orient(ax, ay, bx, by, cx, cy):
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)


def incircle(ax, ay, bx, by, cx, cy, dx, dy):
    """> 0 when d lies strictly inside the circumcircle of the counter-clockwise a, b, c."""
    adx, ady, bdx, bdy, cdx, cdy = ax - dx, ay - dy, bx - dx, by - dy, cx - dx, cy - dy
    ad, bd, cd = adx * adx + ady * ady, bdx * bdx + bdy * bdy, cdx * cdx + cdy * cdy
    return adx * (bdy * cd - bd * cdy) - ady * (bdx * cd - bd * cdx) + ad * (bdx * cdy - bdy * cdx)


def exact_hull(X, Y):
    """Convex hull (monotone chain, exact integer orientations), counter-clockwise, collinear and duplicate points dropped."""
    idx = sorted(range(len(X)), key=lambda i: (X[i], Y[i]))
    def chain(seq):
        h = []
        for i in seq:
            while len(h) >= 2 and orient(X[h[-2]], Y[h[-2]], X[h[-1]], Y[h[-1]], X[i], Y[i]) <= 0:
                h.pop()
            h.append(i)
        return h
    lo, hi = chain(idx), chain(idx[::-1])
    return np.array(lo[:-1] + hi[:-1], dtype=np.int64)


@functools.lru_cache(maxsize=None)
def delaunay_exact(name):
    """SciPy's triangulation of a layout's sources, with every simplex made counter-clockwise and every interior edge
    verified Delaunay with exact in-circle determinants.  Returns (tri, simplices, X, Y, quad_ratio) where quad_ratio is
    |incircle| / (sa + sb + sc)^2 over the interior edges (0 for exactly cocircular quads)."""
    L = layout(name)
    sx, sy = L["sx"], L["sy"]
    (X, Y), _ = exact_ints(sx, sy)
    tri = Delaunay(np.column_stack([sx, sy]))
    simp = tri.simplices.copy()
    neigh = tri.neighbors.copy()
    o = orient(X[simp[:, 0]], Y[simp[:, 0]], X[simp[:, 1]], Y[simp[:, 1]], X[simp[:, 2]], Y[simp[:, 2]])
    assert all(v != 0 for v in o), "degenerate simplex"
    cw = np.array([v < 0 for v in o])
    simp[cw] = simp[cw][:, [0, 2, 1]]
    neigh[cw] = neigh[cw][:, [0, 2, 1]]
    t, j = np.nonzero(neigh >= 0)
    keep = neigh[t, j] > t
    t, j = t[keep], j[keep]
    n = neigh[t, j]
    # the vertex of n that is not in t
    dv = np.array([[v for v in simp[nn] if v not in simp[tt]][0] for tt, nn in zip(t, n)], dtype=np.int64)
    a, b, c = simp[t, 0], simp[t, 1], simp[t, 2]
    v = incircle(X[a], Y[a], X[b], Y[b], X[c], Y[c], X[dv], Y[dv])
    assert all(x <= 0 for x in v), "SciPy's triangulation is not Delaunay in exact arithmetic"
    dd = lambda p: (X[p] - X[dv]) ** 2 + (Y[p] - Y[dv]) ** 2
    s = dd(a) + dd(b) + dd(c)
    ratio = np.array([abs(float(x)) / float(y * y) if y else 0.0 for x, y in zip(v, s)])
    return tri, simp, neigh, X, Y, ratio


def exact_values(name, qx, qy, value_sets):
    """Exact Delaunay-linear interpolation at the queries: for every query SciPy places in a simplex, the simplex that
    contains it in exact arithmetic (a walk over neighbours from SciPy's), and the value of every set in
    ``value_sets`` there, rounded once from the exact rational.  Returns (inside, simplex, values, kappa) where inside is
    True where the exact walk ends in a triangle (False also for points SciPy accepts just outside the hull) and kappa
    is the triangle's 2 * L^2 / |2 area| (L its longest edge), the conditioning of its barycentric weights."""
    tri, simp, neigh, X, Y = delaunay_exact(name)[:5]
    L = layout(name)
    (X, Y, QX, QY), _ = exact_ints(L["sx"], L["sy"], qx, qy)
    s = tri.find_simplex(np.column_stack([qx, qy]))
    inside = np.zeros(qx.size, bool)
    for k in np.nonzero(s >= 0)[0]:
        t = s[k]
        for _ in range(64):
            a, b, c = simp[t]
            w = (orient(X[b], Y[b], X[c], Y[c], QX[k], QY[k]), orient(X[c], Y[c], X[a], Y[a], QX[k], QY[k]),
                 orient(X[a], Y[a], X[b], Y[b], QX[k], QY[k]))
            neg = [i for i in range(3) if w[i] < 0]
            if not neg:
                inside[k] = True
                break
            t = neigh[t, neg[0]]
            if t < 0:
                break
        else:
            raise AssertionError("exact walk did not converge")
        s[k] = t
    idx = np.nonzero(inside)[0]
    a, b, c = simp[s[idx], 0], simp[s[idx], 1], simp[s[idx], 2]
    qxi, qyi = QX[idx], QY[idx]
    wa = orient(X[b], Y[b], X[c], Y[c], qxi, qyi)
    wb = orient(X[c], Y[c], X[a], Y[a], qxi, qyi)
    wc = orient(X[a], Y[a], X[b], Y[b], qxi, qyi)
    area = wa + wb + wc
    out = []
    for vals in value_sets:
        (V,), kv = exact_ints(vals)
        num = wa * V[a] + wb * V[b] + wc * V[c]
        res = np.full(qx.size, np.nan)
        res[idx] = [n / (d << kv) for n, d in zip(num, area)]       # int / int: correctly rounded
        out.append(res)
    pts = np.column_stack([L["sx"], L["sy"]])
    kappa = np.full(qx.size, np.nan)
    e = lambda i, j: np.sum((pts[i] - pts[j]) ** 2, axis=1)
    l2 = np.maximum(np.maximum(e(a, b), e(b, c)), e(c, a))
    kappa[idx] = 2 * l2 / np.abs(orient(pts[a, 0], pts[a, 1], pts[b, 0], pts[b, 1], pts[c, 0], pts[c, 1]))
    return inside, np.where(inside, s, -1), out, kappa


def interp_tol(vals, simplex_vals, kappa):
    """Rounding bound of the kernel's weighted sum wa * fa + wb * fb + wc * fc, wc = 1 - wa - wb, against the exact value.
    The weights are orientations over the area: each orientation rounds coordinate differences, two products and their
    difference, all bounded by L^2 (q lies in the triangle), so |dw| <= 3 eps L^2 / |2 area| + eps / 2 <= (1.5 kappa +
    0.5) eps for wa and wb, and wc adds 2 eps.  As sum(w) = 1 is kept up to that, the value errs by
    dwa (fa - fc) + dwb (fb - fc) + dwc fc plus the rounding of three products and two sums (<= 2.5 eps max|f|, w >= 0):
    <= eps ((3 kappa + 1) spread + 4.5 max|f|), spread = the largest difference of the triangle's values.  Doubled:
    eps (8 kappa spread + 9 max|f|).  A wrong triangle with a keypoint inside its circumcircle by delta px is off by
    about 2 R delta times a barycentric weight, far above this."""
    spread = np.ptp(simplex_vals, axis=1)
    return EPS * (8 * kappa * spread + 9 * np.abs(vals).max())


# ---------------------------------------------------------------------------------------------------- layouts
def _values(sx, sy, rng):
    """Feature-tracking end points for the sources (the k2x, k2y analogues): 1.5 deg rotation, shift, 0.8 px noise."""
    m = syn.rotation_matrix((1000, 1000), 1.5)
    m[:, 2] += (60.0, 45.0)
    vx, vy = syn.apply_affine(m, sx, sy)
    return vx + rng.normal(0, 0.8, sx.size), vy + rng.normal(0, 0.8, sx.size)


def _grid(sx, sy, nx, ny):
    gx, gy = np.meshgrid(np.round(np.linspace(sx.min() - 30, sx.max() + 30, nx)),
                         np.round(np.linspace(sy.min() - 30, sy.max() + 30, ny)))
    return gx.ravel(), gy.ravel()


def _blobs(rng, n_per, sigma, frame=4000):
    centres = rng.uniform(0.2 * frame, 0.8 * frame, (len(n_per), 2))
    return np.concatenate([rng.normal(c, s, (n, 2)) for c, n, s in zip(centres, n_per, sigma)])


def _band_candidates(sx, sy, hull):
    """Points a tiny distance (1e-15 ... 1e-8 px) outside every hull edge of a small integer layout near the origin,
    close to the edge's lower-left end where the coordinates are small enough to resolve such offsets."""
    out = []
    for k in range(hull.size):
        a, b = hull[k], hull[(k + 1) % hull.size]
        ax, ay, bx, by = sx[a], sy[a], sx[b], sy[b]
        if ax + ay > bx + by:
            ax, ay, bx, by = bx, by, ax, ay
        ex, ey = bx - ax, by - ay
        ln = np.hypot(ex, ey)
        nx_, ny_ = ey / ln, -ex / ln
        if nx_ * (ax - sx.mean()) + ny_ * (ay - sy.mean()) < 0:    # outward
            nx_, ny_ = -nx_, -ny_
        for s in (1e-3, 3e-3, 1e-2, 0.3):
            for d in (1e-15, 3e-15, 1e-14, 3e-14, 1e-13, 3e-13, 1e-12, 3e-12, 1e-11, 1e-9, 1e-8):
                out.append((ax + s * ex + d * nx_, ay + s * ey + d * ny_))
    return np.array(out)


_LAYOUTS = {}


def layout(name):
    """A layout by name: built on first use (ORB layouts need the GPU matcher) or registered by ``add_layout``."""
    if name not in _LAYOUTS:
        _LAYOUTS[name] = orb_layout(float(name[3:])) if name.startswith("orb") else seeded_layout(name)
    return _LAYOUTS[name]


def add_layout(name, sx, sy, vx, vy, qx, qy):
    """Register sources, values and queries built elsewhere as a layout (seeds: the values as uint16)."""
    cx, cy = np.round(np.mean(sx)), np.round(np.mean(sy))
    _LAYOUTS[name] = dict(sx=sx, sy=sy, vx=vx, vy=vy, kx=np.uint16(vx).astype(np.float64),
                          ky=np.uint16(vy).astype(np.float64), qx=qx, qy=qy, f=(sx - cx) ** 2 + (sy - cy) ** 2,
                          integer=False, n_band=0)
    delaunay_exact.cache_clear()
    return _LAYOUTS[name]


def seeded_layout(name):
    """Seeded layout: sources sx, sy (interpolation sources), values vx, vy, seeds kx, ky (uint16 keypoints of image 2),
    queries qx, qy (an integer grid over the layout +- 30 px, plus constructed queries), and what the layout is for."""
    rng = np.random.default_rng(sum(map(ord, name)))
    integer, extra = False, []
    if name == "blobs":
        P = _blobs(rng, (500, 1200, 2000, 3000), (25, 40, 60, 80))
    elif name == "blobs_int":
        P = np.unique(np.round(_blobs(rng, (500, 1200, 2000), (25, 50, 80))), axis=0)
        integer = True
    elif name == "blobs_outliers":
        P = np.concatenate([_blobs(rng, (800, 1500), (25, 30)),
                            [[20.5, 31.25], [30000.5, 12.0], [17.0, 29990.75], [29980.0, 30010.5], [15000.25, 40.5]]])
    elif name == "lattice":
        g = np.arange(40) * 7.0 + 100
        P = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
        integer = True
    elif name == "lattice_gap":
        g = np.arange(40) * 7.0 + 100
        P = np.stack(np.meshgrid(g, np.delete(g, 20)), -1).reshape(-1, 2)
        integer = True
    elif name == "ring":
        th = np.sort(rng.uniform(0, 2 * np.pi, 2000))
        P = np.unique(np.round(np.column_stack([5000 * np.cos(th), 5000 * np.sin(th)]) + 5040), axis=0)
        integer = True
    elif name == "strip":
        P = np.column_stack([rng.uniform(40, 20040, 4000), rng.uniform(40, 43, 4000)])
    elif name == "duplicates":
        P = rng.uniform(40, 2040, (3000, 2))
        P = np.concatenate([P, P[rng.choice(3000, 150, replace=False)]])
    elif name == "band":
        # small integer polygon at the origin: a slanted hull edge through (0, 0) and one on the bounding box (x = 0)
        P = np.concatenate([[[0, 0], [1000, 200], [800, 1000], [0, 700]],
                            np.round(rng.uniform(0, 1, (300, 2)) * (700, 600) + (50, 180))]).astype(np.float64)
        integer = True
    elif name == "collinear":
        t = np.arange(200.0)
        P = np.column_stack([60 + 3 * t, 50 + 2 * t])
        integer = True
    elif name == "two":
        P = np.array([[100.0, 120.0], [300.0, 310.0]])
        integer = True
    else:
        raise KeyError(name)
    sx, sy = np.ascontiguousarray(P[:, 0]), np.ascontiguousarray(P[:, 1])
    vx, vy = _values(sx, sy, rng)
    if name == "duplicates":
        vx[3000:] += 5.0                                   # same position, different value
    nx, ny = (400, 5) if name == "strip" else (60, 60)
    qx, qy = _grid(sx, sy, nx, ny)
    if name == "blobs_outliers":                          # the coarse grid misses the clusters: add a fine one over them
        core = P[:-5]
        fx, fy = _grid(core[:, 0], core[:, 1], 50, 50)
        qx, qy = np.concatenate([qx, fx]), np.concatenate([qy, fy])
    qx = np.concatenate([qx, [-900.0, 45000.0, 3.0]])      # far outside the seeds' bounding box: clamped hash cells
    qy = np.concatenate([qy, [-700.0, 52000.0, 61000.0]])
    band = np.zeros((0, 2))
    if P.shape[0] >= 3 and name not in ("collinear",):
        pick = rng.choice(sx.size, min(200, sx.size), replace=False)
        extra.append(np.column_stack([sx[pick], sy[pick]]))                  # on source points
        tri = Delaunay(P)
        hull = np.unique(tri.convex_hull)
        extra.append(P[hull])                                                   # on hull vertices
        if integer:                                                             # on hull-edge midpoints (exact)
            e = tri.convex_hull
            extra.append((P[e[:, 0]] + P[e[:, 1]]) / 2)
        ts = tri.simplices[rng.choice(len(tri.simplices), min(300, len(tri.simplices)), replace=False)]
        A, B, C = P[ts[:, 0]], P[ts[:, 1]], P[ts[:, 2]]                        # circumcentres
        b, c = B - A, C - A
        d = 2 * (b[:, 0] * c[:, 1] - b[:, 1] * c[:, 0])
        ux = (c[:, 1] * (b ** 2).sum(1) - b[:, 1] * (c ** 2).sum(1)) / d
        uy = (b[:, 0] * (c ** 2).sum(1) - c[:, 0] * (b ** 2).sum(1)) / d
        extra.append(A + np.column_stack([ux, uy]))
        if name == "band":
            band = _band_candidates(sx, sy, exact_hull(*exact_ints(sx, sy)[0]))
            extra.append(band)
    if extra:
        E = np.concatenate(extra)
        qx, qy = np.concatenate([qx, E[:, 0]]), np.concatenate([qy, E[:, 1]])
    kx, ky = np.uint16(vx).astype(np.float64), np.uint16(vy).astype(np.float64)
    cx, cy = np.round(sx.mean()), np.round(sy.mean())
    f = (sx - cx) ** 2 + (sy - cy) ** 2
    return dict(sx=sx, sy=sy, vx=vx, vy=vy, kx=kx, ky=ky, qx=qx, qy=qy, f=f, integer=integer, n_band=len(band))


GEOMETRIC = ("blobs", "blobs_int", "blobs_outliers", "lattice", "lattice_gap", "ring", "strip", "duplicates", "band")
# float coordinates: no cocircular cells (duplicates lie on every circle through their twin, so they may give flag 3)
GENERIC = ("blobs", "blobs_outliers", "strip")
DEGENERATE = ("collinear", "two")


def kernel_grid(px, py):
    """(cell, nx, ny, points in the fullest cell) of the kernel's hash grid over a point set (build_grid in sid_api.cu)."""
    n = px.size
    w, h = max(px.max() - px.min(), 1.0), max(py.max() - py.min(), 1.0)
    cell = max(np.sqrt(w * h * 2.0 / max(n, 1)), 1.0)
    nx, ny = min(2048, max(1, int(np.ceil(w / cell)) + 1)), min(2048, max(1, int(np.ceil(h / cell)) + 1))
    cell = max(cell, w / (nx - 0.5), h / (ny - 0.5))
    ix = np.clip(np.floor((px - px.min()) / cell).astype(np.int64), 0, nx - 1)
    iy = np.clip(np.floor((py - py.min()) / cell).astype(np.int64), 0, ny - 1)
    return cell, nx, ny, np.bincount(iy * nx + ix).max()


def nearest_seed_distance(kx, ky, qx, qy):
    """Brute-force exact int64 minimum of dx^2 + dy^2 over the uint16 seeds, then sqrt (integer queries only)."""
    K = np.column_stack([np.uint16(kx).astype(np.int64), np.uint16(ky).astype(np.int64)])
    Q = np.column_stack([qx.astype(np.int64), qy.astype(np.int64)])
    best = np.empty(len(Q), np.int64)
    for i in range(0, len(Q), 512):
        d = Q[i:i + 512, None, :] - K[None, :, :]
        best[i:i + 512] = (d * d).sum(-1).min(1)
    return np.sqrt(best.astype(np.float64))


def scipy_nan(name):
    """Where the host path (LinearNDInterpolator over (y, x), as pmlib.lib.interpolation_near) returns NaN."""
    L = layout(name)
    return np.isnan(lib.interpolation_near(L["sx"], L["sy"], L["vx"], L["vy"], L["qx"], L["qy"])[0])


def hull_distance(name, idx):
    """Signed distance (px, negative outside) of queries ``idx`` from the exact hull of the sources: the smallest
    exact orientation against a hull edge over the edge's length."""
    L = layout(name)
    (X, Y, QX, QY), k = exact_ints(L["sx"], L["sy"], L["qx"][idx], L["qy"][idx])
    h = exact_hull(X, Y)
    a, b = h, np.roll(h, -1)
    ln = np.hypot(L["sx"][b] - L["sx"][a], L["sy"][b] - L["sy"][a])
    return np.array([min(float(Fraction(o, 4 ** k)) / e for o, e in zip(orient(X[a], Y[a], X[b], Y[b], QX[j], QY[j]), ln))
                     for j in range(len(idx))])


def fan_start_queries(name):
    """Queries inside the hull where no triple of the FG_NEAR = 12 nearest sources contains q: the kernel starts these
    from the hull fan (deep inside a void)."""
    from itertools import combinations
    from scipy.spatial import cKDTree
    L = layout(name)
    P, Q = np.column_stack([L["sx"], L["sy"]]), np.column_stack([L["qx"], L["qy"]])
    Q = Q[Delaunay(P).find_simplex(Q) >= 0]
    nb = cKDTree(P).query(Q, 12)[1]
    found = np.zeros(len(Q), bool)
    o = lambda a, b, c: (b[:, 0] - a[:, 0]) * (c[:, 1] - a[:, 1]) - (b[:, 1] - a[:, 1]) * (c[:, 0] - a[:, 0])
    for i, j, k in combinations(range(12), 3):
        a, b, c = P[nb[:, i]], P[nb[:, j]], P[nb[:, k]]
        s = np.sign(o(a, b, c))
        found |= (s != 0) & (s * o(a, b, Q) >= 0) & (s * o(b, c, Q) >= 0) & (s * o(c, a, Q) >= 0)
    return int((~found).sum())


# ---------------------------------------------------------------------------------------------------- CPU: references
@pytest.mark.parametrize("name", ("lattice", "blobs", "ring", "band"))
def test_exact_oracle_against_scipy(name):
    """The exact oracle reproduces the coordinates exactly (linear precision of rational interpolation), and agrees with
    the host path's LinearNDInterpolator to a few ulps of the value scale on the paraboloid and on the real values."""
    L = layout(name)
    t0 = time.perf_counter()
    inside, simplex, (ef, ex, ey, evx), kappa = exact_values(name, L["qx"], L["qy"], (L["f"], L["sx"], L["sy"], L["vx"]))
    print("%s: exact oracle on %d queries (%d inside) in %.2f s" % (name, inside.size, inside.sum(), time.perf_counter() - t0))
    assert inside.sum() > 1000
    assert np.array_equal(ex[inside], L["qx"][inside]) and np.array_equal(ey[inside], L["qy"][inside])
    simp = delaunay_exact(name)[1]
    for vals, exact in ((L["f"], ef), (L["vx"], evx)):
        host = LinearNDInterpolator(np.column_stack([L["sx"], L["sy"]]), vals)(np.column_stack([L["qx"], L["qy"]]))
        tol = host_tol(vals, vals[simp[simplex[inside]]], kappa[inside])
        err = np.abs(host[inside] - exact[inside])
        print("  max |scipy - exact| = %.3g, %.3g of the tolerance" % (err.max(), (err / tol).max()))
        assert np.all(err <= tol)


def host_tol(vals, simplex_vals, kappa):
    """SciPy's own rounding: its barycentric transform is an inverted 2 x 2 matrix (relative error ~ eps * kappa), applied
    to q - r; bounded here as twice the kernel's bound with kappa^2 in place of kappa."""
    return 2 * interp_tol(vals, simplex_vals, kappa * kappa)


def test_nearest_seed_reference_pinned():
    """The brute-force int64 distance equals pmlib._distance_at (KD-tree) and the full EDT of
    get_distance_to_nearest_keypoint, at every pixel of a small image, with seeds on duplicate and edge pixels."""
    rng = np.random.default_rng(5)
    shape = (90, 130)
    x = np.concatenate([rng.uniform(0, 129.99, 40), [0.0, 129.0, 129.5, 7.2, 7.9]])
    y = np.concatenate([rng.uniform(0, 89.99, 40), [0.0, 89.0, 0.25, 3.0, 3.4]])
    gy, gx = np.mgrid[0:shape[0], 0:shape[1]]
    ref = nearest_seed_distance(x, y, gx.ravel(), gy.ravel())
    assert np.array_equal(ref, pmlib._distance_at(x, y, gx.ravel().astype(np.int16), gy.ravel().astype(np.int16)))
    assert np.array_equal(ref, pmlib.get_distance_to_nearest_keypoint(x, y, shape).ravel())


def test_layouts_reach_their_cases():
    """The content reaches the cases it is built for, so it cannot drift back to benign data."""
    # lattices: exactly cocircular cells, collinear points on the hull sides
    for name in ("lattice", "lattice_gap", "ring"):
        ratio = delaunay_exact(name)[5]
        L = layout(name)
        print("%s: %d exactly cocircular quads of %d" % (name, int((ratio == 0).sum()), ratio.size))
        if name != "ring":
            assert (ratio == 0).sum() > 1000
            assert exact_hull(*exact_ints(L["sx"], L["sy"])[0]).size == 4
            assert np.unique(Delaunay(np.column_stack([L["sx"], L["sy"]])).convex_hull).size > 100
    # ring: a quarter of the points or more on the hull
    L = layout("ring")
    assert exact_hull(*exact_ints(L["sx"], L["sy"])[0]).size > 0.25 * L["sx"].size
    # generic float layouts: no quad of the triangulation within the kernel's on-circle tolerance
    for name in GENERIC + ("duplicates",):
        ratio = delaunay_exact(name)[5]
        print("%s: smallest |incircle| / (sa + sb + sc)^2 over the quads: %.3g" % (name, ratio.min()))
        assert ratio.min() > 100 * ON_CIRCLE_TOL
    # voids: starts from the hull fan
    for name in ("blobs", "blobs_int", "ring"):
        n = fan_start_queries(name)
        print("%s: %d queries start from the hull fan" % (name, n))
        assert n >= 20
    # hash grid: hundreds of sources in one cell; the 2048-column cap
    L = layout("blobs_outliers")
    assert kernel_grid(L["sx"], L["sy"])[3] >= 200
    L = layout("strip")
    assert kernel_grid(L["sx"], L["sy"])[1] == 2048
    for name in ("blobs_outliers", "strip"):
        L = layout(name)
        print("%s: hash grid cell %.1f px, %d x %d cells, fullest cell %d" % ((name,) + kernel_grid(L["sx"], L["sy"])))
    # duplicates at identical coordinates with different values
    L = layout("duplicates")
    P = np.column_stack([L["sx"], L["sy"]])
    _, first, counts = np.unique(P, axis=0, return_index=True, return_counts=True)
    assert (counts > 1).sum() == 150
    # collinear sources: a hull of two points
    L = layout("collinear")
    assert exact_hull(*exact_ints(L["sx"], L["sy"])[0]).size == 2
    # band points: inside for SciPy, outside for an exact orientation, beyond a slanted and a bounding-box edge; and
    # points SciPy rejects that still lie within the kernel's (wider) band
    L = layout("band")
    n = L["qx"].size
    band = np.arange(n - L["n_band"], n)
    nan = scipy_nan("band")[band]
    sd = hull_distance("band", band)
    out, dist = sd < 0, -sd
    acc = out & ~nan
    on_box = L["qx"][band] < 0
    print("band: %d constructed, %d exactly outside, %d of them accepted by SciPy (%d beyond the x = 0 edge), "
          "largest accepted distance %.3g px" % (band.size, out.sum(), acc.sum(), (acc & on_box).sum(), dist[acc].max()))
    assert (acc & on_box).sum() >= 4 and (acc & ~on_box).sum() >= 20
    assert np.all(out[nan]) and (out & nan & (dist < 1e-10)).sum() >= 10 and (out & nan & (dist > 1e-9)).sum() >= 10
    assert not np.any(nan & ~out)


def test_collinear_sources_host_path_raises():
    """All-collinear sources: the reference and ``first_guess='host'`` raise QhullError (pinned behaviour)."""
    L = layout("collinear")
    dom = IdentityDomain((200, 1000))
    gx, gy = _grid(L["sx"], L["sy"], 10, 10)
    with pytest.raises(QhullError):
        sid.prepare_first_guess(gx, gy, dom, L["sx"], L["sy"], dom, L["vx"], L["vy"], 35, first_guess="host")


class IdentityDomain(object):
    """Geolocation that maps pixels to themselves exactly, so that integer layouts stay integer on image 2."""

    def __init__(self, shape):
        self._shape = shape

    def shape(self):
        return self._shape

    def transform_points(self, x, y, DstToSrc=0, dst_srs=None):
        return np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)


# ---------------------------------------------------------------------------------------------------- GPU
def orb_layout(rot_deg):
    """ORB keypoints (cv2.ORB, the GPU Hamming matcher) on a speckle pair with a large flat region (no keypoints there),
    as prepare_first_guess sees them: sources c1n2, r1n2, values and seeds the matched positions on image 2.  rot_deg 0
    keeps an integer grid; rot_deg 7 makes it non-integer (distances then go through the rounded int16 grid)."""
    img1 = syn.speckle_image((1200, 1200), seed=9)
    img1[250:800, 300:850] = 128
    img2 = syn.warp_pair(img1, syn.shift_matrix(3.5, -2.25), seed=9)
    x1, y1, x2, y2 = syn.orb_matches(img1, img2, n_features=6000)
    n1, n2 = syn.ArrayDomain(img1, rot_deg=rot_deg), syn.ArrayDomain(img2, rot_deg=rot_deg)
    sx, sy = n2.transform_points(*n1.transform_points(x1, y1), 1)
    if rot_deg:
        lon, lat = np.meshgrid(np.linspace(0.02, 1.18, 45), np.linspace(79.98, 78.82, 45))
        gx, gy = (v.ravel() for v in n2.transform_points(lon, lat, 1))
        qx, qy = np.concatenate([gx, np.round(gx)]), np.concatenate([gy, np.round(gy)])
    else:
        gx, gy = _grid(np.array([0.0, 1199.0]), np.array([0.0, 1199.0]), 45, 45)
        qx, qy = gx, gy
    cx, cy = np.round(sx.mean()), np.round(sy.mean())
    return dict(sx=sx, sy=sy, vx=x2, vy=y2, kx=np.uint16(x2).astype(np.float64), ky=np.uint16(y2).astype(np.float64),
                qx=qx, qy=qy, f=(sx - cx) ** 2 + (sy - cy) ** 2, integer=False, n_band=0,
                orb=(n1, n2, x1, y1, x2, y2, gx, gy))


def check_device(ctx, name, generic):
    """References 1-5 and the flag rules for one layout; returns the flag census."""
    L = layout(name)
    sx, sy, qx, qy, kx, ky = L["sx"], L["sy"], L["qx"], L["qy"], L["kx"], L["ky"]
    t0 = time.perf_counter()
    pf, _, dist, flag = ctx.first_guess(sx, sy, L["f"], L["f"], kx, ky, qx, qy)
    lx, ly, _, flag_l = ctx.first_guess(sx, sy, sx, sy, kx, ky, qx, qy)
    vx, vy, _, flag_v = ctx.first_guess(sx, sy, L["vx"], L["vy"], kx, ky, qx, qy)
    t_dev = time.perf_counter() - t0
    assert np.array_equal(flag, flag_l) and np.array_equal(flag, flag_v)          # the flag depends on geometry only
    census = np.bincount(flag, minlength=4)
    # 5: nearest-keypoint distance, bit for bit, at integer queries
    iq = (qx == np.round(qx)) & (qy == np.round(qy))
    assert np.array_equal(dist[iq], nearest_seed_distance(kx, ky, qx[iq], qy[iq])), name
    # flags against SciPy (the host path) and against exact geometry
    t0 = time.perf_counter()
    nan_host = scipy_nan(name)
    host_vx, host_vy = lib.interpolation_near(sx, sy, L["vx"], L["vy"], qx, qy)
    inside, simplex, (ef, ex, ey, evx, evy), kappa = exact_values(name, qx, qy, (L["f"], sx, sy, L["vx"], L["vy"]))
    # the kernel's band around the hull boundary (sid_fg_kernel.cuh): flag 2 there and only there (no pivot-cap hits)
    diag = np.hypot(np.ptp(sx), np.ptp(sy))
    band_px = HULL_BAND_EPS * diag
    suspect = np.nonzero((flag == 2) | (nan_host != (flag == 1)) | (inside != np.isin(flag, (0, 3))) |
                         (np.arange(qx.size) >= qx.size - L["n_band"]))[0]
    near = np.zeros(qx.size, bool)
    sd = hull_distance(name, suspect)
    near[suspect] = np.abs(sd) <= band_px * 1.01
    bad = suspect[(flag[suspect] == 2) & ~near[suspect]]
    assert bad.size == 0, (name, "flag 2 away from the hull boundary", list(zip(qx[bad][:5], qy[bad][:5])))
    assert np.array_equal(flag[~near] == 1, nan_host[~near]), name           # away from it: SciPy's verdict
    assert np.array_equal(np.isin(flag[~near], (0, 3)), inside[~near]), name
    assert np.all(flag[near & ~inside] == 2) and not np.any((flag == 1) & ~nan_host), name
    if L["n_band"]:                                  # every band point SciPy accepts is exactly outside: host decides
        b = np.arange(qx.size - L["n_band"], qx.size)
        acc = b[~nan_host[b] & ~inside[b]]
        assert acc.size and np.all(flag[acc] == 2), name
    if generic:
        assert not np.any(flag == 3), name
    ok = np.isin(flag, (0, 3))
    assert np.all(inside[ok])
    simp = delaunay_exact(name)[1][simplex[ok]]
    # 1: lifted paraboloid, unique even where the triangulation is not (flag 3, first_guess='device')
    err = np.abs(pf[ok] - ef[ok])
    tol = interp_tol(L["f"], L["f"][simp], kappa[ok])
    assert np.all(err <= tol), (name, "paraboloid", err.max(), int((err > tol).sum()))
    # 2: linear precision
    for got, want, vals in ((lx, qx, sx), (ly, qy, sy)):
        e2 = np.abs(got[ok] - want[ok])
        assert np.all(e2 <= interp_tol(vals, vals[simp], kappa[ok])), (name, "linear precision", e2.max())
    # 3: real values at flag 0: the exact rational interpolation and the host path's LinearNDInterpolator
    z = flag[ok] == 0
    for got, exact, host, vals in ((vx, evx, host_vx, L["vx"]), (vy, evy, host_vy, L["vy"])):
        e3 = np.abs(got[ok] - exact[ok])[z]
        t3 = interp_tol(vals, vals[simp], kappa[ok])[z]
        assert np.all(e3 <= t3), (name, "values", e3.max())
        e4 = np.abs(got[ok] - host[ok])[z]
        assert np.all(e4 <= t3 + host_tol(vals, vals[simp], kappa[ok])[z]), (name, "values vs host", e4.max())
    print("%-15s %6d sources %6d queries  flags 0/1/2/3: %5d %5d %3d %5d   device %.1f ms, references %.2f s  "
          "max paraboloid error %.2g of its bound" % (name, sx.size, qx.size, census[0], census[1], census[2], census[3],
                                                       1e3 * t_dev, time.perf_counter() - t0, (err / tol).max()))
    return census


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEOMETRIC)
def test_device_first_guess_against_exact_geometry(gpu_ctx, name):
    census = check_device(gpu_ctx, name, generic=name in GENERIC)
    if name.startswith("lattice"):
        assert census[3] > 0                         # cocircular cells are detected (then 'auto' falls back)
    if name == "band":
        assert census[2] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEGENERATE)
def test_device_first_guess_degenerate_sources(gpu_ctx, name):
    """All-collinear sources (hull of two points) and fewer than three sources: flag 1 and NaN everywhere, exact
    distances."""
    L = layout(name)
    vx, vy, dist, flag = gpu_ctx.first_guess(L["sx"], L["sy"], L["vx"], L["vy"], L["kx"], L["ky"], L["qx"], L["qy"])
    assert np.all(flag == 1) and np.isnan(vx).all() and np.isnan(vy).all()
    iq = (L["qx"] == np.round(L["qx"])) & (L["qy"] == np.round(L["qy"]))
    assert np.array_equal(dist[iq], nearest_seed_distance(L["kx"], L["ky"], L["qx"][iq], L["qy"][iq]))


def _contract(n1, n2, c1, r1, c2, r2, gx, gy):
    """'auto' (the default) equals 'host' bit for bit for both border rules."""
    for old_border in (True, False):
        auto = sid.prepare_first_guess(gx, gy, n1, c1, r1, n2, c2, r2, 35, old_border=old_border)
        host = sid.prepare_first_guess(gx, gy, n1, c1, r1, n2, c2, r2, 35, old_border=old_border, first_guess="host")
        for what, a, b in zip(("c2fg", "r2fg", "border"), auto, host):
            assert np.array_equal(a, b, equal_nan=True), (what, old_border, int((a != b).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEOMETRIC)
def test_prepare_first_guess_auto_equals_host(gpu_ctx, name):
    """On integer and on non-integer grids (the queries of the layout, band points included, and the same shifted by a
    fraction of a pixel)."""
    L = layout(name)
    dom = IdentityDomain((int(max(L["vy"].max(), L["qy"].max())) + 40, int(max(L["vx"].max(), L["qx"].max())) + 40))
    for dx, dy in ((0.0, 0.0), (0.375, -0.25)):
        _contract(dom, dom, L["sx"], L["sy"], L["vx"], L["vy"], L["qx"] + dx, L["qy"] + dy)


@pytest.mark.gpu
def test_prepare_first_guess_collinear_sources_pinned(gpu_ctx):
    """All-collinear sources: 'auto' returns the polynomial guess and max_border everywhere (the reference and 'host'
    raise QhullError instead, see test_collinear_sources_host_path_raises)."""
    L = layout("collinear")
    dom = IdentityDomain((1000, 1000))
    gx, gy = _grid(L["sx"], L["sy"], 10, 10)
    c2fg, r2fg, border = sid.prepare_first_guess(gx, gy, dom, L["sx"], L["sy"], dom, L["vx"], L["vy"], 35)
    px, py = np.round(lib.interpolation_poly(L["sx"], L["sy"], L["vx"], L["vy"], gx, gy))
    assert np.array_equal(c2fg, px) and np.array_equal(r2fg, py) and np.all(border == 50)


@pytest.mark.gpu
@pytest.mark.parametrize("rot_deg", (0.0, 7.0))
def test_orb_keypoints_with_flat_region(gpu_ctx, rot_deg):
    name = "orb%g" % rot_deg
    L = layout(name)
    assert fan_start_queries(name) > 0                # the flat region is a void inside the hull
    check_device(gpu_ctx, name, generic=False)
    n1, n2, x1, y1, x2, y2, gx, gy = L["orb"]
    assert (gx == np.round(gx)).all() == (rot_deg == 0)
    _contract(n1, n2, x1, y1, x2, y2, gx, gy)
