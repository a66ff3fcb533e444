// sid_fg_kernel.cuh -- first guess for pattern matching on the device (SURVEY 8f rank 1; reference
// pmlib.py:249-324 prepare_first_guess and pmlib.py:61-77 get_distance_to_nearest_keypoint).
//
// What the reference computes per PM grid point q (on image 2):
//   * griddata(method='linear') of the feature-tracking vectors: the value of the piecewise-linear interpolant over the
//     DELAUNAY triangulation of the keypoints at q, NaN outside their convex hull (lib.py:179-201; Qhull);
//   * the distance from q to the nearest keypoint (a full-image Euclidean distance transform sampled at q).
// Here, without building a triangulation: one thread per grid point finds THE Delaunay triangle that contains q by
// pivoting -- start from any keypoint triangle around q, and while some keypoint lies strictly inside its circumcircle
// replace a vertex by the deepest such point so that q stays inside (the simplex step of the 3-variable linear program
// "highest plane below all lifted points at q"; the objective rises with every pivot, so it terminates).  A triangle
// with an empty circumcircle is a Delaunay triangle, and the one containing q is unique unless four keypoints are
// cocircular (then any choice is a valid Delaunay triangulation; Qhull's own choice is arbitrary as well).  Keypoints
// are looked up through a uniform hash grid built by the host.  The nearest-keypoint distance is an exact integer
// ring search on a second grid.
#pragma once
#include "sid_common.cuh"

namespace sid {

struct FgGrid {            // uniform hash grid over a point set (points sorted by cell, host-built)
    const double *x, *y;   // sorted coordinates
    const int *start;      // nx * ny + 1 cell offsets
    const int *index;      // original index of every sorted point (into the value arrays)
    double x0, y0, inv_cell, cell;
    int nx, ny, n;
};

struct FgArgs {
    FgGrid src;            // interpolation sources (keypoints of image 1 mapped onto image 2)
    const double *vx, *vy; // values at the sources (matched positions on image 2), original order
    const double *hx, *hy; // convex hull of the sources, counter-clockwise, nh vertices
    const int *hidx;       // source index of every hull vertex
    const double *hband;   // per hull edge k -> k + 1: FG_HULL_BAND_EPS * |edge| * diagonal of the sources' bounding box
    int nh;
    FgGrid seed;           // integer keypoint positions on image 2 (nearest-keypoint distance)
    long long nq;
    const double *qx, *qy; // query points
    double *out_vx, *out_vy, *out_dist;
    int *out_flag;         // 0 ok, 1 outside the hull (NaN), 2 not resolved numerically or within SciPy's band around the hull
                           // boundary (NaN there), 3 ok but a further keypoint lies ON the
                           // circumcircle: the Delaunay triangulation is not unique there (Qhull's choice may differ)
};

__device__ __forceinline__ double fg_orient(double ax, double ay, double bx, double by, double cx, double cy) {
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);           // > 0: a, b, c counter-clockwise
}
// > 0 when d lies strictly inside the circumcircle of the counter-clockwise triangle a, b, c
__device__ __forceinline__ double fg_incircle(double ax, double ay, double bx, double by, double cx, double cy, double dx, double dy) {
    const double adx = ax - dx, ady = ay - dy, bdx = bx - dx, bdy = by - dy, cdx = cx - dx, cdy = cy - dy;
    const double ad = adx * adx + ady * ady, bd = bdx * bdx + bdy * bdy, cd = cdx * cdx + cdy * cdy;
    return adx * (bdy * cd - bd * cdy) - ady * (bdx * cd - bd * cdx) + ad * (bdx * cdy - bdy * cdx);
}
// Closed triangle test by orientation signs.  The hull test in first_guess_kernel is the same test against the hull edges, but
// SciPy decides "inside" differently: _find_simplex_directed (scipy/spatial/_qhull.pyx) accepts q in a simplex when
// every barycentric coordinate is >= -eps, eps = 100 * DBL_EPSILON, so LinearNDInterpolator / griddata return a value
// slightly OUTSIDE the hull.  Bound on that band: if SciPy accepts q in the triangle v0 v1 v2, q = sum c_i v_i with
// sum c_i = 1 and c_i >= -eps; orient(a, b, .) against a hull edge a b is affine and lies in [0, |ab| * D] on every source
// (D the diagonal of the sources' bounding box), and at most two c_i are negative, so
// orient(a, b, q) >= -2 * eps * |ab| * D.  The kernel widens that by ~10x (FG_HULL_BAND_EPS) to cover the rounding of
// fg_orient and of SciPy's barycentric transform.  That rounding also makes SciPy's answer for a query ON the hull
// boundary arbitrary: on the thin hull triangles of a ring of integer points it returns NaN for integer queries exactly
// on a hull edge.  So the band is two-sided: a query whose orientation against some hull edge lies within
// +-FG_HULL_BAND_EPS * D * |ab| (and below none) is undecided, flag 2, and the host decides.
constexpr double FG_HULL_BAND_EPS = 2048.0 * 2.220446049250313e-16;
// fg_orient without fused multiply-adds: with the two products rounded alike, fg_orient_rn(a, b, b) is exactly 0 (with an
// FMA it is the rounding error of one product, of either sign), so a query ON a keypoint lies on the closed triangles
// that have the keypoint as a vertex; otherwise a pivot onto a keypoint equal to q could find no triangle holding q.
__device__ __forceinline__ double fg_orient_rn(double ax, double ay, double bx, double by, double cx, double cy) {
    return __dsub_rn(__dmul_rn(bx - ax, cy - ay), __dmul_rn(by - ay, cx - ax));
}
__device__ __forceinline__ bool fg_contains(double ax, double ay, double bx, double by, double cx, double cy, double qx, double qy) {
    const double o = fg_orient_rn(ax, ay, bx, by, cx, cy);
    if (o == 0.0) return false;
    const double s = o > 0.0 ? 1.0 : -1.0;
    return s * fg_orient_rn(ax, ay, bx, by, qx, qy) >= 0.0 && s * fg_orient_rn(bx, by, cx, cy, qx, qy) >= 0.0 &&
           s * fg_orient_rn(cx, cy, ax, ay, qx, qy) >= 0.0;
}
__device__ __forceinline__ int fg_cell(double v, double v0, double inv, int n) {
    int c = (int)floor((v - v0) * inv);
    return c < 0 ? 0 : (c >= n ? n - 1 : c);
}

constexpr int FG_NEAR = 12;       // nearest sources examined for the starting triangle
constexpr int FG_MAX_PIVOTS = 256;

__global__ void __launch_bounds__(128) first_guess_kernel(const FgArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.nq) return;
    const double qx = a.qx[t], qy = a.qy[t];

    // ---- nearest integer keypoint (reference pmlib.py:61-77, 300-305): rings of cells until no closer seed can exist
    {
        const FgGrid &g = a.seed;
        double best = 1e300;
        if (g.n > 0) {
            const int cx = fg_cell(qx, g.x0, g.inv_cell, g.nx), cy = fg_cell(qy, g.y0, g.inv_cell, g.ny);
            const int rmax = max(g.nx, g.ny);
            for (int r = 0; r <= rmax; ++r) {
                // every cell at Chebyshev ring distance r is at least (r - 1) * cell away from q (q may sit anywhere in its cell)
                if (r >= 2 && (double)(r - 1) * g.cell * (double)(r - 1) * g.cell > best) break;
                const int x_lo = cx - r, x_hi = cx + r, y_lo = cy - r, y_hi = cy + r;
                for (int yy = max(y_lo, 0); yy <= min(y_hi, g.ny - 1); ++yy) {
                    const bool edge_row = (yy == y_lo || yy == y_hi);
                    for (int xx = max(x_lo, 0); xx <= min(x_hi, g.nx - 1); ++xx) {
                        if (!edge_row && xx != x_lo && xx != x_hi) continue;      // ring cells only
                        const int c = yy * g.nx + xx;
                        for (int k = g.start[c]; k < g.start[c + 1]; ++k) {
                            const double dx = g.x[k] - qx, dy = g.y[k] - qy;
                            const double d2 = dx * dx + dy * dy;
                            best = d2 < best ? d2 : best;
                        }
                    }
                }
            }
        }
        a.out_dist[t] = sqrt(best);
    }

    // ---- inside the convex hull of the sources?  (fan from hull vertex 0; also the fallback starting triangle)
    const FgGrid &g = a.src;
    int fan = -1;
    if (a.nh >= 3) {
        bool inside = true, band = false;
        for (int k = 0; k < a.nh && inside; ++k) {
            const int k2 = k + 1 == a.nh ? 0 : k + 1;
            const double o = fg_orient(a.hx[k], a.hy[k], a.hx[k2], a.hy[k2], qx, qy);
            if (o < -a.hband[k]) inside = false;
            else if (o <= a.hband[k]) band = true;               // on the hull boundary up to SciPy's band (see fg_contains)
        }
        if (inside && band) {
            a.out_vx[t] = a.out_vy[t] = nan("");
            a.out_flag[t] = 2;
            return;
        }
        if (inside)
            for (int k = 1; k + 1 < a.nh; ++k)
                if (fg_contains(a.hx[0], a.hy[0], a.hx[k], a.hy[k], a.hx[k + 1], a.hy[k + 1], qx, qy)) { fan = k; break; }
    }
    if (fan < 0) {
        a.out_vx[t] = a.out_vy[t] = nan("");
        a.out_flag[t] = 1;
        return;
    }

    // ---- starting triangle: the FG_NEAR nearest sources, first triple (by nearness) that contains q
    double nx_[FG_NEAR], ny_[FG_NEAR], nd_[FG_NEAR];
    int ni_[FG_NEAR], nn = 0;
    {
        const int cx = fg_cell(qx, g.x0, g.inv_cell, g.nx), cy = fg_cell(qy, g.y0, g.inv_cell, g.ny);
        const int rmax = max(g.nx, g.ny);
        for (int r = 0; r <= rmax; ++r) {
            if (nn == FG_NEAR && r >= 2 && (double)(r - 1) * g.cell * (double)(r - 1) * g.cell > nd_[nn - 1]) break;
            if (r > 6 && nn >= 3) break;                         // sparse neighbourhood: settle for what was found
            const int x_lo = cx - r, x_hi = cx + r, y_lo = cy - r, y_hi = cy + r;
            for (int yy = max(y_lo, 0); yy <= min(y_hi, g.ny - 1); ++yy) {
                const bool edge_row = (yy == y_lo || yy == y_hi);
                for (int xx = max(x_lo, 0); xx <= min(x_hi, g.nx - 1); ++xx) {
                    if (!edge_row && xx != x_lo && xx != x_hi) continue;
                    const int c = yy * g.nx + xx;
                    for (int k = g.start[c]; k < g.start[c + 1]; ++k) {
                        const double dx = g.x[k] - qx, dy = g.y[k] - qy, d2 = dx * dx + dy * dy;
                        if (nn < FG_NEAR || d2 < nd_[nn - 1]) {     // insertion into the sorted list
                            int pos = nn < FG_NEAR ? nn++ : FG_NEAR - 1;
                            while (pos > 0 && nd_[pos - 1] > d2) {
                                nd_[pos] = nd_[pos - 1]; nx_[pos] = nx_[pos - 1]; ny_[pos] = ny_[pos - 1]; ni_[pos] = ni_[pos - 1];
                                --pos;
                            }
                            nd_[pos] = d2; nx_[pos] = g.x[k]; ny_[pos] = g.y[k]; ni_[pos] = g.index[k];
                        }
                    }
                }
            }
        }
    }
    double ax, ay, bx, by, cx_, cy_;
    int ia = -1, ib = -1, ic = -1;
    for (int k3 = 2; k3 < nn && ia < 0; ++k3)
        for (int k2 = 1; k2 < k3 && ia < 0; ++k2)
            for (int k1 = 0; k1 < k2; ++k1)
                if (fg_contains(nx_[k1], ny_[k1], nx_[k2], ny_[k2], nx_[k3], ny_[k3], qx, qy)) {
                    ax = nx_[k1]; ay = ny_[k1]; ia = ni_[k1];
                    bx = nx_[k2]; by = ny_[k2]; ib = ni_[k2];
                    cx_ = nx_[k3]; cy_ = ny_[k3]; ic = ni_[k3];
                    break;
                }
    if (ia < 0) {                                                // near the hull: the hull fan triangle that contains q
        ax = a.hx[0]; ay = a.hy[0]; ia = a.hidx[0];
        bx = a.hx[fan]; by = a.hy[fan]; ib = a.hidx[fan];
        cx_ = a.hx[fan + 1]; cy_ = a.hy[fan + 1]; ic = a.hidx[fan + 1];
    }
    if (fg_orient(ax, ay, bx, by, cx_, cy_) < 0.0) {             // make it counter-clockwise
        double tx = bx, ty = by; int ti = ib;
        bx = cx_; by = cy_; ib = ic; cx_ = tx; cy_ = ty; ic = ti;
    }

    // ---- pivot until the circumcircle is empty
    int flag = 0;
    for (int it = 0;; ++it) {
        if (it == FG_MAX_PIVOTS) { flag = 2; break; }
        // circumcircle of a, b, c (centre relative to a)
        const double bxa = bx - ax, bya = by - ay, cxa = cx_ - ax, cya = cy_ - ay;
        const double d = 2.0 * (bxa * cya - bya * cxa);
        const double b2 = bxa * bxa + bya * bya, c2 = cxa * cxa + cya * cya;
        const double ux = (cya * b2 - bya * c2) / d, uy = (bxa * c2 - cxa * b2) / d;
        const double rad = sqrt(ux * ux + uy * uy), ox = ax + ux, oy = ay + uy;
        const int x_lo = fg_cell(ox - rad, g.x0, g.inv_cell, g.nx), x_hi = fg_cell(ox + rad, g.x0, g.inv_cell, g.nx);
        const int y_lo = fg_cell(oy - rad, g.y0, g.inv_cell, g.ny), y_hi = fg_cell(oy + rad, g.y0, g.inv_cell, g.ny);
        double deepest = 0.0, px = 0.0, py = 0.0;
        int ip = -1;
        bool on_circle = false;
        // scan the cells under the circle in rings around q's own cell and pivot on the deepest violator of the FIRST ring
        // that holds one: points near q shrink a large circle quickly (a starting triangle at the hull can span the whole
        // point set), and only the final, empty circle is scanned completely
        const int qcx = fg_cell(qx, g.x0, g.inv_cell, g.nx), qcy = fg_cell(qy, g.y0, g.inv_cell, g.ny);
        const int rlast = max(max(qcx - x_lo, x_hi - qcx), max(qcy - y_lo, y_hi - qcy));
        for (int r = 0; r <= rlast && ip < 0; ++r) {
            const int rx_lo = qcx - r, rx_hi = qcx + r, ry_lo = qcy - r, ry_hi = qcy + r;
            for (int yy = max(ry_lo, y_lo); yy <= min(ry_hi, y_hi); ++yy) {
                const bool edge_row = (yy == ry_lo || yy == ry_hi);
                for (int xx = max(rx_lo, x_lo); xx <= min(rx_hi, x_hi); ++xx) {
                    if (!edge_row && xx != rx_lo && xx != rx_hi) continue;
                    const int c = yy * g.nx + xx;
                    for (int k = g.start[c]; k < g.start[c + 1]; ++k) {
                        const int id = g.index[k];
                        if (id == ia || id == ib || id == ic) continue;
                        const double dxk = g.x[k], dyk = g.y[k];
                        const double v = fg_incircle(ax, ay, bx, by, cx_, cy_, dxk, dyk);
                        // |v| at rounding-error level of its own terms (exactly 0 for cocircular integer pixels): not unique
                        const double sa = (ax - dxk) * (ax - dxk) + (ay - dyk) * (ay - dyk), sb = (bx - dxk) * (bx - dxk) + (by - dyk) * (by - dyk),
                                     sc = (cx_ - dxk) * (cx_ - dxk) + (cy_ - dyk) * (cy_ - dyk);
                        const double tol = 4e-14 * (sa + sb + sc) * (sa + sb + sc);
                        if (v > tol) { if (v > deepest) { deepest = v; px = dxk; py = dyk; ip = id; } }
                        else if (v >= -tol) on_circle = true;
                    }
                }
            }
        }
        if (ip < 0) { if (on_circle) flag = 3; break; }          // empty circumcircle: a Delaunay triangle
        // the new triangle has the deepest point p as a vertex and still contains q
        if (fg_contains(px, py, ax, ay, bx, by, qx, qy)) { cx_ = px; cy_ = py; ic = ip; }
        else if (fg_contains(px, py, bx, by, cx_, cy_, qx, qy)) { ax = px; ay = py; ia = ip; }
        else if (fg_contains(px, py, cx_, cy_, ax, ay, qx, qy)) { bx = px; by = py; ib = ip; }
        else { flag = 2; break; }                                // numerically degenerate: let the host decide
        if (fg_orient(ax, ay, bx, by, cx_, cy_) < 0.0) {
            double tx = bx, ty = by; int ti = ib;
            bx = cx_; by = cy_; ib = ic; cx_ = tx; cy_ = ty; ic = ti;
        }
    }
    // ---- barycentric interpolation of the two value sets
    const double area = fg_orient(ax, ay, bx, by, cx_, cy_);
    const double wa = fg_orient(bx, by, cx_, cy_, qx, qy) / area, wb = fg_orient(cx_, cy_, ax, ay, qx, qy) / area;
    const double wc = 1.0 - wa - wb;
    a.out_vx[t] = wa * a.vx[ia] + wb * a.vx[ib] + wc * a.vx[ic];
    a.out_vy[t] = wa * a.vy[ia] + wb * a.vy[ib] + wc * a.vy[ic];
    a.out_flag[t] = flag;
}

}  // namespace sid
