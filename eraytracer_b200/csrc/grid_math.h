// Per-element arithmetic of the grid builders that the host builders (cell_grid.cpp, light_grid.cpp) and the device
// builders (grid_build.cuh) must carry out identically: the cell grid's geometry, a sphere's cell range and the
// `reaches` test, a direction grid's 1-D bound and cell index, and the distance bound of its entries.  Like
// scene_math.h it is compiled by the host compiler and by nvcc with -fmad=false, so both sides produce the same bits.
// Max and min are written as the ternaries std::max / std::min expand to.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#include "scene_math.h"

namespace ert {

// ---- cell grid -------------------------------------------------------------------------------------------------

// Where the cells of a cell grid are (cell_grid.h CellGrid carries the same fields).  eps_d is the inflation in
// double, as `reaches` uses it; eps its float, as cell ranges and the walk use it.
struct CellGridGeom {
    int res[3] = {0, 0, 0};
    float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    float cs = 0, inv_cs = 0, eps = 0;
    double eps_d = 0;
    uint64_t n_cells = 0;
};

// The geometry of the cell grid over n spheres whose boxes [c - |r|, c + |r|] span [lo, hi] (the double bounds),
// abs_max: the largest |coordinate| of any sphere box.  False when the scene does not suit a grid (fewer than
// min_spheres spheres, abs_max beyond 1e6, degenerate extents, more than 2^23 cells); g then holds what was set.
inline bool cell_grid_geometry(const double lo[3], const double hi[3], int64_t n, float abs_max, double density,
                               int min_spheres, int max_res, CellGridGeom &g)
{
    g = CellGridGeom();
    if (n < min_spheres || !(density > 0) || !std::isfinite(abs_max) || abs_max > 1e6f) return false;
    const double u = 5.9604644775390625e-8;
    // The walk follows the FP32 ray within m/2 of the true one (m: the per-ray margin of make_sray,
    // >= 32u(|o|+abs_max)); boxes are inflated by eps and a ray may use the grid iff 4m <= eps.
    const double eps = 1024.0 * u * std::max((double)abs_max, 1.0);
    g.eps_d = eps;
    double ext[3], vol = 1.0;
    for (int a = 0; a < 3; a++) {
        g.lo[a] = f_round_down(lo[a] - 2.0 * eps);
        g.hi[a] = f_round_up(hi[a] + 2.0 * eps);
        ext[a] = (double)g.hi[a] - (double)g.lo[a];
        if (!(ext[a] > 0) || !std::isfinite(ext[a])) return false;
        vol *= ext[a];
    }
    // cubic cells: edge from the wanted cell count, then never so small that an axis needs more
    // than max_res cells
    double cs = std::cbrt(vol / (density * (double)n));
    for (int a = 0; a < 3; a++) cs = std::max(cs, ext[a] / (double)(max_res - 1));
    if (!(cs > 64.0 * eps) || !std::isfinite(cs)) return false;
    g.cs = f_round_up(cs);
    g.inv_cs = (float)(1.0 / (double)g.cs);
    g.eps = (float)eps;
    size_t n_cells = 1;
    for (int a = 0; a < 3; a++) {
        int r = (int)std::ceil(ext[a] / (double)g.cs) + 1;
        g.res[a] = std::min(std::max(r, 1), max_res);
        if ((double)g.res[a] * (double)g.cs < ext[a]) return false;
        n_cells *= (size_t)g.res[a];
    }
    if (n_cells > ((size_t)1 << 23)) return false;           // 256 bytes per cell on the device
    g.n_cells = n_cells;
    return true;
}

// Cell range [i0, i1] of the interval [a, b] along one axis.
ERT_HD void cell_range(const float *g_lo, float g_cs, float g_eps, const int *g_res, int axis, double a, double b,
                       int &i0, int &i1)
{
    const double lo = (double)g_lo[axis], cs = (double)g_cs;
    double f0 = floor((a - (double)g_eps - lo) / cs), f1 = floor((b + (double)g_eps - lo) / cs);
    const double top = (double)(g_res[axis] - 1);
    i0 = (int)d_min(d_max(f0, 0.0), top);
    i1 = (int)d_min(d_max(f1, 0.0), top);
}

// A cell inside the box of a sphere may still be out of the ball's reach (the corners of the box):
// the ball inflated by eps must come within the cell, also inflated by eps for the float planes.
// p: the sphere's centre, rad: its radius.
ERT_HD bool cell_reaches(const float *g_lo, float g_cs, double eps, const double *p, double rad, int x, int y, int z)
{
    const double r = fabs(rad) + 2.0 * eps;
    const int c[3] = {x, y, z};
    double d2 = 0;
    for (int a = 0; a < 3; a++) {
        const double lo_a = (double)g_lo[a] + (double)c[a] * (double)g_cs, hi_a = lo_a + (double)g_cs;
        const double d = p[a] < lo_a ? lo_a - p[a] : (p[a] > hi_a ? p[a] - hi_a : 0.0);
        d2 += d * d;
    }
    return d2 <= r * r * (1.0 + 1e-9);
}

// ---- direction grids -------------------------------------------------------------------------------------------

constexpr double kLgQuarterPi = 0.78539816339744830962;
// Shadow rays find their cell in FP32 (light_grid_cell_f32: direction rounded to float, one reciprocal, two
// products — every step within 6e-8 relative, |u| <= 1, so the cell coordinate is off by < 5e-7, and a direction
// that close to a face edge may land on the neighbouring face).  The slack below is four times that, on the
// half-angle and on the projected bounds, so a sphere is listed in every cell the FP32 computation can name for a
// direction that touches it.
constexpr double kLgAngleSlack = 2e-6;      // radians added to every half-angle
constexpr double kLgCoordSlack = 2e-6;      // added to the projected bounds

// 1-D bound: directions (x, z) with z > 0 and |x/z| <= 1 that can touch the disc (cx, cz, r).
// Returns false when none can.  lo/hi are bounds of x/z inside [-1, 1].
ERT_HD bool axis_bound(double cx, double cz, double r, double &lo, double &hi)
{
    double rho2 = cx * cx + cz * cz;
    if (rho2 <= r * r) { lo = -1.0; hi = 1.0; return true; }       // the origin is inside the disc
    double rho = sqrt(rho2);
    double theta = atan2(cx, cz);                                    // from +z towards +x
    double alpha = asin(d_min(1.0, r / rho)) + kLgAngleSlack;
    if (fabs(theta) - alpha > kLgQuarterPi) return false;
    double a0 = d_max(theta - alpha, -kLgQuarterPi), a1 = d_min(theta + alpha, kLgQuarterPi);
    lo = d_max(-1.0, tan(a0) - kLgCoordSlack);
    hi = d_min(1.0, tan(a1) + kLgCoordSlack);
    return lo <= hi;
}

ERT_HD int cell_index(double x, int res)
{
    int i = (int)floor((x + 1.0) * 0.5 * res);
    i = (i < 0) ? 0 : i;
    return (res - 1 < i) ? res - 1 : i;
}

// The cell rectangle of one cube face that a sphere can cover, seen from the light.
struct LightRect { int face, u0, u1, v0, v1; };

// The rectangles of the sphere (center, radius) seen from `light` at `res` cells per face edge: their number
// (at most 6), or -1 when the sphere (nearly) contains the light and goes to the always-list.
ERT_HD int light_rects(const double *center, double radius, const double *light, int res, LightRect out[6])
{
    double c[3] = {center[0] - light[0], center[1] - light[1], center[2] - light[2]};
    double r = fabs(radius);
    r = r * (1.0 + 1e-6) + 1e-9;
    double d2 = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
    if (!(d2 > r * r)) return -1;                                   // also catches NaN
    int n = 0;
    for (int m = 0; m < 3; m++) {
        int a = (m + 1) % 3, b = (m + 2) % 3;
        for (int sgn = 0; sgn < 2; sgn++) {
            double cz = sgn ? -c[m] : c[m];
            if (cz + r <= 0.0) continue;                            // entirely behind this face
            double ulo, uhi, vlo, vhi;
            if (!axis_bound(c[a], cz, r, ulo, uhi)) continue;
            if (!axis_bound(c[b], cz, r, vlo, vhi)) continue;
            LightRect &q = out[n++];
            q.face = 2 * m + sgn;
            q.u0 = cell_index(ulo, res); q.u1 = cell_index(uhi, res);
            q.v0 = cell_index(vlo, res); q.v1 = cell_index(vhi, res);
        }
    }
    return n;
}

// Lower bound of the distance from the light to a sphere whose centre is at c (relative to the light) and whose
// radius is rad, in float, with relative slack for the shadow kernel's FP32 comparisons.
ERT_HD float light_dmin(const double *c, double rad)
{
    double dist = sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]) - fabs(rad);
    float dmin = (float)(dist * (1.0 - 1e-5) - 1e-6);
    if ((double)dmin > dist) dmin = nextafterf(dmin, -INFINITY);
    return dmin;
}

}  // namespace ert
