// Prune bounds of the triangle BVH walk (DESIGN.md "Triangle BVH"), shared by the device walk
// (ert_device.cuh) and its host restatement in the CPU tests.
//
// The walk only prunes; every triangle it reaches goes through the literal FP64 test of erl:402-455
// (triangle_exact).  What it must guarantee: a triangle that the literal test accepts with a Distance t
// that could still win under (t, list position) lies in a node the walk enters.  Two facts make the
// node test differ from the sphere slabs:
//  * the reference has no sign test on t (erl:442): hits behind the origin count, so the line is
//    walked from -inf, with no clamp of the entry parameter at 0;
//  * the literal test's roundings let it accept lines that pass outside the triangle, and return a t
//    below the line's parameter in the triangle's plane, by amounts that grow as det nears 1e-6.
// Both are bounded here per ray (|O|, |D|) from two constants of the tree (largest edge L, largest
// coordinate V): the boxes are widened by `margin` and the cull is raised by r|t| + a.
#pragma once
#include <cmath>

#ifdef __CUDACC__
#define ERT_HD __host__ __device__ __forceinline__
#else
#define ERT_HD inline
#endif

namespace ert {

struct TriRay {
    double inv[3];       // 1 / D (+-inf for a zero component)
    double cn[3], cf[3]; // near / far plane constants: t = (box plane + c) * inv, planes pushed out by the margin
    double r, a;         // cull slack: a triangle that can still win has its plane parameter <= t + r|t| + a
};

// false: this ray is outside the range the bounds are derived for (non-finite input, a denormal direction
// component, or det's rounding error not small against 1e-6); the caller then tests every triangle.
// `margins` = false drops every rounding term (the CPU tests show that the walk then loses hits).
ERT_HD bool tri_ray_setup(const double O[3], const double D[3], double edge_max, double abs_max, bool margins,
                          TriRay &tr)
{
    const double u = 1.1102230246251565e-16;                // 2^-53
    double oabs = 0, dabs = 0, dmin = INFINITY;
    for (int k = 0; k < 3; k++) {
        oabs = fmax(oabs, fabs(O[k]));
        dabs = fmax(dabs, fabs(D[k]));
        if (D[k] != 0.0) dmin = fmin(dmin, fabs(D[k]));
    }
    // |D|_2 <= sqrt(3) |D|_inf, |O - v1|_2 <= sqrt(3) (|O|_inf + V): each with room for its roundings
    const double rA = 1.7321 * dabs, T = 1.7321 * (oabs + abs_max), L = edge_max;
    // Errors of the literal test's values (each a dot product of a difference with a cross product of
    // rounded differences: a few units of 2^-53 times the product of the norms; 16 covers them):
    const double c = 16.0 * u;
    const double e_det = c * rA * L * L;      // det = E1 . (D x E2)
    const double e_uv = c * T * rA * L;       // u = T . (D x E2),  v = D . (T x E1)
    const double e_q = c * L * L * T;         // E2 . (T x E1)
    const double d_lo = 1e-6 - e_det;         // accepted det >= 1e-6: the exact det is at least this
    // Accepted barycentrics are at most (|err u| + |err v| + |err det|) / det outside [0, 1] (twice: u + v <= det
    // as well); the point in the plane is then within 4 L (2 e_uv + e_det) / det of the triangle.  The rounded
    // edges and T move the triangle and the line by u L and u T.
    double margin = 1.01 * (4.0 * L * (2.0 * e_uv + e_det) / d_lo + 8.0 * u * L + 2.0 * u * T);
    // t = (E2 . Q) / det is at most (err det / det + 2u) |t| + err(E2 . Q) / det below the plane parameter
    double r = 1.01 * (e_det / d_lo + 2.0 * u) + 7.105427357601002e-15;        // + 2^-47 for the cull's own sum
    double a = 1.01 * e_q / d_lo * (1.0 + 7.105427357601002e-15);
    if (!margins) margin = r = a = 0.0;
    const bool ok = oabs <= 1e30 && dabs <= 1e30 && !(dmin < 1e-290) && e_det <= 0.5e-6 && margin <= 1e30;
    if (!ok) return false;
    // the plane constants are rounded once more: widen by that rounding too
    const double m = margin + 8.881784197001252e-16 * (oabs + margin);            // + 2^-50 (|O| + margin)
    for (int k = 0; k < 3; k++) {
        tr.inv[k] = 1.0 / D[k];
        const double s = tr.inv[k] < 0.0 ? -m : m;
        tr.cn[k] = -(O[k] + s);
        tr.cf[k] = -(O[k] - s);
    }
    tr.r = r;
    tr.a = a;
    return true;
}

// plane-parameter cull of the incumbent (Distance t of any kind of object: a triangle's Distance is its plane
// parameter, erl:442, and `better` compares the incumbent's Distance as it is)
ERT_HD double tri_cull(const TriRay &tr, bool have, double t)
{
    if (!have) return INFINITY;
    return t + (fabs(t) * tr.r + tr.a);
}

// Line slab of one box, no clamp at 0.  Each t carries at most three roundings of its exact value (one part in
// 2^51), so widening both ends by 2^-48 keeps every parameter of the line inside the widened box.  A zero
// direction component gives +-inf (outside the slab: an empty interval) or NaN (on a plane: fmax / fmin ignore it).
ERT_HD bool tri_slab(const TriRay &tr, float lox, float hix, float loy, float hiy, float loz, float hiz, double cull,
                     double &tnear)
{
    const double nx = tr.inv[0] < 0.0 ? hix : lox, fx = tr.inv[0] < 0.0 ? lox : hix;
    const double ny = tr.inv[1] < 0.0 ? hiy : loy, fy = tr.inv[1] < 0.0 ? loy : hiy;
    const double nz = tr.inv[2] < 0.0 ? hiz : loz, fz = tr.inv[2] < 0.0 ? loz : hiz;
    const double t0x = (nx + tr.cn[0]) * tr.inv[0], t1x = (fx + tr.cf[0]) * tr.inv[0];
    const double t0y = (ny + tr.cn[1]) * tr.inv[1], t1y = (fy + tr.cf[1]) * tr.inv[1];
    const double t0z = (nz + tr.cn[2]) * tr.inv[2], t1z = (fz + tr.cf[2]) * tr.inv[2];
    const double tn = fmax(fmax(t0x, t0y), t0z), tf = fmin(fmin(t1x, t1y), t1z);
    tnear = tn - fabs(tn) * 3.552713678800501e-15;               // 2^-48
    const double tfar = tf + fabs(tf) * 3.552713678800501e-15;
    return tnear <= tfar && tnear <= cull;
}

}  // namespace ert
