// Per-element arithmetic that the host builders and the device update kernels (ert_update.cuh) must carry out
// identically: outward rounding to float, the FP32 filter sphere, a triangle's extent, and the refit of one BVH
// node.  Compiled by the host compiler for flatten() and the builders, and by nvcc for the update kernels (with
// -fmad=false, like the host's uncontracted arithmetic), so a quantity recomputed on the GPU has the bits the host
// computed at create.  Max and min are written as the ternaries std::max / std::min expand to.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <vector>

#include "bvh_build.h"

#ifndef ERT_HD
#ifdef __CUDACC__
#define ERT_HD __host__ __device__ __forceinline__
#else
#define ERT_HD inline
#endif
#endif

namespace ert {

ERT_HD float f_round_down(double x)
{
    float f = (float)x;
    if ((double)f > x) f = nextafterf(f, -INFINITY);
    return f;
}
ERT_HD float f_round_up(double x)
{
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}
ERT_HD double d_max(double a, double b) { return (a < b) ? b : a; }
ERT_HD double d_min(double a, double b) { return (b < a) ? b : a; }

// FP32 filter sphere {fl(c), R}: R >= r^2 with the slack the stage-1 bound needs
// (DESIGN.md "Filter bounds"): r^2 (1 + 2^-18) + 16 r eta_c + 4 eta_c^2 / u.
ERT_HD void make_filter_sphere(const double *c, double r, float out[4], float &pad_c, float &eta_c)
{
    const double u = 5.9604644775390625e-8;
    double eta = 0;
    for (int a = 0; a < 3; a++) {
        out[a] = (float)c[a];
        eta = d_max(eta, fabs(c[a] - (double)out[a]));
    }
    eta *= 2.0;
    r = fabs(r);
    double pad = 16.0 * r * eta + 4.0 * eta * eta / u;
    double R = r * r * (1.0 + 3.814697265625e-6) + pad;
    out[3] = nextafterf(f_round_up(R), INFINITY);
    pad_c = f_round_up(pad);
    eta_c = f_round_up(eta);
}

// Largest edge (2-norm, as the literal test forms the edges) and largest |coordinate| of a triangle {v1, v2, v3}.
ERT_HD void triangle_extent(const double *v, double &edge, double &amax)
{
    double e = 0, m = 0;
    for (int k = 0; k < 3; k++) {
        const double *p = v + 3 * k, *q = v + 3 * ((k + 1) % 3);
        double dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
        e = d_max(e, sqrt(dx * dx + dy * dy + dz * dz));
        for (int a = 0; a < 3; a++) m = d_max(m, fabs(p[a]));
    }
    edge = e;
    amax = m;
}

// ---- refit -----------------------------------------------------------------------------------------------------
// A refit keeps the builder's topology and leaf order and recomputes every stored child box bottom-up: a leaf's box
// is the union of its primitives' outward-rounded boxes, an inner child's box the union of that node's two boxes.
// Both are what build_box_bvh stored (the union of the primitives below, min/max being exact), so a refit of
// unmoved primitives gives the builder's node array back byte for byte.

// [c - |r|, c + |r|] rounded outward (build_sphere_bvh); s = {cx, cy, cz, r}
ERT_HD void sphere_box(const double *s, float lo[3], float hi[3])
{
    const double r = fabs(s[3]);
    for (int a = 0; a < 3; a++) {
        lo[a] = f_round_down(s[a] - r);
        hi[a] = f_round_up(s[a] + r);
    }
}
// the vertices' bounds rounded outward (build_triangle_bvh); v = {v1, v2, v3}
ERT_HD void triangle_box(const double *v, float lo[3], float hi[3])
{
    for (int a = 0; a < 3; a++) {
        lo[a] = f_round_down(d_min(v[a], d_min(v[3 + a], v[6 + a])));
        hi[a] = f_round_up(d_max(v[a], d_max(v[3 + a], v[6 + a])));
    }
}

ERT_HD void box_grow(float lo[3], float hi[3], const float plo[3], const float phi[3])
{
    for (int a = 0; a < 3; a++) {
        lo[a] = (plo[a] < lo[a]) ? plo[a] : lo[a];
        hi[a] = (hi[a] < phi[a]) ? phi[a] : hi[a];
    }
}

ERT_HD void child_box(const BvhNode &n, int k, float lo[3], float hi[3])
{
    const float *x = k == 0 ? n.c0x : n.c1x, *y = k == 0 ? n.c0y : n.c1y, *z = k == 0 ? n.c0z : n.c1z;
    lo[0] = x[0]; hi[0] = x[1]; lo[1] = y[0]; hi[1] = y[1]; lo[2] = z[0]; hi[2] = z[1];
}

// Surface area / 2 of a child box, 0 for an unused (inverted) one: the refit's degradation signal.
ERT_HD double child_half_area(const BvhNode &n, int k)
{
    float lo[3], hi[3];
    child_box(n, k, lo, hi);
    if (lo[0] > hi[0]) return 0.0;
    double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
}

// Refits node i from its children.  leaf_box(slot, lo, hi) gives the outward-rounded box of the primitive in leaf
// slot `slot`.  An unused child keeps its inverted box (a refitted box is never inverted, so the test is stable).
template <typename LeafBox>
ERT_HD void refit_node(BvhNode *nodes, int i, const LeafBox &leaf_box)
{
    BvhNode &n = nodes[i];
    for (int k = 0; k < 2; k++) {
        float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        float blo[3], bhi[3];
        child_box(n, k, blo, bhi);
        if (blo[0] > bhi[0]) continue;
        const int32_t c = n.child[k];
        if (c < 0) {
            const int32_t code = ~c, first = code >> 3, count = (code & 7) + 1;
            for (int32_t s = first; s < first + count; s++) {
                leaf_box(s, blo, bhi);
                box_grow(lo, hi, blo, bhi);
            }
        } else {
            for (int kk = 0; kk < 2; kk++) {
                child_box(nodes[c], kk, blo, bhi);
                box_grow(lo, hi, blo, bhi);
            }
        }
        float *x = k == 0 ? n.c0x : n.c1x, *y = k == 0 ? n.c0y : n.c1y, *z = k == 0 ? n.c0z : n.c1z;
        x[0] = lo[0]; x[1] = hi[0]; y[0] = lo[1]; y[1] = hi[1]; z[0] = lo[2]; z[1] = hi[2];
    }
}

// The refit schedule: node indices by depth (order), level d being order[off[d] .. off[d+1]).  The builder emits a
// node before its subtrees, so depths follow in one forward pass; refitting the levels deepest first sees every
// inner child already refitted.
inline void refit_levels(const std::vector<BvhNode> &nodes, std::vector<int32_t> &order, std::vector<int32_t> &off)
{
    std::vector<int32_t> depth(nodes.size(), 0);
    int32_t max_depth = 0;
    for (size_t i = 0; i < nodes.size(); i++)
        for (int k = 0; k < 2; k++)
            if (nodes[i].child[k] >= 0) {
                depth[(size_t)nodes[i].child[k]] = depth[i] + 1;
                max_depth = depth[i] + 1 > max_depth ? depth[i] + 1 : max_depth;
            }
    off.assign((size_t)max_depth + 2, 0);
    for (int32_t d : depth) off[(size_t)d + 1]++;
    for (size_t d = 1; d < off.size(); d++) off[d] += off[d - 1];
    order.assign(nodes.size(), 0);
    std::vector<int32_t> fill(off.begin(), off.end() - 1);
    for (size_t i = 0; i < nodes.size(); i++) order[(size_t)fill[(size_t)depth[i]]++] = (int32_t)i;
}

}  // namespace ert
