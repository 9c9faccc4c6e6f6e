// Test-only C shim around the triangle BVH builder (eraytracer_b200/csrc/bvh_build.cpp) plus a restatement in
// host C++ of the device walk (scan_tris_bvh in ert_device.cuh) over the same prune bounds (tri_walk.h).  The CPU
// suite uses it to check the one property the walk needs: a triangle the literal FP64 test accepts, and that
// could still win, lies in a leaf the walk enters or on the always-list.  Built with -ffp-contract=off, like the
// device code's -fmad=false.
#include <cstring>
#include <vector>

#include "../../eraytracer_b200/csrc/bvh_build.h"
#include "../../eraytracer_b200/csrc/tri_walk.h"

using namespace ert;

namespace {
// erl:402-455, as triangle_exact in ert_device.cuh
bool triangle_exact(const double O[3], const double D[3], const double *tr, double &t)
{
    const double e1[3] = {tr[3] - tr[0], tr[4] - tr[1], tr[5] - tr[2]};
    const double e2[3] = {tr[6] - tr[0], tr[7] - tr[1], tr[8] - tr[2]};
    const double p[3] = {D[1] * e2[2] - D[2] * e2[1], D[2] * e2[0] - D[0] * e2[2], D[0] * e2[1] - D[1] * e2[0]};
    const double det = e1[0] * p[0] + e1[1] * p[1] + e1[2] * p[2];
    if (det < 0.000001) return false;
    const double tv[3] = {O[0] - tr[0], O[1] - tr[1], O[2] - tr[2]};
    const double u = tv[0] * p[0] + tv[1] * p[1] + tv[2] * p[2];
    if (u < 0.0 || u > det) return false;
    const double q[3] = {tv[1] * e1[2] - tv[2] * e1[1], tv[2] * e1[0] - tv[0] * e1[2], tv[0] * e1[1] - tv[1] * e1[0]};
    const double v = D[0] * q[0] + D[1] * q[1] + D[2] * q[2];
    if (v < 0.0 || u + v > det) return false;
    t = (e2[0] * q[0] + e2[1] * q[1] + e2[2] * q[2]) / det;
    return true;
}

// leaf slots the walk enters with the incumbent's cull fixed at `cull` (the cull only falls during a walk)
void walk(const TriBvh &b, const TriRay &tr, double cull, std::vector<char> &entered)
{
    int stack[kBvhStack];
    int sp = 0, node = 0;
    while (true) {
        if (node >= 0) {
            const BvhNode &n = b.bvh.nodes[(size_t)node];
            double tn0, tn1;
            bool h0 = tri_slab(tr, n.c0x[0], n.c0x[1], n.c0y[0], n.c0y[1], n.c0z[0], n.c0z[1], cull, tn0);
            bool h1 = tri_slab(tr, n.c1x[0], n.c1x[1], n.c1y[0], n.c1y[1], n.c1z[0], n.c1z[1], cull, tn1);
            if (h0 && h1) {
                bool swap = tn1 < tn0;
                stack[sp++] = swap ? n.child[0] : n.child[1];
                node = swap ? n.child[1] : n.child[0];
                continue;
            } else if (h0) { node = n.child[0]; continue; }
            else if (h1) { node = n.child[1]; continue; }
        } else {
            int code = ~node;
            int first = code >> 3, cnt = (code & 7) + 1;
            for (int k = first; k < first + cnt; k++) entered[(size_t)k] = 1;
        }
        if (sp == 0) return;
        node = stack[--sp];
    }
}
}  // namespace

extern "C" {

void *tb_build(const double *tris, long long n)
{
    TriBvh *b = new TriBvh();
    build_triangle_bvh(tris, n, *b);
    return b;
}
void tb_free(void *p) { delete (TriBvh *)p; }
long long tb_n_always(void *p) { return (long long)((TriBvh *)p)->always.size(); }
long long tb_n_tree(void *p) { return (long long)((TriBvh *)p)->bvh.leaf_prim.size(); }
int tb_depth(void *p) { return ((TriBvh *)p)->bvh.depth; }
void tb_constants(void *p, double *out)
{
    out[0] = ((TriBvh *)p)->edge_max;
    out[1] = ((TriBvh *)p)->abs_max;
}

// For every ray and every triangle the literal test accepts (Distance t): the walk with the cull of an incumbent
// at Distance t must enter the triangle's leaf, unless it is on the always-list or the ray falls back to the
// linear scan.  stats[0] = accepted (ray, triangle) pairs, [1] = pairs missed, [2] = rays that fell back, [3] = first
// missed ray index (or -1).
void tb_check(void *p, const double *tris, long long n_tris, const double *rays, long long n_rays, int margins,
              long long *stats)
{
    const TriBvh &b = *(TriBvh *)p;
    std::vector<int> slot_of((size_t)n_tris, -1);
    for (size_t k = 0; k < b.bvh.leaf_prim.size(); k++) slot_of[(size_t)b.bvh.leaf_prim[k]] = (int)k;
    std::vector<char> entered(b.bvh.leaf_prim.size());
    stats[0] = stats[1] = stats[2] = 0;
    stats[3] = -1;
    for (long long r = 0; r < n_rays; r++) {
        const double *O = rays + 6 * r, *D = rays + 6 * r + 3;
        TriRay tr;
        const bool ok = tri_ray_setup(O, D, b.edge_max, b.abs_max, margins != 0, tr);
        if (!ok) stats[2]++;
        for (long long i = 0; i < n_tris; i++) {
            double t;
            if (!triangle_exact(O, D, tris + 9 * i, t)) continue;
            stats[0]++;
            if (!ok || slot_of[(size_t)i] < 0) continue;
            std::fill(entered.begin(), entered.end(), 0);
            walk(b, tr, tri_cull(tr, true, t), entered);
            if (!entered[(size_t)slot_of[(size_t)i]]) {
                stats[1]++;
                if (stats[3] < 0) stats[3] = r;
            }
        }
    }
}

// node array and leaf order of a sphere tree, for the digest that pins it
long long tb_sphere_tree(const double *centers, const double *radii, long long n, unsigned char *out, long long cap)
{
    Bvh b;
    build_sphere_bvh(centers, radii, n, b, kBvhLeafMax, kBvhTravCost);
    const size_t nb = b.nodes.size() * sizeof(BvhNode), lb = b.leaf_prim.size() * sizeof(int32_t);
    if ((long long)(nb + lb) <= cap) {
        memcpy(out, b.nodes.data(), nb);
        memcpy(out + nb, b.leaf_prim.data(), lb);
    }
    return (long long)(nb + lb);
}
}
