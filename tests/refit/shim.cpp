// Test-only C shim around the refit of ert_scene_update: the per-node refit and the level schedule of
// eraytracer_b200/csrc/scene_math.h (the code the device kernels of ert_update.cuh run), over trees made by
// bvh_build.cpp.  Built with -ffp-contract=off, like the device code's -fmad=false.
#include <cstring>
#include <vector>

#include "../../eraytracer_b200/csrc/bvh_build.h"
#include "../../eraytracer_b200/csrc/scene_math.h"

using namespace ert;

namespace {
// refit by levels, deepest first, as ert_api.cu launches upd_refit_level
template <typename LeafBox>
void refit(std::vector<BvhNode> &nodes, const LeafBox &leaf_box)
{
    std::vector<int32_t> order, off;
    refit_levels(nodes, order, off);
    for (int lvl = (int)off.size() - 2; lvl >= 0; lvl--)
        for (int32_t j = off[(size_t)lvl]; j < off[(size_t)lvl + 1]; j++) refit_node(nodes.data(), order[(size_t)j], leaf_box);
}

// stored child boxes that do not contain the box of a primitive below them
template <typename PrimBox>
long long violations(const std::vector<BvhNode> &nodes, const PrimBox &prim_box)
{
    long long bad = 0;
    // depth-first with the chain of ancestor boxes
    struct Frame { int32_t child; std::vector<float> chain; };
    std::vector<Frame> work;
    for (int k = 0; k < 2; k++) {
        float lo[3], hi[3];
        child_box(nodes[0], k, lo, hi);
        if (lo[0] > hi[0]) continue;
        work.push_back({nodes[0].child[k], {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]}});
    }
    while (!work.empty()) {
        Frame f = std::move(work.back());
        work.pop_back();
        if (f.child < 0) {
            const int32_t code = ~f.child, first = code >> 3, count = (code & 7) + 1;
            for (int32_t s = first; s < first + count; s++) {
                float lo[3], hi[3];
                prim_box(s, lo, hi);
                for (size_t b = 0; b < f.chain.size(); b += 6)
                    for (int a = 0; a < 3; a++)
                        if (lo[a] < f.chain[b + a] || hi[a] > f.chain[b + 3 + a]) { bad++; goto next_prim; }
            next_prim:;
            }
            continue;
        }
        for (int k = 0; k < 2; k++) {
            float lo[3], hi[3];
            child_box(nodes[(size_t)f.child], k, lo, hi);
            if (lo[0] > hi[0]) continue;
            Frame g{nodes[(size_t)f.child].child[k], f.chain};
            g.chain.insert(g.chain.end(), {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]});
            work.push_back(std::move(g));
        }
    }
    return bad;
}

struct Spheres {
    std::vector<double> s;      // [n][4] c, r
    Bvh bvh;
};
struct SphereBox {
    const Spheres *sp;
    void operator()(int slot, float lo[3], float hi[3]) const { sphere_box(&sp->s[4 * (size_t)sp->bvh.leaf_prim[(size_t)slot]], lo, hi); }
};
struct TriBox {
    const TriBvh *t;
    void operator()(int slot, float lo[3], float hi[3]) const { triangle_box(&t->leaf_tris[9 * (size_t)slot], lo, hi); }
};
}  // namespace

extern "C" {

void *rf_sphere_build(const double *c, const double *r, long long n)
{
    Spheres *sp = new Spheres();
    build_sphere_bvh(c, r, n, sp->bvh, kBvhLeafMax, kBvhTravCost);
    sp->s.resize((size_t)n * 4);
    for (long long i = 0; i < n; i++) {
        for (int a = 0; a < 3; a++) sp->s[4 * i + a] = c[3 * i + a];
        sp->s[4 * i + 3] = r[i];
    }
    return sp;
}
void rf_sphere_free(void *p) { delete (Spheres *)p; }

// new centres and radii, then the refit
void rf_sphere_refit(void *p, const double *c, const double *r)
{
    Spheres &sp = *(Spheres *)p;
    for (size_t i = 0; i < sp.s.size() / 4; i++) {
        for (int a = 0; a < 3; a++) sp.s[4 * i + a] = c[3 * i + a];
        sp.s[4 * i + 3] = r[i];
    }
    refit(sp.bvh.nodes, SphereBox{&sp});
}
long long rf_sphere_nodes(void *p, unsigned char *out, long long cap)
{
    const Bvh &b = ((Spheres *)p)->bvh;
    const size_t bytes = b.nodes.size() * sizeof(BvhNode);
    if ((long long)bytes <= cap) memcpy(out, b.nodes.data(), bytes);
    return (long long)bytes;
}
long long rf_sphere_violations(void *p)
{
    const Spheres &sp = *(Spheres *)p;
    return violations(sp.bvh.nodes, SphereBox{&sp});
}

void *rf_tri_build(const double *tris, long long n)
{
    TriBvh *t = new TriBvh();
    build_triangle_bvh(tris, n, *t);
    return t;
}
void rf_tri_free(void *p) { delete (TriBvh *)p; }

// new vertices: the leaf-ordered copy gathered again, the tree's constants recomputed, then the refit (what
// upd_triangles and upd_refit_level do).  Returns the largest |coordinate| of a tree triangle.
double rf_tri_refit(void *p, const double *tris)
{
    TriBvh &t = *(TriBvh *)p;
    double e_max = 0, a_max = 0;
    for (size_t k = 0; k < t.bvh.leaf_prim.size(); k++) {
        memcpy(&t.leaf_tris[9 * k], tris + 9 * (size_t)t.bvh.leaf_prim[k], 9 * sizeof(double));
        double e, m;
        triangle_extent(&t.leaf_tris[9 * k], e, m);
        e_max = d_max(e_max, e);
        a_max = d_max(a_max, m);
    }
    t.edge_max = e_max * (1.0 + 1.0 / 1099511627776.0);
    t.abs_max = a_max;
    refit(t.bvh.nodes, TriBox{&t});
    return a_max;
}
long long rf_tri_nodes(void *p, unsigned char *out, long long cap)
{
    const TriBvh &t = *(TriBvh *)p;
    const size_t bytes = t.bvh.nodes.size() * sizeof(BvhNode);
    if ((long long)bytes <= cap) memcpy(out, t.bvh.nodes.data(), bytes);
    return (long long)bytes;
}
void rf_tri_constants(void *p, double *out)
{
    out[0] = ((TriBvh *)p)->edge_max;
    out[1] = ((TriBvh *)p)->abs_max;
}
long long rf_tri_violations(void *p)
{
    const TriBvh &t = *(TriBvh *)p;
    return violations(t.bvh.nodes, TriBox{&t});
}

// the FP32 filter spheres of a scene, as flatten() and upd_spheres make them
void rf_filters(const double *c, const double *r, long long n, float *out)
{
    for (long long i = 0; i < n; i++) {
        float pad_c, eta_c;
        make_filter_sphere(c + 3 * i, r[i], out + 4 * i, pad_c, eta_c);
    }
}
}
