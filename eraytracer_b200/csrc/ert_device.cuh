// Device side of the eraytracer hot path for sm_100a.
//
// Numerical contract (see DESIGN.md "Exactness"):
//  * Every value that feeds a discrete decision of the reference — ray origins and
//    directions, hit distances, hit points, normals, the comparisons of
//    raytracer.erl:319/378/381/416/426/434/464/468 — is computed in IEEE double in the
//    literal operation order of raytracer.erl.  This translation unit is compiled with
//    -fmad=false so no double (or float) multiply-add is contracted; BEAM never fuses.
//  * FP32 appears only in *conservative filters* (ray/sphere discriminant with error
//    slack, ray/AABB slabs with margins).  A filter may let a non-hit through, never
//    drop a hit; whatever passes is decided by the FP64 literal test.  FFMAs in the
//    filters are written explicitly with __fmaf_rn.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "bvh_build.h"
#include "light_grid.h"
#include "tri_walk.h"

namespace ert {

// ------------------------------------------------------------------ scene on device
enum ObjType : int { OBJ_SPHERE = 0, OBJ_PLANE = 1, OBJ_TRIANGLE = 2 };
__host__ __device__ inline int obj_code(int type, int index) { return (type << 28) | index; }
__host__ __device__ inline int obj_type(int code) { return (code >> 28) & 3; }
__host__ __device__ inline int obj_index(int code) { return code & 0x0fffffff; }

struct DevScene {
    // lights in list order: [n][9] = diffuse rgb, location xyz, specular rgb (erl:81)
    int n_lights;
    const double *lights;
    // planes / triangles: decided directly in FP64 (few of them, unbounded / t<0 quirks)
    int n_planes;
    const double *planes;        // [n][4] normal xyz, distance
    const double *plane_mat;     // [n][6]
    const int *plane_order;
    int n_tris;
    const double *tris;          // [n][9] v1 v2 v3
    const double *tri_mat;       // [n][6]
    const int *tri_order;
    // spheres, in list order among spheres
    int n_spheres;
    const double4 *sph_exact;    // {cx, cy, cz, radius}
    const double *sph_mat;       // [n][6] colour rgb, specular_power, shininess, reflectivity
    const double *sph_refl;      // [n] reflectivity again, dense: the emitters of the wavefront need nothing else of the
                                 // material, and 8 bytes per sphere stay in L2 where 48-byte rows do not
    const int *sph_order;        // list position
    const float4 *sph_filter;    // {fl(cx), fl(cy), fl(cz), R} — see make_filter_sphere()
    const float4 *sph_pairs;     // the same list pair-interleaved for the packed scan (ert_scan.cuh): spheres 2p, 2p+1 as
                                 // {cx0,cx1,cy0,cy1},{cz0,cz1,R0,R1}; padded to whole tiles with spheres that never pass
    // BVH over spheres
    const BvhNode *nodes;
    int n_nodes;
    const float4 *leaf_filter;   // filter spheres in leaf order
    const int *leaf_sph;         // leaf slot -> sphere index
    // filter constants of the scene
    float r_max;                 // largest |radius|
    float pad_c_max;             // largest centre-rounding pad folded into any R
    float eta_c_max;             // largest centre rounding error bound
    float abs_max;               // largest |coordinate| of any sphere box
    // uniform grid over the sphere bounds, used only to order the wavefront queues
    float grid_lo[3], grid_scale[3];
    // direction grids of the first lg_count lights (light_grid.h): shadow-ray candidates by direction
    const struct LightGridDev *lgrids;
    int lg_count;
    // uniform cell grid over the spheres (cell_grid.h): path-ray candidates by 3-D DDA
    struct CellGridDev {
        const uint4 *blocks;         // [rx*ry*rz][2] 128-byte CellBlock (cell_grid.h): 6 filter spheres, 6 indices, count, overflow
        const float4 *over_filter;   // filter spheres of the lists longer than a block, in groups of four
        const int *over_sph;         // overflow entry -> sphere index
        const int *big;              // spheres every ray tests (too large for the cells)
        int n_big, enabled;
        int rx, ry, rz;
        float lo[3], hi[3];
        float cs, eps;
    } cg;
    // BVH over triangles (scenes with >= kTriBvhMin triangles): walked by the kernels instantiated with TRI
    const BvhNode *tri_nodes;
    const double *tri_leaf;      // [slot][9] v1 v2 v3 in leaf order
    const int *tri_leaf_id;      // leaf slot -> triangle index
    const int *tri_always;       // triangles outside the tree: every ray tests them
    int n_tri_tree, n_tri_always;
    double tri_edge_max, tri_abs_max;   // the tree's constants of tri_walk.h
};

struct LightGridDev {
    const unsigned int *cell_off;    // [6*res*res + 1]
    const LightGridCand *head;       // [6*res*res] the first (nearest) candidate of every cell, its pad[] holding
                                     // the range [pad[0], pad[1]) of the remaining ones in `cand`; an empty cell
                                     // has dmin = +inf: one fetch per shadow ray instead of offsets, then entry
    const LightGridCand *cand;       // nearest first inside a cell
    const int *always;               // spheres that contain the light: candidates of every ray
    int n_always;
    int res;
};

struct FrameParams {
    int width, height, depth, format;
    int band_rows, n_parts, part, local_rows;
    double cam[3];
    double focal;                // focal_length(fov, screen_width), computed on the host with glibc tan
    double screen_w, screen_h;
    void *out;                   // compact framebuffer of this part: local_rows * width pixels
    unsigned long long *counters;
    // ray space: pixel (X, Y) casts the ray of pixel (ss*X + ss_i, ss*Y + ss_j) of the (ss*width) x (ss*height)
    // frame (one sample pass of a supersampled frame; a plain frame has ss = 1, ss_i = ss_j = 0).  Last in the
    // struct, with ray_w = ss*width and ray_h = ss*height as exact doubles: the existing kernels keep their registers.
    int ss, ss_i, ss_j;
    double ray_w, ray_h;
    // ERT_FLAG_CAMERA_ROTATION with a matrix other than the identity: primary directions are turned by the row-major
    // rot (include/ert_b200.h).  Appended so that the fields above keep their offsets.
    double rot[9];
    int rotate;
};

#ifdef ERT_PROBE
enum Counter : int { CNT_RAYS = 0, CNT_FILTER = 1, CNT_BOX = 2, CNT_EXACT_SPH = 3, CNT_EXACT_OTHER = 4, CNT_CELL = 5, CNT_PROBE = 8, CNT_N = 16 };
#else
enum Counter : int { CNT_RAYS = 0, CNT_FILTER = 1, CNT_BOX = 2, CNT_EXACT_SPH = 3, CNT_EXACT_OTHER = 4, CNT_CELL = 5, CNT_N = 8 };
#endif
constexpr int kCounterSets = 2;      // [0]: megakernels and wf_trace_path*, [1]: wf_trace_shadow

// ------------------------------------------------------------------ FP64 literal algebra
struct d3 { double x, y, z; };
__device__ __forceinline__ d3 mk(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
// erl:524-527
__device__ __forceinline__ d3 vadd(d3 a, d3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
// erl:529-532
__device__ __forceinline__ d3 vsub(d3 a, d3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
// erl:540-541
__device__ __forceinline__ d3 vscale(d3 a, double s) { return mk(a.x * s, a.y * s, a.z * s); }
// erl:543-544
__device__ __forceinline__ d3 vcmul(d3 a, d3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
// erl:546-547
__device__ __forceinline__ double vdot(d3 a, d3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
// erl:549-552
__device__ __forceinline__ d3 vcross(d3 a, d3 b)
{
    return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// erl:554-560
__device__ __forceinline__ d3 vnormalize(d3 a)
{
    double mag = sqrt(a.x * a.x + a.y * a.y + a.z * a.z);
    if (mag == 0.0) return mk(0.0, 0.0, 0.0);
    return vscale(a, 1.0 / mag);
}
// erl:562-563
__device__ __forceinline__ d3 vneg(d3 a) { return mk(-a.x, -a.y, -a.z); }
// erl:568-573
__device__ __forceinline__ d3 vbounce(d3 v, d3 n) { return vadd(vscale(n, 2.0 * vdot(n, vneg(v))), v); }
// lists:max([0, X]) erl:275, 290
__device__ __forceinline__ double max0(double x) { return x > 0.0 ? x : 0.0; }

// 32-byte records in ONE 256-bit transaction (LDG.E.256 / STG.E.256, sm_100): an FP64 sphere {cx, cy, cz, r}
// (read-only for the life of a kernel), and the queue records one kernel writes for the next.
__device__ __forceinline__ double4 ld_sphere(const double4 *p)
{
    double4 r;
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ double4 ld_rec32(const void *p)
{
    double4 r;
    asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
    return r;
}
// the same, read once (evict-first): queue entries must not push the scene out of L1/L2
__device__ __forceinline__ double4 ld_rec32_cs(const void *p)
{
    double4 r;
    asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_rec32(void *p, double a, double b, double c, double d)
{
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

struct Hit {
    double t;
    int order;     // list position of the object
    int obj;       // obj_code or -1 for 'none'
};
// strict '>' of erl:319 over list order == lexicographic (t, order)
__device__ __forceinline__ bool better(double t, int order, const Hit &h)
{
    return h.obj < 0 || t < h.t || (t == h.t && order < h.order);
}

// erl:364-397 — literal.  `a` is Xd*Xd + Yd*Yd + Zd*Zd of the same ray.
__device__ __forceinline__ bool sphere_exact(d3 O, d3 D, double a, double4 s, double &t)
{
    double ox = O.x - s.x, oy = O.y - s.y, oz = O.z - s.z;
    double b = 2.0 * (D.x * ox + D.y * oy + D.z * oz);
    double c = ox * ox + oy * oy + oz * oz - s.w * s.w;
    double disc = b * b - 4.0 * a * c;
    if (disc >= 0.001) {
        double sq = sqrt(disc);
        double t0 = (-b + sq) / 2.0;
        double t1 = (-b - sq) / 2.0;
        if (t0 >= 0.0 && t1 >= 0.0) {
            t = t0 < t1 ? t0 : t1;
            return true;
        }
    }
    return false;
}

// erl:461-480
__device__ __forceinline__ bool plane_exact(d3 O, d3 D, const double *p, double &t)
{
    d3 n = mk(p[0], p[1], p[2]);
    double vd = vdot(n, D);
    if (vd < 0.0) {
        double v0 = -(vdot(n, O) + p[3]);
        double dist = v0 / vd;
        if (dist < 0.001) return false;
        t = dist;
        return true;
    }
    return false;
}

// erl:402-455
__device__ __forceinline__ bool triangle_exact(d3 O, d3 D, const double *tr, double &t)
{
    d3 v1 = mk(tr[0], tr[1], tr[2]), v2 = mk(tr[3], tr[4], tr[5]), v3 = mk(tr[6], tr[7], tr[8]);
    d3 e1 = vsub(v2, v1), e2 = vsub(v3, v1);
    d3 p = vcross(D, e2);
    double det = vdot(e1, p);
    if (det < 0.000001) return false;
    d3 tv = vsub(O, v1);
    double u = vdot(tv, p);
    if (u < 0.0 || u > det) return false;
    d3 q = vcross(tv, e1);
    double v = vdot(D, q);
    if (v < 0.0 || u + v > det) return false;
    t = vdot(e2, q) / det;
    return true;
}

template <bool COUNT>
struct Tally {
    unsigned int filter = 0, box = 0, exact_sph = 0, exact_other = 0, cell = 0;
#ifdef ERT_PROBE
    unsigned int p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
};
template <>
struct Tally<false> {};
#define TALLY(field) do { if constexpr (COUNT) tl.field++; } while (0)
#ifdef ERT_PROBE
#define PROBE(k, n) do { if constexpr (COUNT) tl.p[k] += (n); } while (0)
#else
#define PROBE(k, n) do { } while (0)
#endif

// one triangle through the literal test, folded into `best`
template <bool COUNT>
__device__ __forceinline__ void try_triangle(const DevScene &sc, d3 O, d3 D, const double *tr, int i, int skip_obj,
                                             Hit &best, Tally<COUNT> &tl)
{
    int code = obj_code(OBJ_TRIANGLE, i);
    if (code == skip_obj) return;
    double t;
    TALLY(exact_other);
    if (triangle_exact(O, D, tr, t)) {
        int ord = sc.tri_order[i];
        if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
    }
}

// The triangles of a scene with a triangle BVH (tri_walk.h): the always-list, then a front-to-back walk of the
// whole line from -inf that leaves a node when its entry parameter is beyond the incumbent's cull.  With ANY the
// walk stops at the first improvement of the incumbent (shadow queries, which start from their target).
template <bool COUNT>
__device__ __noinline__ void scan_tris_bvh(const DevScene &sc, d3 O, d3 D, Hit &best, int skip_obj, bool any,
                                           Tally<COUNT> &tl)
{
    for (int k = 0; k < sc.n_tri_always; k++) {
        const int i = __ldg(sc.tri_always + k);
        try_triangle<COUNT>(sc, O, D, sc.tris + 9 * (size_t)i, i, skip_obj, best, tl);
        if (any && best.obj != skip_obj) return;
    }
    const double Oa[3] = {O.x, O.y, O.z}, Da[3] = {D.x, D.y, D.z};
    TriRay tr;
    if (!tri_ray_setup(Oa, Da, sc.tri_edge_max, sc.tri_abs_max, true, tr)) {
        // the bounds do not hold for this ray: every tree triangle
        for (int k = 0; k < sc.n_tri_tree; k++) {
            try_triangle<COUNT>(sc, O, D, sc.tri_leaf + 9 * (size_t)k, __ldg(sc.tri_leaf_id + k), skip_obj, best, tl);
            if (any && best.obj != skip_obj) return;
        }
        return;
    }
    int stack[kBvhStack];
    int sp = 0;
    int node = 0;
    double cull = tri_cull(tr, best.obj >= 0, best.t);
    while (true) {
        if (node >= 0) {
            const float4 *np = reinterpret_cast<const float4 *>(sc.tri_nodes + node);
            float4 a0 = __ldg(np), a1 = __ldg(np + 1), a2 = __ldg(np + 2);
            int4 ch = __ldg(reinterpret_cast<const int4 *>(np + 3));
            double tn0, tn1;
            if constexpr (COUNT) tl.box += 2;
            bool h0 = tri_slab(tr, a0.x, a0.y, a0.z, a0.w, a2.x, a2.y, cull, tn0);
            bool h1 = tri_slab(tr, a1.x, a1.y, a1.z, a1.w, a2.z, a2.w, cull, tn1);
            if (h0 && h1) {
                bool swap = tn1 < tn0;
                int nearc = swap ? ch.y : ch.x, farc = swap ? ch.x : ch.y;
                if (sp < kBvhStack) stack[sp++] = farc;      // always true: ert_scene_create rejects trees of depth >= kBvhStack
                node = nearc;
                continue;
            } else if (h0) { node = ch.x; continue; }
            else if (h1) { node = ch.y; continue; }
        } else {
            int code = ~node;
            int first = code >> 3, cnt = (code & 7) + 1;
            for (int k = first; k < first + cnt; k++)
                try_triangle<COUNT>(sc, O, D, sc.tri_leaf + 9 * (size_t)k, __ldg(sc.tri_leaf_id + k), skip_obj, best, tl);
            if (any && best.obj != skip_obj) return;
            cull = tri_cull(tr, best.obj >= 0, best.t);
        }
        if (sp == 0) return;
        node = stack[--sp];
    }
}

// planes and triangles (erl:353-356): always FP64, list order kept through `order`.  TRI: the scene has a
// triangle BVH and its triangles are reached through scan_tris_bvh.
template <bool COUNT, bool TRI = false>
__device__ __forceinline__ void scan_others(const DevScene &sc, d3 O, d3 D, Hit &best, int skip_obj,
                                            Tally<COUNT> &tl)
{
    if constexpr (TRI) {
        scan_tris_bvh<COUNT>(sc, O, D, best, skip_obj, false, tl);
    } else {
        for (int i = 0; i < sc.n_tris; i++) {
            int code = obj_code(OBJ_TRIANGLE, i);
            if (code == skip_obj) continue;
            double t;
            TALLY(exact_other);
            if (triangle_exact(O, D, sc.tris + 9 * i, t)) {
                int ord = sc.tri_order[i];
                if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
            }
        }
    }
    for (int i = 0; i < sc.n_planes; i++) {
        int code = obj_code(OBJ_PLANE, i);
        if (code == skip_obj) continue;
        double t;
        TALLY(exact_other);
        if (plane_exact(O, D, sc.planes + 4 * i, t)) {
            int ord = sc.plane_order[i];
            if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
        }
    }
}

// Planes and triangles of a shadow query (erl:256-267): `best` holds the target and the only question is whether
// something beats its (Distance, list position).  A plane certainly farther than the target is dismissed before the
// division of erl:468: with Vd < 0, Distance = V0 / Vd >= X  <=>  V0 <= X * Vd, and X = Distance(target) * (1 + 1e-9)
// leaves seven decimal orders for the roundings of the products.  Everything nearer goes through the literal test.
template <bool COUNT, bool TRI = false>
__device__ __forceinline__ void scan_others_shadow(const DevScene &sc, d3 O, d3 D, Hit &best, int skip_obj,
                                                   Tally<COUNT> &tl)
{
    if constexpr (TRI) {
        scan_tris_bvh<COUNT>(sc, O, D, best, skip_obj, true, tl);
    } else {
        for (int i = 0; i < sc.n_tris; i++) {
            int code = obj_code(OBJ_TRIANGLE, i);
            if (code == skip_obj) continue;
            double t;
            TALLY(exact_other);
            if (triangle_exact(O, D, sc.tris + 9 * i, t)) {
                int ord = sc.tri_order[i];
                if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
            }
        }
    }
    for (int i = 0; i < sc.n_planes; i++) {
        int code = obj_code(OBJ_PLANE, i);
        if (code == skip_obj) continue;
        TALLY(exact_other);
        const double *p = sc.planes + 4 * i;
        const d3 n = mk(p[0], p[1], p[2]);
        const double vd = vdot(n, D);
        if (!(vd < 0.0)) continue;                                   // erl:464
        if (best.obj >= 0) {
            if (best.t <= 0.0) continue;                             // a plane hit has Distance >= 0.001 (erl:469)
            const double v0 = -(vdot(n, O) + p[3]);
            if (v0 <= (best.t * (1.0 + 1e-9)) * vd) continue;        // certainly beyond the target
        }
        double t;
        if (plane_exact(O, D, p, t)) {
            int ord = sc.plane_order[i];
            if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
        }
    }
}

// the literal test of one known object (used to seed shadow queries with their target)
__device__ __forceinline__ bool object_exact(const DevScene &sc, int code, d3 O, d3 D, double a, double &t)
{
    int i = obj_index(code);
    switch (obj_type(code)) {
    case OBJ_SPHERE: return sphere_exact(O, D, a, ld_sphere(sc.sph_exact + i), t);
    case OBJ_PLANE: return plane_exact(O, D, sc.planes + 4 * i, t);
    default: return triangle_exact(O, D, sc.tris + 9 * i, t);
    }
}
__device__ __forceinline__ int object_order(const DevScene &sc, int code)
{
    int i = obj_index(code);
    switch (obj_type(code)) {
    case OBJ_SPHERE: return sc.sph_order[i];
    case OBJ_PLANE: return sc.plane_order[i];
    default: return sc.tri_order[i];
    }
}

// ------------------------------------------------------------------ FP32 conservative filter
// Constants (u = 2^-24).  Derivation in DESIGN.md "Filter bounds".
#define ERT_U        5.9604644775390625e-8f          /* 2^-24 */
#define ERT_KD       1.0000019073486328125           /* 1 + 2^-19: direction inflation */
#define ERT_REL16    1.52587890625e-5f               /* 2^-16 */
#define ERT_REL17    7.62939453125e-6f               /* 2^-17 */

struct FRay {
    float ox, oy, oz;       // fl32(O)
    float dx, dy, dz;       // fl32(D/|D| * KD)
    float theta;            // stage 1 accepts iff !(v < -theta)
    float bcull;            // stage 2 rejects spheres with b < -bcull (entirely behind)
    float pad2;             // absolute slack under the stage-2 square root
    float ix, iy, iz;       // slab reciprocals
    float nx, ny, nz;       // near-plane constants  -(o + s*m) * inv
    float fx, fy, fz;       // far-plane constants   -(o - s*m) * inv
    float m4;               // absolute slack of the cull distance
    double inv_sqrt_a;      // reference distance -> geometric distance
    double a;               // Xd*Xd + Yd*Yd + Zd*Zd (literal, for the exact test)
};

__device__ __forceinline__ float clamp_dir(float d)
{
    // keep 1/d finite; 1e-20 is far below any direction component that matters
    if (fabsf(d) < 1e-20f) return d < 0.f ? -1e-20f : 1e-20f;
    return d;
}

// The range of the filter bounds: a ray may use the FP32 filters, slabs and cells iff |o|_inf + abs_max lies below
// this.  Then |c - o|^2 <= 3e34 and every slab constant (|o| + m) / d with |d| >= 1e-20 stays far inside float.
// Beyond it |c - o|^2 - R can overflow to +Inf and stage 1 would reject a sphere the ray hits (DESIGN.md "Filter
// bounds"), so make_fray / make_sray return false: a walk decides every sphere with the literal test instead
// (scan_spheres_instead), and the scans that have no tree to leave pass every sphere through the filter (make_fray
// sets its constants so that both stages do; wf_scan sets its own stage-1 threshold).
constexpr float kFilterRange = 1e17f;

__device__ __forceinline__ bool make_fray(const DevScene &sc, d3 O, d3 D, FRay &f, bool want_slabs)
{
    f.a = D.x * D.x + D.y * D.y + D.z * D.z;
    double inv = 1.0 / sqrt(f.a);
    f.inv_sqrt_a = inv;
    f.ox = (float)O.x; f.oy = (float)O.y; f.oz = (float)O.z;
    double k = inv * ERT_KD;
    f.dx = (float)(D.x * k); f.dy = (float)(D.y * k); f.dz = (float)(D.z * k);
    // eta_o: twice the actual rounding error of the origin
    float eo = 2.0f * fmaxf(fmaxf(fabsf((float)(O.x - (double)f.ox)), fabsf((float)(O.y - (double)f.oy))),
                            fabsf((float)(O.z - (double)f.oz)));
    eo *= 1.0001f;
    f.theta = 16.0f * sc.r_max * eo + 8.0f * eo * (eo / ERT_U);
    f.bcull = 2.0f * (5.0f * ERT_U * sc.r_max + 2.0f * eo + 2.0f * sc.eta_c_max);
    f.pad2 = 2.0f * (f.theta + sc.pad_c_max) + 1e-30f;
    float oabs = fmaxf(fmaxf(fabsf(f.ox), fabsf(f.oy)), fabsf(f.oz));
    float m = eo + 32.0f * ERT_U * (oabs + sc.abs_max);
    f.m4 = 4.0f * m;
    if (want_slabs) {
        float dx = clamp_dir(f.dx), dy = clamp_dir(f.dy), dz = clamp_dir(f.dz);
        f.ix = 1.0f / dx; f.iy = 1.0f / dy; f.iz = 1.0f / dz;
        float sx = dx < 0.f ? -m : m, sy = dy < 0.f ? -m : m, sz = dz < 0.f ? -m : m;
        // near plane pushed outward by m, far plane pushed outward by m
        f.nx = -(f.ox + sx) * f.ix; f.ny = -(f.oy + sy) * f.iy; f.nz = -(f.oz + sz) * f.iz;
        f.fx = -(f.ox - sx) * f.ix; f.fy = -(f.oy - sy) * f.iy; f.fz = -(f.oz - sz) * f.iz;
    }
    // false for NaN and Inf as well; out of range, both stages pass every sphere
    const bool in_range = oabs + sc.abs_max < kFilterRange;
    if (!in_range) f.theta = f.bcull = f.m4 = __int_as_float(0x7f800000);
    return in_range;
}

// reference Distance of the incumbent -> filter-space cull distance (upper bound)
template <class R>
__device__ __forceinline__ float cull_from(const R &f, const Hit &best)
{
    if (best.obj < 0) return __int_as_float(0x7f800000);
    double s = best.t * f.inv_sqrt_a;
    float sf = __double2float_ru(s);
    return sf + fabsf(sf) * ERT_REL16 + f.m4;
}

// Stage 1: 10 FP32-pipe instructions (3 FADD, 1 FMUL, 6 FFMA) + 1 compare.
// v = b^2 - (|oc|^2 - R);  accept iff !(v < -theta).
template <class R>
__device__ __forceinline__ bool filter_stage1(const R &f, float4 s, float &b, float &v)
{
    float cx = s.x - f.ox, cy = s.y - f.oy, cz = s.z - f.oz;
    b = __fmaf_rn(f.dz, cz, __fmaf_rn(f.dy, cy, f.dx * cx));
    float w = __fmaf_rn(cx, cx, __fmaf_rn(cy, cy, __fmaf_rn(cz, cz, -s.w)));
    v = __fmaf_rn(b, b, -w);
    return !(v < -f.theta);
}

// Stage 2 (only for stage-1 survivors): behind-the-origin and beyond-the-incumbent culls.
template <class R>
__device__ __forceinline__ bool filter_stage2(const R &f, float4 s, float b, float v, float cull)
{
    if (b < -f.bcull) return false;
    if (cull == __int_as_float(0x7f800000)) return true;      // no incumbent yet: nothing is "beyond" it
    float arg = fmaxf(v, 0.f) + ERT_REL17 * (b * b + s.w) + f.pad2;
    float s_lo = b - fabsf(b) * ERT_REL16 - sqrtf(arg) * 1.000001f - f.bcull;
    return !(s_lo > cull);
}

// One filtered sphere: filter, then the literal FP64 test on survivors.
template <bool COUNT>
__device__ __forceinline__ void try_sphere(const DevScene &sc, const FRay &f, d3 O, d3 D, float4 fs, int sph,
                                           int skip_obj, Hit &best, float &cull, Tally<COUNT> &tl)
{
    float b, v;
    TALLY(filter);
    if (!filter_stage1(f, fs, b, v)) return;
    if (!filter_stage2(f, fs, b, v, cull)) return;
    int code = obj_code(OBJ_SPHERE, sph);
    if (code == skip_obj) return;
    double t;
    TALLY(exact_sph);
    if (sphere_exact(O, D, f.a, ld_sphere(sc.sph_exact + sph), t)) {
        int ord = sc.sph_order[sph];
        if (better(t, ord, best)) {
            best.t = t; best.order = ord; best.obj = code;
            cull = cull_from(f, best);
        }
    }
}

// ------------------------------------------------------------------ nearest hit: three strategies
// All take an incumbent `best` (none, or the shadow target) and improve it.  With ANY set the
// search may stop at the first improvement (shadow queries only need to know whether one exists).

// ERT_ACCEL_EXACT: every sphere through the literal test.
template <bool COUNT>
__device__ __forceinline__ void scan_spheres_exact(const DevScene &sc, d3 O, d3 D, double a, Hit &best,
                                                   int skip_obj, bool any, int seed_obj, Tally<COUNT> &tl)
{
    for (int s = 0; s < sc.n_spheres; s++) {
        int code = obj_code(OBJ_SPHERE, s);
        if (code == skip_obj) continue;
        double t;
        TALLY(exact_sph);
        if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + s), t)) {
            int ord = sc.sph_order[s];
            if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
        }
        if (any && best.obj != seed_obj) return;
    }
}

__device__ __forceinline__ bool slab_hit(const FRay &f, float lox, float hix, float loy, float hiy, float loz,
                                         float hiz, float cull, float &tnear)
{
    float nx = f.dx < 0.f ? hix : lox, fx = f.dx < 0.f ? lox : hix;
    float ny = f.dy < 0.f ? hiy : loy, fy = f.dy < 0.f ? loy : hiy;
    float nz = f.dz < 0.f ? hiz : loz, fz = f.dz < 0.f ? loz : hiz;
    float t0x = __fmaf_rn(nx, f.ix, f.nx), t1x = __fmaf_rn(fx, f.ix, f.fx);
    float t0y = __fmaf_rn(ny, f.iy, f.ny), t1y = __fmaf_rn(fy, f.iy, f.fy);
    float t0z = __fmaf_rn(nz, f.iz, f.nz), t1z = __fmaf_rn(fz, f.iz, f.fz);
    tnear = fmaxf(fmaxf(t0x, t0y), fmaxf(t0z, 0.f));
    float tfar = fminf(fminf(t1x, t1y), fminf(t1z, cull));
    // relative slack for the roundings of the six FFMAs
    return tnear - fabsf(tnear) * ERT_REL16 <= tfar + fabsf(tfar) * ERT_REL16;
}

// A ray beyond the filter's range (make_fray / make_sray returned false) decides every sphere with the literal test,
// as ERT_ACCEL_EXACT does: no filter, box, cell or direction cell.  `any`: a shadow query seeded with its target,
// which may stop at the first improvement.  Inlined (as a call, its ABI made ptxas spill in the cell-grid path
// kernels) and kept to one rolled loop, so that the kernels that never take it keep their size.
__device__ __forceinline__ Hit scan_spheres_instead(const DevScene *scp, d3 O, d3 D, Hit best, int skip_obj, bool any,
                                                    int seed_obj)
{
    const DevScene &sc = *scp;
    const double a = D.x * D.x + D.y * D.y + D.z * D.z;
#pragma unroll 1
    for (int s = 0; s < sc.n_spheres; s++) {
        const int code = obj_code(OBJ_SPHERE, s);
        double t;
        if (code != skip_obj && sphere_exact(O, D, a, ld_sphere(sc.sph_exact + s), t)) {
            const int ord = sc.sph_order[s];
            if (better(t, ord, best)) { best.t = t; best.order = ord; best.obj = code; }
        }
        if (any && best.obj != seed_obj) break;
    }
    return best;
}

// ERT_ACCEL_BVH
template <bool COUNT>
__device__ __forceinline__ void scan_spheres_bvh(const DevScene &sc, d3 O, d3 D, const FRay &f, Hit &best,
                                                 int skip_obj, bool any, int seed_obj, Tally<COUNT> &tl)
{
    int stack[kBvhStack];
    int sp = 0;
    int node = 0;
    float cull = cull_from(f, best);
    while (true) {
        if (node >= 0) {
            const float4 *np = reinterpret_cast<const float4 *>(sc.nodes + node);
            float4 a0 = __ldg(np), a1 = __ldg(np + 1), a2 = __ldg(np + 2);
            int4 ch = __ldg(reinterpret_cast<const int4 *>(np + 3));
            float tn0, tn1;
            if constexpr (COUNT) tl.box += 2;
            bool h0 = slab_hit(f, a0.x, a0.y, a0.z, a0.w, a2.x, a2.y, cull, tn0);
            bool h1 = slab_hit(f, a1.x, a1.y, a1.z, a1.w, a2.z, a2.w, cull, tn1);
            if (h0 && h1) {
                bool swap = tn1 < tn0;
                int nearc = swap ? ch.y : ch.x, farc = swap ? ch.x : ch.y;
                if (sp < kBvhStack) stack[sp++] = farc;      // always true: ert_scene_create rejects trees of depth >= kBvhStack
                node = nearc;
                continue;
            } else if (h0) { node = ch.x; continue; }
            else if (h1) { node = ch.y; continue; }
        } else {
            int code = ~node;
            int first = code >> 3, cnt = (code & 7) + 1;
            for (int k = 0; k < cnt; k++) {
                float4 fs = __ldg(sc.leaf_filter + first + k);
                try_sphere<COUNT>(sc, f, O, D, fs, __ldg(sc.leaf_sph + first + k), skip_obj, best, cull, tl);
            }
            if (any && best.obj != seed_obj) return;
        }
        if (sp == 0) return;
        node = stack[--sp];
    }
}

// ------------------------------------------------------------------ per-pixel state machine
// One converged "resolve a ray" site serves path rays and shadow rays of all lanes.
struct Pix {
    d3 O, D;            // current path ray (erl:180-184 / 219-221)
    d3 P, N;            // current hit location and normal
    d3 S;               // sum over lights of (LightColour (*) (Diffuse+Specular)) * Shadow at this hit
    d3 C;               // pixel colour so far
    double W;           // product over earlier bounces of (number of lights * reflectivity)
    int hit_obj, hit_order;
    int phase;          // 0: path ray; l+1: shadow ray of light l
    int bounce;
    int rays;
    bool alive;
};

struct Query {
    d3 O, D;
    Hit best;
    int seed_obj;       // incumbent object the query starts from (-1 none)
    bool any;           // stop at the first improvement
    bool need;          // false: nothing to search (lane idle or target missed)
};

// erl:486-511, with X/Width and Y/Height as at erl:95-97 in ray space (the host keeps ss*width, ss*height <= INT32_MAX)
__device__ __forceinline__ void primary_ray(const FrameParams &fp, int X, int Y, d3 &O, d3 &D)
{
    double x = (double)(X * fp.ss + fp.ss_i) / fp.ray_w;
    double y = (double)(Y * fp.ss + fp.ss_j) / fp.ray_h;
    d3 loc = mk(fp.cam[0], fp.cam[1], fp.cam[2]);
    d3 acc = loc;
    acc = vadd(vscale(mk(0.0, 0.0, 1.0), fp.focal), acc);
    acc = vadd(mk((x - 0.5) * fp.screen_w, 0.0, 0.0), acc);
    acc = vadd(mk(0.0, (y - 0.5) * fp.screen_h, 0.0), acc);
    O = loc;
    d3 v = vsub(acc, loc);
    if (fp.rotate) {
        // d_i = (M[i][0]*v.x + M[i][1]*v.y) + M[i][2]*v.z, uncontracted (-fmad=false)
        const double *m = fp.rot;
        v = mk((m[0] * v.x + m[1] * v.y) + m[2] * v.z, (m[3] * v.x + m[4] * v.y) + m[5] * v.z,
               (m[6] * v.x + m[7] * v.y) + m[8] * v.z);
    }
    D = vnormalize(v);
}

__device__ __forceinline__ void pix_init(Pix &p, const DevScene &sc, const FrameParams &fp, int X, int Y, bool inside)
{
    p.C = mk(0.0, 0.0, 0.0);
    p.S = mk(0.0, 0.0, 0.0);
    p.P = p.N = mk(0.0, 0.0, 0.0);
    p.W = 1.0;
    p.phase = 0;
    p.bounce = 0;
    p.rays = 0;
    p.hit_obj = -1;
    p.hit_order = -1;
    // erl:186-187: depth 0 is black without tracing; no lights => the fold at erl:211-252 is (0,0,0)
    p.alive = inside && fp.depth > 0;
    if (inside) primary_ray(fp, X, Y, p.O, p.D);
    else { p.O = mk(0, 0, 0); p.D = mk(0, 0, 1); }
}

__device__ __forceinline__ double reflectivity_of(const DevScene &sc, int code)
{
    int i = obj_index(code);
    switch (obj_type(code)) {
    case OBJ_SPHERE: return __ldg(sc.sph_refl + i);
    case OBJ_PLANE: return sc.plane_mat[6 * (size_t)i + 5];
    default: return sc.tri_mat[6 * (size_t)i + 5];
    }
}

__device__ __forceinline__ const double *material_ptr(const DevScene &sc, int code)
{
    int i = obj_index(code);
    switch (obj_type(code)) {
    case OBJ_SPHERE: return sc.sph_mat + 6 * (size_t)i;
    case OBJ_PLANE: return sc.plane_mat + 6 * (size_t)i;
    default: return sc.tri_mat + 6 * (size_t)i;
    }
}

// Builds the next query of this pixel.
__device__ __forceinline__ void pix_prepare(const Pix &p, const DevScene &sc, Query &q)
{
    q.best.obj = -1; q.best.t = 0.0; q.best.order = 0x7fffffff;
    q.seed_obj = -1;
    q.any = false;
    q.need = p.alive;
    if (!p.alive) { q.O = p.O; q.D = p.D; return; }
    if (p.phase == 0) {
        q.O = p.O; q.D = p.D;
    } else {
        // shadow_factor erl:256-260: from the light towards the hit location
        const double *l = sc.lights + 9 * (p.phase - 1);
        q.O = mk(l[3], l[4], l[5]);
        q.D = vnormalize(vsub(p.P, q.O));
        // "nearest == Object" (erl:263) <=> Object is hit and nothing beats its (t, order)
        double a = q.D.x * q.D.x + q.D.y * q.D.y + q.D.z * q.D.z;
        double t;
        if (object_exact(sc, p.hit_obj, q.O, q.D, a, t)) {
            q.best.t = t; q.best.order = p.hit_order; q.best.obj = p.hit_obj;
            q.seed_obj = p.hit_obj;
            q.any = true;
        } else {
            q.need = false;          // the target itself is missed: shadow factor 0
        }
    }
}

// hit normal by object kind (erl:388-390, 476, 448-451)
__device__ __forceinline__ d3 hit_normal(const DevScene &sc, int obj, d3 P)
{
    int i = obj_index(obj);
    switch (obj_type(obj)) {
    case OBJ_SPHERE: {
        double4 s = ld_sphere(sc.sph_exact + i);
        return vnormalize(vsub(P, mk(s.x, s.y, s.z)));
    }
    case OBJ_PLANE:
        return mk(sc.planes[4 * i], sc.planes[4 * i + 1], sc.planes[4 * i + 2]);
    default: {
        const double *tr = sc.tris + 9 * i;
        return vnormalize(vcross(mk(tr[0], tr[1], tr[2]), mk(tr[3], tr[4], tr[5])));
    }
    }
}

// math:pow(Base, Power) of specular_term (erl:293).  Base is max(0, .) <= 1 + rounding.  Specular
// powers are small whole numbers in every scene of the reference (618-665) and the benchmarks; for
// those, square-and-multiply (<= 11 DMULs, each correctly rounded: a few ulp from the exact power,
// like CUDA's pow, which is 2 ulp from glibc's) replaces the ~150-instruction general routine.
__device__ __forceinline__ double spec_pow(double base, double power)
{
    if (power >= 0.0 && power <= 64.0 && power == floor(power)) {
        unsigned int n = (unsigned int)power;
        double r = 1.0, b = base;
        while (n) {
            if (n & 1u) r *= b;
            b *= b;
            n >>= 1;
        }
        return r;
    }
    return pow(base, power);
}

// LightColour (*) (Diffuse + Specular) of one unshadowed light (erl:225-247, 272-297);
// D is the direction of the ray that hit.
__device__ __forceinline__ d3 light_term(const double *l, const double *mat, d3 P, d3 N, d3 D)
{
    d3 lpos = mk(l[3], l[4], l[5]);
    d3 ldir = vnormalize(vsub(lpos, P));
    // diffuse_term erl:272-279
    d3 diffuse = vscale(mk(mat[0], mat[1], mat[2]), max0(vdot(N, ldir)));
    // specular_term erl:285-297
    double base = max0(vdot(vnormalize(vadd(ldir, vneg(D))), N));
    d3 specular = vscale(mk(l[6], l[7], l[8]), mat[4] * spec_pow(base, mat[3]));
    d3 contribution = vadd(diffuse, specular);                       // erl:225-238
    return vscale(vcmul(mk(l[0], l[1], l[2]), contribution), 1.0);   // erl:243-247, shadow = 1
}

// Consumes the resolved query: shading of erl:209-252 in forward (weight-carrying) form.
__device__ __forceinline__ void pix_consume(Pix &p, const DevScene &sc, const FrameParams &fp, const Query &q)
{
    if (!p.alive) return;
    p.rays++;
    const int L = sc.n_lights;
    if (p.phase == 0) {
        if (q.best.obj < 0) { p.alive = false; return; }     // BACKGROUND_COLOUR erl:202
        p.hit_obj = q.best.obj;
        p.hit_order = q.best.order;
        p.P = vadd(p.O, vscale(p.D, q.best.t));               // erl:384-387 / 443-447 / 471-475
        p.N = hit_normal(sc, p.hit_obj, p.P);
        p.S = mk(0.0, 0.0, 0.0);
        if (L == 0) { p.alive = false; return; }
        p.phase = 1;
        return;
    }
    // a shadow query came back
    const double *mat = material_ptr(sc, p.hit_obj);
    bool lit = q.need && q.best.obj == p.hit_obj;
    if (lit) {
        d3 term = light_term(sc.lights + 9 * (p.phase - 1), mat, p.P, p.N, p.D);
        p.S = vadd(p.S, term);
    }
    p.phase++;
    if (p.phase > L) {
        // all lights folded: Final = sum_l (Reflection + local_l) = L*refl*child + S
        p.C = vadd(p.C, vscale(p.S, p.W));
        double refl = mat[5];
        p.bounce++;
        if (p.bounce >= fp.depth || refl == 0.0 || p.W == 0.0) { p.alive = false; return; }
        p.W = p.W * ((double)L * refl);
        d3 nd = vbounce(p.D, p.N);                                        // erl:219-221
        p.O = p.P;
        p.D = nd;
        p.phase = 0;
    }
}

// The one quantisation rule of every output format: colour C of element triple idx of `out`.
__device__ __forceinline__ void colour_store(void *out, int format, size_t idx, d3 C)
{
    if (format == 0) {
        // erl:678-680: min(trunc(C*255), 255); negative values clamp to 0 in the byte format
        unsigned char *o = (unsigned char *)out + idx;
        double c[3] = {C.x, C.y, C.z};
#pragma unroll
        for (int k = 0; k < 3; k++) {
            double v = trunc(c[k] * 255.0);
            v = v < 255.0 ? v : 255.0;
            v = v > 0.0 ? v : 0.0;
            o[k] = (unsigned char)(int)v;
        }
    } else if (format == 1) {
        float *o = (float *)out + idx;
        o[0] = (float)C.x; o[1] = (float)C.y; o[2] = (float)C.z;
    } else {
        double *o = (double *)out + idx;
        o[0] = C.x; o[1] = C.y; o[2] = C.z;
    }
}

__device__ __forceinline__ void pix_store(const Pix &p, const FrameParams &fp, int X, int local_y)
{
    colour_store(fp.out, fp.format, ((size_t)local_y * fp.width + X) * 3, p.C);
}

// pixel coordinates of this thread: 8x4 pixels per warp, 4x2 warps per 256-thread block
__device__ __forceinline__ void pixel_of_thread(const FrameParams &fp, int &X, int &local_y, int &Y, bool &inside)
{
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int lx = (warp & 3) * 8 + (lane & 7);
    int ly = (warp >> 2) * 4 + (lane >> 3);
    X = blockIdx.x * 32 + lx;
    local_y = blockIdx.y * 8 + ly;
    if (fp.n_parts > 1 && fp.band_rows > 0) {
        int j = local_y / fp.band_rows;
        Y = (fp.part + j * fp.n_parts) * fp.band_rows + (local_y - j * fp.band_rows);
    } else {
        Y = local_y;
    }
    inside = X < fp.width && local_y < fp.local_rows && Y < fp.height;
}

template <bool COUNT>
__device__ __forceinline__ void flush_counters(const FrameParams &fp, int rays, const Tally<COUNT> &tl)
{
    unsigned int r = __reduce_add_sync(0xffffffffu, (unsigned int)rays);
    if ((threadIdx.x & 31) == 0 && r) atomicAdd(fp.counters + CNT_RAYS, (unsigned long long)r);
    if constexpr (COUNT) {
        unsigned int a = __reduce_add_sync(0xffffffffu, tl.filter);
        unsigned int b = __reduce_add_sync(0xffffffffu, tl.box);
        unsigned int c = __reduce_add_sync(0xffffffffu, tl.exact_sph);
        unsigned int d = __reduce_add_sync(0xffffffffu, tl.exact_other);
        unsigned int e = __reduce_add_sync(0xffffffffu, tl.cell);
        if ((threadIdx.x & 31) == 0) {
            if (e) atomicAdd(fp.counters + CNT_CELL, (unsigned long long)e);
            if (a) atomicAdd(fp.counters + CNT_FILTER, (unsigned long long)a);
            if (b) atomicAdd(fp.counters + CNT_BOX, (unsigned long long)b);
            if (c) atomicAdd(fp.counters + CNT_EXACT_SPH, (unsigned long long)c);
            if (d) atomicAdd(fp.counters + CNT_EXACT_OTHER, (unsigned long long)d);
        }
#ifdef ERT_PROBE
        for (int k = 0; k < 8; k++) {
            unsigned int q = __reduce_add_sync(0xffffffffu, tl.p[k]);
            if ((threadIdx.x & 31) == 0 && q) atomicAdd(fp.counters + CNT_PROBE + k, (unsigned long long)q);
        }
#endif
    }
}

// resolve one query without block cooperation (EXACT and BVH strategies)
template <int ACCEL, bool COUNT, bool TRI>
__device__ __forceinline__ void resolve_free(const DevScene &sc, Query &q, Tally<COUNT> &tl)
{
    if (!q.need) return;
    // a shadow query that starts from its target skips re-testing the target
    int skip = q.seed_obj;
    scan_others<COUNT, TRI>(sc, q.O, q.D, q.best, skip, tl);
    if (q.any && q.best.obj != q.seed_obj) return;
    if constexpr (ACCEL == 1) {
        double a = q.D.x * q.D.x + q.D.y * q.D.y + q.D.z * q.D.z;
        scan_spheres_exact<COUNT>(sc, q.O, q.D, a, q.best, skip, q.any, q.seed_obj, tl);
    } else {
        FRay f;
        if (make_fray(sc, q.O, q.D, f, true)) scan_spheres_bvh<COUNT>(sc, q.O, q.D, f, q.best, skip, q.any, q.seed_obj, tl);
        else q.best = scan_spheres_instead(&sc, q.O, q.D, q.best, skip, q.any, q.seed_obj);
    }
}

// ------------------------------------------------------------------ kernels
template <int ACCEL, bool COUNT, bool TRI = false>
__global__ void __launch_bounds__(256)
render_free_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp)
{
    int X, ly, Y;
    bool inside;
    pixel_of_thread(fp, X, ly, Y, inside);
    Pix p;
    pix_init(p, sc, fp, X, Y, inside);
    Tally<COUNT> tl;
    while (__any_sync(0xffffffffu, p.alive)) {
        Query q;
        pix_prepare(p, sc, q);
        resolve_free<ACCEL, COUNT, TRI>(sc, q, tl);
        pix_consume(p, sc, fp, q);
    }
    if (inside) pix_store(p, fp, X, ly);
    flush_counters<COUNT>(fp, p.rays, tl);
}

// ---- ERT_ACCEL_LINEAR: block-synchronous passes over shared-memory sphere tiles ----------
// Tiles of the FP32 filter array are streamed global -> shared with 1-D bulk async copies
// (cp.async.bulk + mbarrier, the TMA unit) into a double buffer; every thread of the block
// scans the tile for its own current ray.
constexpr int kTileSpheres = 2048;                       // 32 KB per buffer

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <bool COUNT, bool TRI = false>
__global__ void __launch_bounds__(256)
render_tiled_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4 *tiles = reinterpret_cast<float4 *>(smem_raw);                 // 2 * kTileSpheres
    __shared__ __align__(8) uint64_t bars[2];

    int X, ly, Y;
    bool inside;
    pixel_of_thread(fp, X, ly, Y, inside);
    Pix p;
    pix_init(p, sc, fp, X, Y, inside);
    Tally<COUNT> tl;

    const int n = sc.n_spheres;
    const int n_tiles = (n + kTileSpheres - 1) / kTileSpheres;
    uint32_t phase_bits = 0;          // parity per buffer
    bool resident = false;            // single-tile scenes stay in buffer 0
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    while (__syncthreads_or(p.alive)) {
        Query q;
        pix_prepare(p, sc, q);
        bool active = q.need;
        int skip = q.seed_obj;
        FRay f;
        float cull = 0.f;
        if (active) {
            scan_others<COUNT, TRI>(sc, q.O, q.D, q.best, skip, tl);
            if (q.any && q.best.obj != q.seed_obj) active = false;
        }
        if (active) {
            make_fray(sc, q.O, q.D, f, false);          // out of range: every sphere passes the filter
            cull = cull_from(f, q.best);
        }
        if (n_tiles > 0 && !resident) {
            if (threadIdx.x == 0) {
                int cnt = min(kTileSpheres, n);
                mbar_expect_tx(&bars[0], cnt * 16u);
                bulk_g2s(tiles, sc.sph_filter, cnt * 16u, &bars[0]);
            }
        }
        for (int t = 0; t < n_tiles; t++) {
            int buf = t & 1;
            if (t + 1 < n_tiles) {
                __syncthreads();              // everyone is done with the other buffer
                if (threadIdx.x == 0) {
                    int cnt = min(kTileSpheres, n - (t + 1) * kTileSpheres);
                    mbar_expect_tx(&bars[buf ^ 1], cnt * 16u);
                    bulk_g2s(tiles + (buf ^ 1) * kTileSpheres, sc.sph_filter + (size_t)(t + 1) * kTileSpheres,
                             cnt * 16u, &bars[buf ^ 1]);
                }
            }
            if (!resident) {
                mbar_wait(&bars[buf], (phase_bits >> buf) & 1u);
                phase_bits ^= 1u << buf;
            }
            if (active) {
                const float4 *tile = tiles + buf * kTileSpheres;
                int cnt = min(kTileSpheres, n - t * kTileSpheres);
                int base = t * kTileSpheres;
#pragma unroll 4
                for (int k = 0; k < cnt; k++) {
                    float4 fs = tile[k];
                    float b, v;
                    TALLY(filter);
                    if (filter_stage1(f, fs, b, v)) {
                        if (filter_stage2(f, fs, b, v, cull)) {
                            int sph = base + k;
                            int code = obj_code(OBJ_SPHERE, sph);
                            if (code != skip) {
                                double tt;
                                TALLY(exact_sph);
                                if (sphere_exact(q.O, q.D, f.a, ld_sphere(sc.sph_exact + sph), tt)) {
                                    int ord = sc.sph_order[sph];
                                    if (better(tt, ord, q.best)) {
                                        q.best.t = tt; q.best.order = ord; q.best.obj = code;
                                        cull = cull_from(f, q.best);
                                    }
                                }
                            }
                        }
                    }
                }
                if (q.any && q.best.obj != q.seed_obj) active = false;
            }
        }
        if (n_tiles == 1) resident = true;
        // (n_tiles > 1: buffer 0 is reloaded only after the barrier at the top of the next pass)
        pix_consume(p, sc, fp, q);
    }
    if (inside) pix_store(p, fp, X, ly);
    flush_counters<COUNT>(fp, p.rays, tl);
}

__device__ void trace_ray_wavefront(const DevScene &sc, d3 O, d3 D, Hit &best);   // ert_wavefront.cuh
__device__ void trace_ray_grid(const DevScene &sc, d3 O, d3 D, Hit &best);        // ert_wavefront.cuh

// ---- ray batch: nearest_object_intersecting_ray/2 for arbitrary rays (tests, BVH == scan) ----
template <int ACCEL, bool TRI = false>
__global__ void __launch_bounds__(256)
trace_rays_kernel(const __grid_constant__ DevScene sc, long long n_rays, const double *__restrict__ rays6,
                  int *__restrict__ order_out, double *__restrict__ t_out)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rays) return;
    Query q;
    q.O = mk(rays6[6 * i], rays6[6 * i + 1], rays6[6 * i + 2]);
    q.D = mk(rays6[6 * i + 3], rays6[6 * i + 4], rays6[6 * i + 5]);
    q.best.obj = -1; q.best.t = 0.0; q.best.order = 0x7fffffff;
    q.seed_obj = -1; q.any = false; q.need = true;
    Tally<false> tl;
    if constexpr (ACCEL == 2) {
        // same filter as the tiled kernel, spheres read straight from global memory
        scan_others<false, TRI>(sc, q.O, q.D, q.best, -1, tl);
        FRay f;
        make_fray(sc, q.O, q.D, f, false);              // out of range: every sphere passes the filter
        float cull = cull_from(f, q.best);
        for (int s = 0; s < sc.n_spheres; s++)
            try_sphere<false>(sc, f, q.O, q.D, __ldg(sc.sph_filter + s), s, -1, q.best, cull, tl);
    } else if constexpr (ACCEL == 4) {
        // the traversal of the wavefront kernels (ert_wavefront.cuh)
        scan_others<false, TRI>(sc, q.O, q.D, q.best, -1, tl);
        if (sc.n_spheres > 0) trace_ray_wavefront(sc, q.O, q.D, q.best);
    } else if constexpr (ACCEL == 5) {
        // the cell-grid walk of the wavefront's path kernels (ert_wavefront.cuh)
        scan_others<false, TRI>(sc, q.O, q.D, q.best, -1, tl);
        if (sc.n_spheres > 0) trace_ray_grid(sc, q.O, q.D, q.best);
    } else {
        resolve_free<ACCEL, false, TRI>(sc, q, tl);
    }
    order_out[i] = q.best.obj < 0 ? -1 : q.best.order;
    t_out[i] = q.best.obj < 0 ? 0.0 : q.best.t;
}

// ---- ray batch, one warp per ray (ERT_ACCEL_WARP): warp-wide nearest-hit reduction ----
// The scan of erl:300-346 split over the 32 lanes of a warp: lane k takes spheres k, k+32, ... through the FP32 filter
// and the literal test, planes and triangles go to lane 0, and the nearest object is the lexicographic minimum of
// (Distance, list position) over the lanes' results — erl:319's strict '>' over the list order — found with three
// __reduce_min_sync steps on the order-preserving integer image of the double.
__device__ __forceinline__ unsigned long long sortable_bits(double t)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(t);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
template <bool TRI = false>
__global__ void __launch_bounds__(256)
trace_rays_warp_kernel(const __grid_constant__ DevScene sc, long long n_rays, const double *__restrict__ rays6,
                       int *__restrict__ order_out, double *__restrict__ t_out)
{
    const int lane = threadIdx.x & 31;
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n_rays) return;                                   // the whole warp leaves together
    const d3 O = mk(rays6[6 * i], rays6[6 * i + 1], rays6[6 * i + 2]);
    const d3 D = mk(rays6[6 * i + 3], rays6[6 * i + 4], rays6[6 * i + 5]);
    Tally<false> tl;
    Hit best;
    best.obj = -1; best.t = 0.0; best.order = 0x7fffffff;
    if (lane == 0) scan_others<false, TRI>(sc, O, D, best, -1, tl);
    // every lane starts from lane 0's plane / triangle incumbent: it culls, and it is a candidate of the minimum
    best.t = __shfl_sync(0xffffffffu, best.t, 0);
    best.order = __shfl_sync(0xffffffffu, best.order, 0);
    best.obj = __shfl_sync(0xffffffffu, best.obj, 0);
    FRay f;
    make_fray(sc, O, D, f, false);                      // out of range: every sphere passes the filter
    float cull = cull_from(f, best);
    for (int s = lane; s < sc.n_spheres; s += 32)
        try_sphere<false>(sc, f, O, D, __ldg(sc.sph_filter + s), s, -1, best, cull, tl);
    // lexicographic minimum of (Distance, list position) over the lanes
    const bool have = best.obj >= 0;
    const unsigned long long key = have ? sortable_bits(best.t) : ~0ull;
    const unsigned int hi = (unsigned int)(key >> 32), lo = (unsigned int)key;
    const unsigned int min_hi = __reduce_min_sync(0xffffffffu, hi);
    const unsigned int min_lo = __reduce_min_sync(0xffffffffu, hi == min_hi ? lo : 0xffffffffu);
    const bool tied = have && hi == min_hi && lo == min_lo;
    const unsigned int min_ord = __reduce_min_sync(0xffffffffu, tied ? (unsigned int)best.order ^ 0x80000000u : 0xffffffffu);
    const unsigned int winners = __ballot_sync(0xffffffffu, tied && ((unsigned int)best.order ^ 0x80000000u) == min_ord);
    if (winners == 0u) {
        if (lane == 0) { order_out[i] = -1; t_out[i] = 0.0; }
    } else if (lane == __ffs((int)winners) - 1) {
        order_out[i] = best.order;
        t_out[i] = best.t;
    }
}

// ---- FP32 issue-peak probe: register-resident FFMA chains --------------------------------
__global__ void __launch_bounds__(256) fp32_peak_kernel(float *out, int iters, float seed)
{
    float a0 = seed + threadIdx.x, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
    float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.9999f, c = 0.0001f;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
            a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
        }
    }
    float s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 12345.678f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
constexpr int kPeakFfmaPerIter = 16 * 8;

// The same loop with three REGISTER operands per FFMA (multiplier and addend are run-time values):
// the form the intersection kernels actually issue (box planes, sphere centres and ray constants all
// live in registers).
__global__ void __launch_bounds__(256) fp32_peak_rrr_kernel(float *out, int iters, const float *__restrict__ in)
{
    float a0 = in[0] + threadIdx.x, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
    float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m0 = in[1], m1 = in[2], c0 = in[3], c1 = in[4];
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a0 = __fmaf_rn(a0, m0, c0); a1 = __fmaf_rn(a1, m1, c1); a2 = __fmaf_rn(a2, m0, c1); a3 = __fmaf_rn(a3, m1, c0);
            a4 = __fmaf_rn(a4, m0, c0); a5 = __fmaf_rn(a5, m1, c1); a6 = __fmaf_rn(a6, m0, c1); a7 = __fmaf_rn(a7, m1, c0);
        }
    }
    float s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 12345.678f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// FP64 counterpart (the literal tests of the small-scene kernels are DADD/DMUL/DFMA chains)
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, const double *__restrict__ in)
{
    double a0 = in[0] + threadIdx.x, a1 = a0 + 1., a2 = a0 + 2., a3 = a0 + 3.;
    double a4 = a0 + 4., a5 = a0 + 5., a6 = a0 + 6., a7 = a0 + 7.;
    const double m0 = in[1], m1 = in[2], c0 = in[3], c1 = in[4];
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a0 = __fma_rn(a0, m0, c0); a1 = __fma_rn(a1, m1, c1); a2 = __fma_rn(a2, m0, c1); a3 = __fma_rn(a3, m1, c0);
            a4 = __fma_rn(a4, m0, c0); a5 = __fma_rn(a5, m1, c1); a6 = __fma_rn(a6, m0, c1); a7 = __fma_rn(a7, m1, c0);
        }
    }
    double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void l2_flush_kernel(uint4 *buf, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) buf[i] = make_uint4(0, 0, 0, 0);
}

}  // namespace ert
