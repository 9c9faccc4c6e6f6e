// Host-side BVH builders over spheres and triangles (binned SAH, binary, two child boxes per node).
// The reference has no acceleration structure: nearest_object_intersecting_ray
// (raytracer.erl:300-346) is a linear scan.  The BVH only prunes; every sphere
// it lets through is still decided by the literal FP64 test, so the result is
// the linear scan's.
#pragma once
#include <cstdint>
#include <vector>

namespace ert {

// 64-byte node, children boxes stored in the parent so one node fetch decides both.
// child >= 0: inner node index.  child < 0: leaf, ~child = (first << 3) | (count - 1).
// An unused child has an inverted box (lo > hi) and can never be entered.
struct alignas(16) BvhNode {
    float c0x[2], c0y[2];   // child 0: lo.x hi.x lo.y hi.y
    float c1x[2], c1y[2];   // child 1
    float c0z[2], c1z[2];   // lo.z hi.z of child 0, then of child 1
    int32_t child[2];
    int32_t pad[2];
};
static_assert(sizeof(BvhNode) == 64, "BvhNode must be 64 bytes");

constexpr int kBvhLeafMax = 4;      // default spheres per leaf (<= 8 by the encoding)
constexpr float kBvhTravCost = 0.f; // default SAH traversal cost (see build_sphere_bvh)
constexpr int kSahMaxDepth = 30;    // below this depth splits fall back to the median (log2 n more levels)
constexpr int kBvhStack = 64;       // traversal stack entries (depth <= 30 + log2(n) + 1)

struct Bvh {
    std::vector<BvhNode> nodes;     // nodes[0] is the root (always an inner node)
    std::vector<int32_t> leaf_prim; // leaf-ordered sphere indices
    int depth = 0;
};

// boxes: n*6 floats {lo xyz, hi xyz}, centroids: n*3 floats.  The tree every other builder produces.
void build_box_bvh(const float *boxes, const float *centroids, int64_t n, Bvh &out, int leaf_max = kBvhLeafMax,
                   float trav_cost = 0.f);

// centers: n*3 doubles, radii: n doubles.  Boxes are [c-r, c+r] rounded outward to float.
// leaf_max: largest leaf (1..8).  trav_cost: cost of visiting one inner node in units of one
// ray/sphere filter test; a range of <= leaf_max spheres stays a leaf when the SAH says a
// split would not pay (trav_cost <= 0: always split down to leaf_max, the round-1 behaviour).
void build_sphere_bvh(const double *centers, const double *radii, int64_t n, Bvh &out, int leaf_max = kBvhLeafMax,
                      float trav_cost = 0.f);

// Scenes with at least this many triangles get a triangle BVH (DESIGN.md "Triangle BVH"); smaller ones keep the
// linear FP64 scan of every triangle.
constexpr int kTriBvhMin = 64;
// A triangle whose largest edge exceeds kTriAlwaysEdge times the median one, or with a coordinate beyond
// kTriAlwaysAbs, is left out of the tree and tested by every ray.
constexpr double kTriAlwaysEdge = 64.0;
constexpr double kTriAlwaysAbs = 1e30;

struct TriBvh {
    Bvh bvh;                          // leaf_prim: leaf slot -> triangle index
    std::vector<double> leaf_tris;    // [slot][9] v1 v2 v3 of the tree triangles in leaf order
    std::vector<int32_t> always;      // triangles outside the tree: every ray tests them
    double edge_max = 0;              // largest edge length (2-norm) of a tree triangle, rounded up
    double abs_max = 0;               // largest |coordinate| of a tree triangle
};

// tris: n*9 doubles {v1, v2, v3}.  Boxes are the vertices' bounds rounded outward to float; the walk widens them
// per ray by the margin of tri_walk.h.
void build_triangle_bvh(const double *tris, int64_t n, TriBvh &out);

}  // namespace ert
