// Binned-SAH builder for the sphere and triangle BVHs.  See bvh_build.h.
#include "bvh_build.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <future>
#include <thread>

#include "scene_math.h"

namespace ert {
namespace {

struct Box {
    float lo[3], hi[3];
    void reset()
    {
        for (int a = 0; a < 3; a++) { lo[a] = FLT_MAX; hi[a] = -FLT_MAX; }
    }
    void grow(const Box &b)
    {
        for (int a = 0; a < 3; a++) {
            lo[a] = std::min(lo[a], b.lo[a]);
            hi[a] = std::max(hi[a], b.hi[a]);
        }
    }
    float half_area() const
    {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (dx < 0 || dy < 0 || dz < 0) return 0.f;
        return dx * dy + dy * dz + dz * dx;
    }
};

// SAH bin of a centroid at x bins from the range's low end: trunc(x) clamped to [0, nb - 1].  Written with compares
// before the cast, so that a centroid past the float range (an Inf, or a NaN from Inf - Inf or Inf * 0) lands in an
// end bin instead of being cast to int, which C++ leaves undefined.
inline int sah_bin(float x, int nb)
{
    if (!(x >= 0.f)) return 0;
    if (x >= (float)(nb - 1)) return nb - 1;
    return (int)x;
}

struct TmpNode {
    Box box;
    int32_t left = -1, right = -1;   // tmp indices; -1 => leaf
    int32_t first = 0, count = 0;
    int32_t depth = 0;
};

struct Builder {
    std::vector<Box> prim;
    std::vector<float> cen;          // n*3
    std::vector<int32_t> idx;
    std::vector<TmpNode> tmp;
    std::atomic<int32_t> next{0};
    int max_depth_seen = 0;
    std::atomic<int> live_tasks{0};
    int max_tasks = 1;
    int leaf_max = kBvhLeafMax;
    float trav_cost = 0.f;

    int32_t alloc() { return next.fetch_add(1); }

    int32_t build(int32_t first, int32_t count, int depth)
    {
        int32_t me = alloc();
        TmpNode &n = tmp[me];
        n.first = first;
        n.count = count;
        n.depth = depth;
        n.box.reset();
        float clo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, chi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        for (int32_t i = first; i < first + count; i++) {
            int32_t p = idx[i];
            n.box.grow(prim[p]);
            for (int a = 0; a < 3; a++) {
                clo[a] = std::min(clo[a], cen[3 * (size_t)p + a]);
                chi[a] = std::max(chi[a], cen[3 * (size_t)p + a]);
            }
        }
        if (count <= 1 || (count <= leaf_max && trav_cost <= 0.f)) return me;

        int32_t mid = -1;
        if (depth < kSahMaxDepth) {
            // binned SAH over the three axes
            constexpr int NB = 16;
            float best_cost = FLT_MAX;
            int best_axis = -1, best_bin = -1;
            for (int a = 0; a < 3; a++) {
                float ext = chi[a] - clo[a];
                if (!(ext > 0.f)) continue;
                Box bb[NB];
                int32_t bc[NB];
                for (int b = 0; b < NB; b++) { bb[b].reset(); bc[b] = 0; }
                float scale = NB / ext;
                for (int32_t i = first; i < first + count; i++) {
                    int32_t p = idx[i];
                    const int b = sah_bin((cen[3 * (size_t)p + a] - clo[a]) * scale, NB);
                    bb[b].grow(prim[p]);
                    bc[b]++;
                }
                float right_area[NB];
                int32_t right_cnt[NB];
                Box acc;
                acc.reset();
                int32_t c = 0;
                for (int b = NB - 1; b > 0; b--) {
                    acc.grow(bb[b]);
                    c += bc[b];
                    right_area[b] = acc.half_area();
                    right_cnt[b] = c;
                }
                acc.reset();
                c = 0;
                for (int b = 0; b < NB - 1; b++) {
                    acc.grow(bb[b]);
                    c += bc[b];
                    if (c == 0 || right_cnt[b + 1] == 0) continue;
                    float cost = acc.half_area() * c + right_area[b + 1] * right_cnt[b + 1];
                    if (cost < best_cost) { best_cost = cost; best_axis = a; best_bin = b; }
                }
            }
            // SAH termination: a small range stays a leaf when splitting does not pay
            if (count <= leaf_max && best_axis >= 0) {
                float area = n.box.half_area();
                if (!(area > 0.f) || trav_cost + best_cost / area >= (float)count) return me;
            }
            if (best_axis >= 0) {
                float ext = chi[best_axis] - clo[best_axis];
                float scale = NB / ext;
                float lo = clo[best_axis];
                int a = best_axis, bbin = best_bin;
                auto it = std::partition(idx.begin() + first, idx.begin() + first + count,
                                         [&](int32_t p) {
                                             return sah_bin((cen[3 * (size_t)p + a] - lo) * scale, NB) <= bbin;
                                         });
                mid = (int32_t)(it - idx.begin());
            }
        }
        if ((mid <= first || mid >= first + count) && count <= leaf_max) return me;
        if (mid <= first || mid >= first + count) {
            // degenerate (coincident centroids) or too deep: split by index at the median
            // along the widest axis so depth stays logarithmic
            int a = 0;
            float e0 = chi[0] - clo[0], e1 = chi[1] - clo[1], e2 = chi[2] - clo[2];
            if (e1 > e0 && e1 >= e2) a = 1;
            else if (e2 > e0 && e2 > e1) a = 2;
            mid = first + count / 2;
            std::nth_element(idx.begin() + first, idx.begin() + mid, idx.begin() + first + count,
                             [&](int32_t p, int32_t q) {
                                 float cp = cen[3 * (size_t)p + a], cq = cen[3 * (size_t)q + a];
                                 return cp < cq || (cp == cq && p < q);
                             });
        }
        int32_t lcount = mid - first, rcount = count - lcount;
        int32_t l, r;
        if (count > 32768 && live_tasks.load() < max_tasks) {
            live_tasks.fetch_add(1);
            auto fut = std::async(std::launch::async,
                                  [this, first, lcount, depth] { return build(first, lcount, depth + 1); });
            r = build(mid, rcount, depth + 1);
            l = fut.get();
            live_tasks.fetch_sub(1);
        } else {
            l = build(first, lcount, depth + 1);
            r = build(mid, rcount, depth + 1);
        }
        tmp[me].left = l;
        tmp[me].right = r;
        return me;
    }
};

inline int32_t leaf_code(int32_t first, int32_t count) { return ~((first << 3) | (count - 1)); }

}  // namespace

void build_box_bvh(const float *boxes, const float *centroids, int64_t n, Bvh &out, int leaf_max, float trav_cost)
{
    leaf_max = std::min(std::max(leaf_max, 1), 8);
    out.nodes.clear();
    out.leaf_prim.clear();
    out.depth = 0;

    BvhNode empty{};
    for (int k = 0; k < 2; k++) {
        empty.c0x[k] = empty.c0y[k] = empty.c0z[k] = (k == 0) ? FLT_MAX : -FLT_MAX;
        empty.c1x[k] = empty.c1y[k] = empty.c1z[k] = (k == 0) ? FLT_MAX : -FLT_MAX;
    }
    empty.child[0] = empty.child[1] = leaf_code(0, 1);   // never entered: boxes are inverted
    if (n <= 0) {
        out.nodes.push_back(empty);
        return;
    }

    Builder b;
    b.prim.resize((size_t)n);
    b.cen.assign(centroids, centroids + (size_t)n * 3);
    b.idx.resize((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        for (int a = 0; a < 3; a++) {
            b.prim[(size_t)i].lo[a] = boxes[6 * i + a];
            b.prim[(size_t)i].hi[a] = boxes[6 * i + 3 + a];
        }
        b.idx[(size_t)i] = (int32_t)i;
    }
    b.leaf_max = leaf_max;
    b.trav_cost = trav_cost;
    b.tmp.resize((size_t)2 * n + 2);
    b.max_tasks = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    int32_t root = b.build(0, (int32_t)n, 0);

    auto set_child = [](BvhNode &nd, int k, const Box &bx, int32_t code) {
        float *x = k == 0 ? nd.c0x : nd.c1x;
        float *y = k == 0 ? nd.c0y : nd.c1y;
        float *z = k == 0 ? nd.c0z : nd.c1z;
        x[0] = bx.lo[0]; x[1] = bx.hi[0];
        y[0] = bx.lo[1]; y[1] = bx.hi[1];
        z[0] = bx.lo[2]; z[1] = bx.hi[2];
        nd.child[k] = code;
    };

    if (b.tmp[root].left < 0) {                 // the whole scene fits one leaf
        BvhNode nd = empty;
        set_child(nd, 0, b.tmp[root].box, leaf_code(0, (int32_t)n));
        out.nodes.push_back(nd);
    } else {
        // depth-first emission: a node, then its left subtree, then its right subtree
        struct Item { int32_t tmp, out; };
        std::vector<Item> stack;
        out.nodes.reserve((size_t)n);
        out.nodes.push_back(empty);
        stack.push_back({root, 0});
        while (!stack.empty()) {
            Item it = stack.back();
            stack.pop_back();
            const TmpNode &t = b.tmp[it.tmp];
            out.depth = std::max(out.depth, t.depth + 1);
            int32_t kids[2] = {t.left, t.right};
            int32_t inner_out[2] = {-1, -1};
            for (int k = 0; k < 2; k++) {
                const TmpNode &c = b.tmp[kids[k]];
                if (c.left < 0) {
                    set_child(out.nodes[it.out], k, c.box, leaf_code(c.first, c.count));
                } else {
                    inner_out[k] = (int32_t)out.nodes.size();
                    out.nodes.push_back(empty);
                    set_child(out.nodes[it.out], k, c.box, inner_out[k]);
                }
            }
            // push right first so the left subtree is emitted next (contiguous)
            if (inner_out[1] >= 0) stack.push_back({kids[1], inner_out[1]});
            if (inner_out[0] >= 0) stack.push_back({kids[0], inner_out[0]});
        }
    }
    out.leaf_prim = std::move(b.idx);
}

void build_sphere_bvh(const double *centers, const double *radii, int64_t n, Bvh &out, int leaf_max, float trav_cost)
{
    std::vector<float> boxes((size_t)std::max<int64_t>(n, 0) * 6), cen((size_t)std::max<int64_t>(n, 0) * 3);
    for (int64_t i = 0; i < n; i++) {
        for (int a = 0; a < 3; a++) {
            double c = centers[3 * i + a], r = std::fabs(radii[i]);
            boxes[6 * (size_t)i + a] = f_round_down(c - r);
            boxes[6 * (size_t)i + 3 + a] = f_round_up(c + r);
            cen[3 * (size_t)i + a] = (float)c;
        }
    }
    build_box_bvh(boxes.data(), cen.data(), n, out, leaf_max, trav_cost);
}

void build_triangle_bvh(const double *tris, int64_t n, TriBvh &out)
{
    out = TriBvh{};
    // per triangle: largest edge (2-norm, as the literal test forms the edges) and largest |coordinate|
    std::vector<double> edge((size_t)n), amax((size_t)n);
    for (int64_t i = 0; i < n; i++) triangle_extent(tris + 9 * i, edge[(size_t)i], amax[(size_t)i]);
    // A tree triangle's prune margin grows with the largest edge and coordinate of the tree (tri_walk.h), so a
    // triangle far larger than the typical one, or one whose box float cannot hold, is tested by every ray instead.
    double median = 0;
    if (n > 0) {
        std::vector<double> s = edge;
        std::nth_element(s.begin(), s.begin() + n / 2, s.end());
        median = s[(size_t)n / 2];
    }
    const double edge_cap = kTriAlwaysEdge * median;
    std::vector<int32_t> tree;
    tree.reserve((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        if (!(edge[(size_t)i] <= edge_cap) || !(amax[(size_t)i] <= kTriAlwaysAbs)) out.always.push_back((int32_t)i);
        else tree.push_back((int32_t)i);
    }
    const size_t m = tree.size();
    std::vector<float> boxes(m * 6), cen(m * 3);
    for (size_t j = 0; j < m; j++) {
        const double *v = tris + 9 * (size_t)tree[j];
        triangle_box(v, &boxes[6 * j], &boxes[6 * j + 3]);
        for (int a = 0; a < 3; a++) {
            double lo = std::min(v[a], std::min(v[3 + a], v[6 + a]));
            double hi = std::max(v[a], std::max(v[3 + a], v[6 + a]));
            cen[3 * j + a] = (float)(0.5 * lo + 0.5 * hi);
        }
        out.edge_max = std::max(out.edge_max, edge[(size_t)tree[j]]);
        out.abs_max = std::max(out.abs_max, amax[(size_t)tree[j]]);
    }
    // the sqrt and the sums above are correctly rounded: one part in 2^40 covers them
    out.edge_max *= 1.0 + 1.0 / 1099511627776.0;
    build_box_bvh(boxes.data(), cen.data(), (int64_t)m, out.bvh, kBvhLeafMax, 0.f);
    for (int32_t &p : out.bvh.leaf_prim) p = tree[(size_t)p];
    out.leaf_tris.resize(m * 9);
    for (size_t j = 0; j < m; j++)
        std::copy(tris + 9 * (size_t)out.bvh.leaf_prim[j], tris + 9 * (size_t)out.bvh.leaf_prim[j] + 9, &out.leaf_tris[9 * j]);
}

}  // namespace ert
