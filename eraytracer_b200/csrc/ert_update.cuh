// In-place scene update (ert_scene_update): the device side.  The host uploads the element tables that changed;
// these kernels recompute what create derived from them on the host, with the same per-element code
// (scene_math.h): the sphere filters in list and in leaf order, the pair-interleaved scan copy, the leaf-ordered
// triangle vertices, the scene constants, and the child boxes of both BVHs (a refit: same topology, new boxes).
#pragma once
#include "ert_device.cuh"
#include "ert_scan.cuh"
#include "scene_math.h"

namespace ert {

constexpr int kUpdThreads = 256;

// Reductions of one update, read back by the host.  Floats and doubles that are >= 0 order like their bit patterns;
// the signed bounds of the queue-ordering grid go through an order-preserving key (dkey).
struct UpdateScalars {
    unsigned int r_max, pad_c_max, eta_c_max, abs_max;   // float bits
    unsigned long long lo[3], hi[3];                     // dkey of min (c - |r|), max (c + |r|)
    unsigned long long tri_edge, tri_abs;                // double bits: largest edge / |coordinate| of a tree triangle
    double area_sph, area_tri;                           // sum of the child-box half areas after the refit
};

__host__ __device__ inline unsigned long long dkey(double x)
{
    unsigned long long b;
    memcpy(&b, &x, 8);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double dkey_value(unsigned long long k)
{
    unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    double x;
    memcpy(&x, &b, 8);
    return x;
}

__device__ inline unsigned long long warp_max_u64(unsigned long long v)
{
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}
__device__ inline unsigned long long warp_min_u64(unsigned long long v)
{
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w < v ? w : v;
    }
    return v;
}
__device__ inline double warp_sum(double v)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sphere k: its filter sphere in list order (sph_filter, sph_pairs) and the filter of leaf slot k (leaf_filter), and
// its share of the scene constants (flatten() in ert_api.cu).  The padding of sph_pairs never changes.
__global__ void __launch_bounds__(kUpdThreads) upd_spheres(const double4 *__restrict__ sph_exact,
                                                           const int *__restrict__ leaf_sph, int n, float4 *sph_filter,
                                                           float *sph_pairs, float4 *leaf_filter, UpdateScalars *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int r_max = 0, pad_max = 0, eta_max = 0, abs_max = 0;
    unsigned long long lo[3], hi[3];
    for (int a = 0; a < 3; a++) { lo[a] = ~0ull; hi[a] = 0; }
    if (k < n) {
        const double4 s = sph_exact[k];
        const double c[3] = {s.x, s.y, s.z};
        float f[4], pad_c, eta_c;
        make_filter_sphere(c, s.w, f, pad_c, eta_c);
        sph_filter[k] = make_float4(f[0], f[1], f[2], f[3]);
        float *o = &sph_pairs[(size_t)(k >> 1) * 8 + (k & 1)];
        o[0] = f[0]; o[2] = f[1]; o[4] = f[2]; o[6] = f[3];
        pad_max = __float_as_uint(pad_c);
        eta_max = __float_as_uint(eta_c);
        const double r = fabs(s.w);
        r_max = __float_as_uint(f_round_up(r));
        for (int a = 0; a < 3; a++) {
            abs_max = max(abs_max, __float_as_uint(f_round_up(fabs(c[a]) + r)));
            lo[a] = dkey(c[a] - r);
            hi[a] = dkey(c[a] + r);
        }
        const double4 l = sph_exact[leaf_sph[k]];
        const double lc[3] = {l.x, l.y, l.z};
        make_filter_sphere(lc, l.w, f, pad_c, eta_c);
        leaf_filter[k] = make_float4(f[0], f[1], f[2], f[3]);
    }
    r_max = __reduce_max_sync(0xffffffffu, r_max);
    pad_max = __reduce_max_sync(0xffffffffu, pad_max);
    eta_max = __reduce_max_sync(0xffffffffu, eta_max);
    abs_max = __reduce_max_sync(0xffffffffu, abs_max);
    for (int a = 0; a < 3; a++) { lo[a] = warp_min_u64(lo[a]); hi[a] = warp_max_u64(hi[a]); }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&out->r_max, r_max);
        atomicMax(&out->pad_c_max, pad_max);
        atomicMax(&out->eta_c_max, eta_max);
        atomicMax(&out->abs_max, abs_max);
        for (int a = 0; a < 3; a++) { atomicMin(&out->lo[a], lo[a]); atomicMax(&out->hi[a], hi[a]); }
    }
}

// Tree slot k of the triangle BVH: its vertices gathered again in leaf order, and the tree's constants of tri_walk.h.
__global__ void __launch_bounds__(kUpdThreads) upd_triangles(const double *__restrict__ tris,
                                                             const int *__restrict__ leaf_id, int n_tree,
                                                             double *tri_leaf, UpdateScalars *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long e_bits = 0, a_bits = 0;
    if (k < n_tree) {
        const double *src = tris + (size_t)leaf_id[k] * 9;
        double v[9];
        for (int j = 0; j < 9; j++) v[j] = src[j];
        for (int j = 0; j < 9; j++) tri_leaf[(size_t)k * 9 + j] = v[j];
        double e, m;
        triangle_extent(v, e, m);
        e_bits = (unsigned long long)__double_as_longlong(e);
        a_bits = (unsigned long long)__double_as_longlong(m);
    }
    e_bits = warp_max_u64(e_bits);
    a_bits = warp_max_u64(a_bits);
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&out->tri_edge, e_bits);
        atomicMax(&out->tri_abs, a_bits);
    }
}

struct SphereLeafBox {
    const double4 *sph;
    const int *leaf;
    __device__ void operator()(int slot, float lo[3], float hi[3]) const
    {
        const double4 s = sph[leaf[slot]];
        const double v[4] = {s.x, s.y, s.z, s.w};
        sphere_box(v, lo, hi);
    }
};
struct TriangleLeafBox {
    const double *leaf_tris;
    __device__ void operator()(int slot, float lo[3], float hi[3]) const { triangle_box(leaf_tris + (size_t)slot * 9, lo, hi); }
};

// One level of the refit (scene_math.h): the nodes order[0 .. count), whose inner children are refitted already.
// Adds the level's child-box half areas to *area.
template <typename LeafBox>
__global__ void __launch_bounds__(kUpdThreads) upd_refit_level(BvhNode *nodes, const int *__restrict__ order, int count,
                                                               LeafBox leaf_box, double *area)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    double a = 0;
    if (j < count) {
        const int i = order[j];
        refit_node(nodes, i, leaf_box);
        a = child_half_area(nodes[i], 0) + child_half_area(nodes[i], 1);
    }
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0 && a != 0) atomicAdd(area, a);
}

}  // namespace ert
