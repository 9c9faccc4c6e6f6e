// C ABI of the B200-native eraytracer hot path (include/ert_b200.h).
// Host side: scene flattening to SoA, BVH build, upload, launches, band placement.
// No CPU rendering path exists in this library.
#include "../../include/ert_b200.h"

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <new>
#include <string>
#include <vector>

#include "bvh_build.h"
#include "light_grid.h"
#include "cell_grid.h"
#include "host_threads.h"
#include "ert_device.cuh"
#include "ert_wavefront.cuh"
#include "ert_scan.cuh"
#include "ert_update.cuh"
#include "grid_build.cuh"
#include "scene_math.h"
#include "scene_tables.h"

// ERT_ACCEL_LINEAR: scenes up to this many spheres stay in the single-launch tiled kernel (one resident
// tile, no queue traffic); larger ones run the wavefront with the brute-force scan kernels.
constexpr int kWfScanFrom = 192;

// ERT_ACCEL_AUTO for a scene with a triangle BVH and few spheres (DESIGN.md "Triangle BVH": measured on m4)
constexpr int kTriAutoAccel = ERT_ACCEL_BVH_MEGAKERNEL;

#ifndef ERT_WF_REFILL_FROM
#define ERT_WF_REFILL_FROM 2        /* first bounce whose path rays use the refilling kernel */
#endif

using namespace ert;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what)
{
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    g_err = buf;
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? ERT_ERR_NO_DEVICE : ERT_ERR_CUDA;
}
#define CU(call)                                                  \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);     \
    } while (0)

// Host copy of the flattened scene (kept so ert_scene_clone needs no rebuild).
struct HostScene {
    ert_camera camera;
    std::vector<double> tab[T_COUNT];  // the element tables (scene_tables.h)
    std::vector<int> order[K_COUNT];   // the list positions of each kind's elements (lights, spheres: ascending)
    std::vector<float> sph_filter;     // [n][4]
    std::vector<float> sph_pairs;      // pair-interleaved, padded to whole scan tiles (ert_scan.cuh)
    std::vector<float> leaf_filter;    // [n][4]
    Bvh bvh;
    TriBvh tbvh;                       // triangle BVH (n_tris >= kTriBvhMin); leaf-ordered vertices, always-list
    bool has_tri_bvh = false;
    std::vector<LightGrid> lgrids;     // direction grids of the first lights (shadow queries)
    CellGrid cgrid;                    // uniform cell grid over the spheres (path rays)
    float r_max = 0, pad_c_max = 0, eta_c_max = 0, abs_max = 0;
    float grid_lo[3] = {0, 0, 0}, grid_scale[3] = {0, 0, 0};
    int n_lights = 0, n_planes = 0, n_tris = 0, n_spheres = 0;
    // ert_scene_update
    bool derived_stale = false;        // filters, pairs, leaf filters, tree nodes, leaf vertices: the device holds the
                                       // current ones (a clone downloads them)
    bool cgrid_dropped = false;        // an update dropped the cell grid / direction grids (ERT_UPDATE_REBUILD_GRIDS
    bool lgrids_dropped = false;       // builds them again)
    bool cgrid_dev = false;            // the cell grid / direction grid g was built on the device: the host mirror keeps
    bool lgrid_dev[kMaxLightGrids] = {};   // its geometry only (a clone builds it again on its own device)
    double sph_lo[3] = {0, 0, 0}, sph_hi[3] = {0, 0, 0};   // min (c - |r|), max (c + |r|): the cell grid's bounds
    double sph_build_area = 0, tri_build_area = 0;   // total child-box half area at the trees' last build (0: not yet taken)
};

// Node indices of a tree by depth, on the device (scene_math.h refit_levels), made on the first update.
struct RefitPlan {
    int *order = nullptr;
    std::vector<int32_t> off;
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;                // shadow + shading of bounce b, while `stream` traces bounce b+1
    std::vector<cudaEvent_t> ev_path, ev_shade;    // per bounce: hits of the bounce emitted / colours of the bounce folded
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    void *fb = nullptr;
    size_t fb_cap = 0;
    // wavefront queues (ERT_ACCEL_BVH), allocated on first use
    void *wf_mem = nullptr;
    size_t wf_cap = 0;
    void *scan_mem = nullptr;                      // partial results of the brute-force scan (ert_scan.cuh)
    size_t scan_cap = 0;
    unsigned int *wf_ctr = nullptr;
    int wf_ctr_depth = 0;
    unsigned int *wf_ctr_host = nullptr;           // pinned, for the early-out check of deep recursions
    unsigned int *wf_ctr_all_host = nullptr;       // pinned, the counters of the first ERT_MAX_BOUNCE_STATS levels
    int wf_levels = 0;                             // levels copied there by the last wavefront frame
    std::vector<cudaEvent_t> ticks;                // ERT_FLAG_TIME_KERNELS: one event before/after every launch
    std::vector<int> tick_class;                   // class of the launch between ticks[i] and ticks[i+1]
    unsigned long long *counters_dev = nullptr;
    unsigned long long *counters_host = nullptr;   // pinned
    ert_render_params params{};
    bool has_frame = false;
    bool busy = false;
    int local_rows = 0;
    ert_stats stats{};
    int pending_error = ERT_OK;
    std::string pending_msg;
};

}  // namespace

struct ert_scene {
    int device = 0;
    int wf_grid[7] = {0, 0, 0, 0, 0, 0, 0};   // persistent grid sizes: path(first), path, shadow, shade, cell-grid path(first), path, shadow+shade
    int wf_grid_scan = 0;              // brute-force scan kernels (2 blocks per SM)
    int wf_grid_fin = 0;               // wf_finalize: a streaming pass, every resident slot filled
    HostScene host;
    DevScene dev{};
    const double *tab_dev[T_COUNT] = {};        // host.tab on the device, where the DevScene fields point
    std::vector<void *> allocs;
    // the grids' arrays, whether uploaded from the host builders or built on the device (grid_build.cuh); each
    // direction grid owns its own, so an update rebuilds only the stale ones
    CellGridDevOut cg_buf;
    std::vector<LightGridDevOut> lg_buf;
    DevBuf lg_desc;                             // the LightGridDev array
    GridScratch grid_tmp;
    uint64_t uploaded = 0;                      // bytes upload() has copied to the device
    Slot slots[ERT_MAX_SLOTS];
    std::mutex mu;
    // ert_scene_update
    bool broken = false;                        // a CUDA call failed during an update: renders refuse until one succeeds
    unsigned char *staging = nullptr;           // pinned: the new element tables, then their uploads
    size_t staging_cap = 0;
    UpdateScalars *upd_dev = nullptr, *upd_host = nullptr;
    cudaEvent_t upd_ev[2] = {nullptr, nullptr};
    RefitPlan plan_sph, plan_tri;
};

namespace {

float f_up(double x) { return f_round_up(x); }

// the uniform grid that orders the wavefront queues, from the bounds of every [c - |r|, c + |r|]
void set_sort_grid(HostScene &h, const double lo[3], const double hi[3])
{
    for (int a = 0; a < 3; a++) {
        double ext = hi[a] - lo[a];
        h.grid_lo[a] = (float)lo[a];
        h.grid_scale[a] = ext > 0 ? (float)((double)(1 << kSortBits) / ext) : 0.f;
        if (!std::isfinite(h.grid_scale[a]) || !std::isfinite(h.grid_lo[a])) { h.grid_lo[a] = 0; h.grid_scale[a] = 0; }
    }
}

// direction-grid resolution (ERT_LIGHT_GRID_RES, 0 turns them off) and the number of lights that get one
int light_grid_res()
{
    int res = kLightGridRes;
    if (const char *e = getenv("ERT_LIGHT_GRID_RES")) res = atoi(e);
    return std::min(std::max(res, 0), 1024);
}
int light_grid_target(const HostScene &h, int res)
{
    return (res > 0 && h.n_spheres >= kLightGridMinSpheres) ? std::min(h.n_lights, kMaxLightGrids) : 0;
}
// ERT_CELL_GRID=0 turns the cell grid off, ERT_CELL_GRID_DENSITY = cells per sphere
bool cell_grid_wanted(double &density)
{
    density = kCellGridDensity;
    if (const char *e = getenv("ERT_CELL_GRID_DENSITY")) density = atof(e);
    const char *off = getenv("ERT_CELL_GRID");
    return !(off && atoi(off) == 0);
}

int flatten(const ert_scene_desc *d, HostScene &h)
{
    SourceOrder src;
    std::string err = check_create(d, src, h.order);
    if (!err.empty()) return fail(ERT_ERR_BADARG, err);
    double *tab[T_COUNT];
    for (int t = 0; t < T_COUNT; t++) {
        h.tab[t].resize(h.order[kTables[t].kind].size() * kTables[t].per);
        tab[t] = h.tab[t].data();
    }
    if (!(err = pack_tables(*d, src, tab)).empty()) return fail(ERT_ERR_BADARG, err);
    h.camera = d->camera;
    h.n_lights = (int)d->n_lights; h.n_planes = (int)d->n_planes;
    h.n_tris = (int)d->n_triangles; h.n_spheres = (int)d->n_spheres;
    h.sph_filter.resize((size_t)h.n_spheres * 4);
    std::vector<double> centers((size_t)h.n_spheres * 3), radii((size_t)h.n_spheres);
    for (int64_t k = 0; k < h.n_spheres; k++) {
        const double *c = &h.tab[T_SPH_EXACT][(size_t)k * 4], r = c[3];
        float pad_c, eta_c;
        make_filter_sphere(c, r, &h.sph_filter[(size_t)k * 4], pad_c, eta_c);
        h.pad_c_max = std::max(h.pad_c_max, pad_c);
        h.eta_c_max = std::max(h.eta_c_max, eta_c);
        h.r_max = std::max(h.r_max, f_up(std::fabs(r)));
        for (int a = 0; a < 3; a++) {
            centers[(size_t)k * 3 + a] = c[a];
            h.abs_max = std::max(h.abs_max, f_up(std::fabs(c[a]) + std::fabs(r)));
        }
        radii[(size_t)k] = r;
    }
    {
        // the same filter spheres pair-interleaved for the packed brute-force scan; the padding never passes
        // stage 1 (R = -3e38)
        const size_t n_tiles = ((size_t)h.n_spheres + kScanTile - 1) / kScanTile;
        h.sph_pairs.assign(n_tiles * kScanTile * 4, 0.f);
        for (size_t k = 0; k < n_tiles * kScanTile; k++) {
            float *o = &h.sph_pairs[(k >> 1) * 8 + (k & 1)];
            if (k < (size_t)h.n_spheres) {
                const float *f = &h.sph_filter[k * 4];
                o[0] = f[0]; o[2] = f[1]; o[4] = f[2]; o[6] = f[3];
            } else {
                o[0] = o[2] = o[4] = 0.f; o[6] = -3.0e38f;
            }
        }
    }
    // The builders (BVH, cell grid, one direction grid per light) are independent and run side by side; an
    // exception in any of them (std::bad_alloc, std::system_error) comes back through join() below.
    WorkerGroup builders;
    {
        builders.spawn([&h, &centers, &radii] {
            build_sphere_bvh(centers.data(), radii.data(), h.n_spheres, h.bvh, kBvhLeafMax, kBvhTravCost);
        });
    }
    h.has_tri_bvh = h.n_tris >= kTriBvhMin;
    if (h.has_tri_bvh) builders.spawn([&h] { build_triangle_bvh(h.tab[T_TRIS].data(), h.n_tris, h.tbvh); });
    if (h.n_spheres > 0) {
        double lo[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, hi[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
        for (int64_t k = 0; k < h.n_spheres; k++)
            for (int a = 0; a < 3; a++) {
                lo[a] = std::min(lo[a], centers[(size_t)k * 3 + a] - std::fabs(radii[(size_t)k]));
                hi[a] = std::max(hi[a], centers[(size_t)k * 3 + a] + std::fabs(radii[(size_t)k]));
            }
        set_sort_grid(h, lo, hi);
        for (int a = 0; a < 3; a++) { h.sph_lo[a] = lo[a]; h.sph_hi[a] = hi[a]; }
    }
    {
        // cell grid for the path rays
        double density;
        if (cell_grid_wanted(density))
            builders.spawn([&h, &centers, &radii, density] {
                build_cell_grid(centers.data(), radii.data(), h.sph_filter.data(), h.n_spheres, h.abs_max, density, h.cgrid);
            });
    }
    std::vector<char> lg_built;
    {
        // direction grids for shadow rays: worth their memory once a walk through the BVH costs more
        // than a handful of candidate tests
        const int res = light_grid_res();
        const int n_grids = light_grid_target(h, res);
        h.lgrids.resize((size_t)n_grids);
        lg_built.assign((size_t)n_grids, 0);
        for (int g = 0; g < n_grids; g++)
            builders.spawn([&h, &centers, &radii, &lg_built, g, res] {
                lg_built[(size_t)g] = build_light_grid(centers.data(), radii.data(), h.sph_filter.data(), h.n_spheres,
                                                       &h.tab[T_LIGHTS][(size_t)g * 9 + 3], res, h.lgrids[(size_t)g]) ? 1 : 0;
            });
    }
    builders.join();
    {
        // the device code gives the first lg_count lights a grid: a light whose grid went over its entry budget
        // ends the run of grids
        size_t keep = 0;
        while (keep < lg_built.size() && lg_built[keep]) keep++;
        h.lgrids.resize(keep);
    }
    // the traversal stacks hold kBvhStack entries; the builder's depth bound (SAH levels + median levels) keeps
    // trees far below that, and a tree that is not must not be walked with a stack that silently drops subtrees
    if (h.bvh.depth >= kBvhStack)
        return fail(ERT_ERR_BADARG, "sphere BVH is deeper than the traversal stack");
    if (h.has_tri_bvh && h.tbvh.bvh.depth >= kBvhStack)
        return fail(ERT_ERR_BADARG, "triangle BVH is deeper than the traversal stack");
    h.leaf_filter.resize((size_t)h.n_spheres * 4);
    for (int64_t k = 0; k < h.n_spheres; k++)
        memcpy(&h.leaf_filter[(size_t)k * 4], &h.sph_filter[(size_t)h.bvh.leaf_prim[(size_t)k] * 4], 16);
    return ERT_OK;
}

// owner: the list the allocation is freed from (the scene's tables by default)
template <typename T>
int upload(ert_scene *s, const std::vector<T> &v, const T **out, std::vector<void *> *owner = nullptr)
{
    *out = nullptr;
    size_t bytes = std::max<size_t>(v.size() * sizeof(T), 16);
    void *p = nullptr;
    CU(cudaMalloc(&p, bytes));
    (owner ? owner : &s->allocs)->push_back(p);
    if (!v.empty()) CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    s->uploaded += v.size() * sizeof(T);
    *out = (const T *)p;
    return ERT_OK;
}

// v into the device array b (grown if needed)
template <typename T>
int upload_buf(ert_scene *s, DevBuf &b, const std::vector<T> &v)
{
    CU(b.reserve(v.size() * sizeof(T)));
    if (!v.empty()) CU(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    s->uploaded += v.size() * sizeof(T);
    return ERT_OK;
}

// The LightGridDev array of the first `count` direction grids (s->lg_buf) to the device, on stream st; adds its
// bytes to *h2d.
int write_light_desc(ert_scene *s, int count, cudaStream_t st, uint64_t *h2d)
{
    std::vector<LightGridDev> lg((size_t)count);
    for (int g = 0; g < count; g++) {
        const LightGridDevOut &o = s->lg_buf[(size_t)g];
        lg[(size_t)g].cell_off = o.cell_off.as<const unsigned int>();
        lg[(size_t)g].cand = o.cand.as<const LightGridCand>();
        lg[(size_t)g].head = o.head.as<const LightGridCand>();
        lg[(size_t)g].always = o.always.as<const int>();
        lg[(size_t)g].n_always = o.n_always;
        lg[(size_t)g].res = o.res;
    }
    const size_t bytes = lg.size() * sizeof(LightGridDev);
    CU(s->lg_desc.reserve(bytes));
    if (bytes) CU(cudaMemcpyAsync(s->lg_desc.p, lg.data(), bytes, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));                  // lg is pageable and goes out of scope
    s->uploaded += bytes;
    if (h2d) *h2d += bytes;
    s->dev.lgrids = s->lg_desc.as<const LightGridDev>();
    s->dev.lg_count = count;
    return ERT_OK;
}

// the direction grids of h.lgrids (replacing any the device had)
int upload_light_grids(ert_scene *s)
{
    HostScene &h = s->host;
    int rc;
    if (s->lg_buf.size() < h.lgrids.size()) s->lg_buf.resize(h.lgrids.size());
    std::vector<LightGridCand> cand, head;
    for (size_t g = 0; g < h.lgrids.size(); g++) {
        const LightGrid &G = h.lgrids[g];
        LightGridDevOut &o = s->lg_buf[g];
        pack_light_grid(G, cand, head);
        if ((rc = upload_buf(s, o.cell_off, G.cell_off)) != ERT_OK) return rc;
        if ((rc = upload_buf(s, o.cand, cand)) != ERT_OK) return rc;
        if ((rc = upload_buf(s, o.head, head)) != ERT_OK) return rc;
        if ((rc = upload_buf(s, o.always, G.always)) != ERT_OK) return rc;
        o.ok = true;
        o.res = G.res;
        o.n_always = (int)G.always.size();
        o.n_entries = G.entries.size();
    }
    return write_light_desc(s, (int)h.lgrids.size(), 0, nullptr);
}

// the kernels' view of s->cg_buf
void set_cell_desc(ert_scene *s)
{
    DevScene &d = s->dev;
    const CellGridDevOut &G = s->cg_buf;
    d.cg.blocks = G.blocks.as<const uint4>(); d.cg.over_filter = G.over_filter.as<const float4>();
    d.cg.over_sph = G.over_sph.as<const int>(); d.cg.big = G.big.as<const int>();
    d.cg.n_big = G.n_big; d.cg.enabled = G.enabled ? 1 : 0;
    d.cg.rx = G.geo.res[0]; d.cg.ry = G.geo.res[1]; d.cg.rz = G.geo.res[2];
    for (int a = 0; a < 3; a++) { d.cg.lo[a] = G.geo.lo[a]; d.cg.hi[a] = G.geo.hi[a]; }
    d.cg.cs = G.geo.cs; d.cg.eps = G.geo.eps;
}

// the cell grid of h.cgrid (replacing any the device had)
int upload_cell_grid(ert_scene *s)
{
    const CellGrid &G = s->host.cgrid;
    CellGridDevOut &o = s->cg_buf;
    int rc;
    if ((rc = upload_buf(s, o.blocks, G.blocks)) != ERT_OK) return rc;
    if ((rc = upload_buf(s, o.over_filter, G.over_filter)) != ERT_OK) return rc;
    if ((rc = upload_buf(s, o.over_sph, G.over_sph)) != ERT_OK) return rc;
    if ((rc = upload_buf(s, o.big, G.big)) != ERT_OK) return rc;
    o.enabled = G.enabled;
    o.n_big = (int)G.big.size();
    o.n_over = G.over_sph.size();
    o.geo = CellGridGeom();
    for (int a = 0; a < 3; a++) { o.geo.res[a] = G.res[a]; o.geo.lo[a] = G.lo[a]; o.geo.hi[a] = G.hi[a]; }
    o.geo.cs = G.cs; o.geo.inv_cs = G.inv_cs; o.geo.eps = G.eps;
    set_cell_desc(s);
    return ERT_OK;
}

// the scene constants of h in the kernels' parameter block
void set_constants(ert_scene *s)
{
    HostScene &h = s->host;
    DevScene &d = s->dev;
    for (int a = 0; a < 3; a++) { d.grid_lo[a] = h.grid_lo[a]; d.grid_scale[a] = h.grid_scale[a]; }
    d.r_max = h.r_max; d.pad_c_max = h.pad_c_max; d.eta_c_max = h.eta_c_max; d.abs_max = h.abs_max;
    if (h.has_tri_bvh) { d.tri_edge_max = h.tbvh.edge_max; d.tri_abs_max = h.tbvh.abs_max; }
}

// every table, tree and grid of s->host to the device (the scene's streams are untouched)
int upload_tables(ert_scene *s)
{
    HostScene &h = s->host;
    DevScene &d = s->dev;
    int rc;
    CU(cudaSetDevice(s->device));
    d.n_lights = h.n_lights; d.n_planes = h.n_planes; d.n_tris = h.n_tris; d.n_spheres = h.n_spheres;
#define UP(vec, field, T)                                                         \
    do {                                                                          \
        const T *p__;                                                             \
        if ((rc = upload<T>(s, vec, &p__)) != ERT_OK) return rc;                  \
        d.field = reinterpret_cast<decltype(d.field)>(p__);                       \
    } while (0)
    for (int t = 0; t < T_COUNT; t++)
        if ((rc = upload(s, h.tab[t], &s->tab_dev[t])) != ERT_OK) return rc;
    const double *const *tp = s->tab_dev;
    d.lights = tp[T_LIGHTS]; d.planes = tp[T_PLANES]; d.plane_mat = tp[T_PLANE_MAT]; d.tris = tp[T_TRIS];
    d.tri_mat = tp[T_TRI_MAT]; d.sph_mat = tp[T_SPH_MAT]; d.sph_refl = tp[T_SPH_REFL];
    d.sph_exact = reinterpret_cast<const double4 *>(tp[T_SPH_EXACT]);
    UP(h.order[K_PLANES], plane_order, int);
    UP(h.order[K_TRIS], tri_order, int);
    UP(h.order[K_SPHERES], sph_order, int);
    UP(h.sph_filter, sph_filter, float);
    UP(h.sph_pairs, sph_pairs, float);
    UP(h.leaf_filter, leaf_filter, float);
    UP(h.bvh.leaf_prim, leaf_sph, int);
    UP(h.bvh.nodes, nodes, BvhNode);
    if (h.has_tri_bvh) {
        UP(h.tbvh.bvh.nodes, tri_nodes, BvhNode);
        UP(h.tbvh.leaf_tris, tri_leaf, double);
        UP(h.tbvh.bvh.leaf_prim, tri_leaf_id, int);
        UP(h.tbvh.always, tri_always, int);
        d.n_tri_tree = (int)h.tbvh.bvh.leaf_prim.size();
        d.n_tri_always = (int)h.tbvh.always.size();
    }
#undef UP
    if ((rc = upload_light_grids(s)) != ERT_OK) return rc;
    if ((rc = upload_cell_grid(s)) != ERT_OK) return rc;
    d.n_nodes = (int)h.bvh.nodes.size();
    set_constants(s);
    return ERT_OK;
}

int upload_scene(ert_scene *s)
{
    int rc;
    if ((rc = upload_tables(s)) != ERT_OK) return rc;
    for (int i = 0; i < ERT_MAX_SLOTS; i++) {
        Slot &sl = s->slots[i];
        {
            // the path rays are the critical chain of a frame: their stream gets the higher priority, the shadow rays
            // and the shading of the previous bounce fill what the path kernels leave idle
            int prio_lo = 0, prio_hi = 0;
            CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            CU(cudaStreamCreateWithPriority(&sl.stream, cudaStreamNonBlocking, prio_hi));
            CU(cudaStreamCreateWithPriority(&sl.stream2, cudaStreamNonBlocking, prio_lo));
        }
        CU(cudaEventCreate(&sl.ev0));
        CU(cudaEventCreate(&sl.ev1));
        CU(cudaEventCreate(&sl.ev2));
        CU(cudaMalloc(&sl.counters_dev, kCounterSets * CNT_N * sizeof(unsigned long long)));
        CU(cudaMallocHost(&sl.counters_host, kCounterSets * CNT_N * sizeof(unsigned long long)));
    }
    // opt in to the 64 KB double buffer of the tiled kernel
    CU(cudaFuncSetAttribute(render_tiled_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            2 * kTileSpheres * 16));
    CU(cudaFuncSetAttribute(render_tiled_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            2 * kTileSpheres * 16));
    CU(cudaFuncSetAttribute(render_tiled_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            2 * kTileSpheres * 16));
    CU(cudaFuncSetAttribute(render_tiled_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            2 * kTileSpheres * 16));
    {
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, s->device));
        int nb = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_trace_path<true, false, true, false>, kWfThreads, 0));
        s->wf_grid[0] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_trace_path<false, false, true, false>, kWfThreads, 0));
        s->wf_grid[1] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_trace_path<true, false, true, true>, kWfThreads, 0));
        s->wf_grid[4] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_finalize, kWfThreads, 0));
        s->wf_grid_fin = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_trace_path_refill<false, true, true>, kWfThreads, 0));
        s->wf_grid[5] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_trace_shadow<false, true>, kWfThreads, 0));
        s->wf_grid[2] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_shade, kWfThreads, 0));
        s->wf_grid[3] = prop.multiProcessorCount * std::max(nb, 1);
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_shadow_shade<false>, kWfThreads, 0));
        s->wf_grid[6] = prop.multiProcessorCount * std::max(nb, 1);
        // The walks live on L1 (tree nodes + the local-memory stacks).  Ask for exactly the shared memory
        // the resident blocks need, so that the rest of the 256 KB array serves as L1 (measured on C4:
        // 23.5 -> 23.1 ms against the driver's default split; too small a carve-out halves the occupancy).
        auto carve = [&](const void *fn, int blocks_per_sm) -> int {
            cudaFuncAttributes fa;
            CU(cudaFuncGetAttributes(&fa, fn));
            size_t need = (size_t)blocks_per_sm * (fa.sharedSizeBytes + 1024);      // 1 KB per block is reserved
            int pct = (int)((need * 100 + prop.sharedMemPerMultiprocessor - 1) / prop.sharedMemPerMultiprocessor) + 1;
            CU(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, std::min(pct, 100)));
            return ERT_OK;
        };
        if ((rc = carve((const void *)wf_trace_path<true, false, true, false>, s->wf_grid[0] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path<false, false, true, false>, s->wf_grid[1] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path<false, false, false, false>, s->wf_grid[1] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path_refill<false, false, true>, s->wf_grid[1] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path<true, false, true, true>, s->wf_grid[4] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path<false, false, true, true>, s->wf_grid[5] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path<false, false, false, true>, s->wf_grid[5] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_path_refill<false, true, true>, s->wf_grid[5] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_shadow<false, true>, s->wf_grid[2] / prop.multiProcessorCount)) != ERT_OK) return rc;
        if ((rc = carve((const void *)wf_trace_shadow<false, false>, s->wf_grid[2] / prop.multiProcessorCount)) != ERT_OK) return rc;
        CU(cudaFuncSetAttribute(wf_scan<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaFuncSetAttribute(wf_scan<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaFuncSetAttribute(wf_scan<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaFuncSetAttribute(wf_scan<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaFuncSetAttribute(wf_scan<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaFuncSetAttribute(wf_scan<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wf_scan<false, false, false>, kScanThreads, kScanSmem));
        int nb2 = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb2, wf_scan<true, false, false>, kScanThreads, kScanSmem));
        // Several short blocks per resident slot: the hardware hands a new block to an SM as soon as one retires, so
        // the SM stays full until the grid drains (with exactly one block per slot the warp schedulers let some
        // blocks run ahead and the launch ends with one or two warps per scheduler: 2.8 of 4 resident on average,
        // FMA pipe 75 % busy, profiles/r02_c4_scan_full.txt)
        int scan_waves = 8;
        if (const char *e = getenv("ERT_SCAN_WAVES")) scan_waves = std::min(std::max(atoi(e), 1), 64);
        s->wf_grid_scan = prop.multiProcessorCount * std::max(std::min(nb, nb2), 1) * scan_waves;
    }
    return ERT_OK;
}

void destroy(ert_scene *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    for (int i = 0; i < ERT_MAX_SLOTS; i++) {
        Slot &sl = s->slots[i];
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        if (sl.fb) cudaFree(sl.fb);
        if (sl.wf_mem) cudaFree(sl.wf_mem);
        if (sl.scan_mem) cudaFree(sl.scan_mem);
        if (sl.wf_ctr) cudaFree(sl.wf_ctr);
        if (sl.wf_ctr_host) cudaFreeHost(sl.wf_ctr_host);
        if (sl.wf_ctr_all_host) cudaFreeHost(sl.wf_ctr_all_host);
        for (cudaEvent_t e : sl.ticks) cudaEventDestroy(e);
        for (cudaEvent_t e : sl.ev_path) cudaEventDestroy(e);
        for (cudaEvent_t e : sl.ev_shade) cudaEventDestroy(e);
        if (sl.stream2) cudaStreamDestroy(sl.stream2);
        if (sl.counters_dev) cudaFree(sl.counters_dev);
        if (sl.counters_host) cudaFreeHost(sl.counters_host);
        if (sl.ev0) cudaEventDestroy(sl.ev0);
        if (sl.ev1) cudaEventDestroy(sl.ev1);
        if (sl.ev2) cudaEventDestroy(sl.ev2);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    for (void *p : s->allocs) cudaFree(p);
    s->cg_buf.release();
    for (LightGridDevOut &o : s->lg_buf) o.release();
    s->lg_desc.release();
    s->grid_tmp.release();
    if (s->plan_sph.order) cudaFree(s->plan_sph.order);
    if (s->plan_tri.order) cudaFree(s->plan_tri.order);
    if (s->upd_dev) cudaFree(s->upd_dev);
    if (s->upd_host) cudaFreeHost(s->upd_host);
    if (s->staging) cudaFreeHost(s->staging);
    for (cudaEvent_t e : s->upd_ev)
        if (e) cudaEventDestroy(e);
    delete s;
}

size_t bytes_per_channel(int format) { return format == ERT_FMT_RGB8 ? 1 : (format == ERT_FMT_F32 ? 4 : 8); }

// rows of this part and their count; band b -> part b % n_parts
int local_rows_of(const ert_render_params &p)
{
    if (p.n_parts <= 1 || p.band_rows <= 0) return p.height;
    int rows = 0;
    int n_bands = (p.height + p.band_rows - 1) / p.band_rows;
    for (int b = p.part; b < n_bands; b += p.n_parts) rows += std::min(p.band_rows, p.height - b * p.band_rows);
    return rows;
}

int check_params(const ert_render_params *p)
{
    if (!p) return fail(ERT_ERR_BADARG, "render params are NULL");
    if (p->width <= 0 || p->height <= 0) return fail(ERT_ERR_BADARG, "width and height must be > 0 (erl:89)");
    if (p->depth < 0) return fail(ERT_ERR_BADARG, "recursion depth must be >= 0");
    if (p->format < ERT_FMT_RGB8 || p->format > ERT_FMT_F64) return fail(ERT_ERR_BADARG, "unknown output format");
    if (p->accel < ERT_ACCEL_AUTO || p->accel > ERT_ACCEL_GRID) return fail(ERT_ERR_BADARG, "unknown accel");
    if (p->n_parts > 1 && p->band_rows > 0 && (p->part < 0 || p->part >= p->n_parts))
        return fail(ERT_ERR_BADARG, "part must be in [0, n_parts)");
    if (p->band_rows < 0) return fail(ERT_ERR_BADARG, "band_rows must be >= 0");
    return ERT_OK;
}

int pick_accel(const ert_scene *s, int requested)
{
    if (requested == ERT_ACCEL_GRID) return s->host.cgrid.enabled ? ERT_ACCEL_GRID : ERT_ACCEL_BVH;
    if (requested != ERT_ACCEL_AUTO) return requested;
    // a scene with a triangle BVH never goes to the linear triangle scan of ERT_ACCEL_EXACT (DESIGN.md "Triangle BVH")
    if (s->host.has_tri_bvh && s->host.n_spheres <= 192) return kTriAutoAccel;
    if (s->host.n_spheres <= 16) return ERT_ACCEL_EXACT;
    if (s->host.n_spheres <= 192) return ERT_ACCEL_LINEAR;
    return s->host.cgrid.enabled ? ERT_ACCEL_GRID : ERT_ACCEL_BVH;
}

// device -> host placement of the part's rows inside the full frame
int copy_part_to_host(ert_scene *s, Slot &sl, const ert_render_params &p, void *host_frame, size_t host_bytes,
                      uint64_t *bytes_out)
{
    size_t row_bytes = (size_t)p.width * 3 * bytes_per_channel(p.format);
    size_t need = row_bytes * (size_t)p.height;
    if (host_bytes < need) return fail(ERT_ERR_BADARG, "host frame buffer is smaller than width*height*3 elements");
    unsigned char *dst = (unsigned char *)host_frame;
    const unsigned char *src = (const unsigned char *)sl.fb;
    uint64_t total = 0;
    if (p.n_parts <= 1 || p.band_rows <= 0) {
        CU(cudaMemcpyAsync(dst, src, need, cudaMemcpyDeviceToHost, sl.stream));
        total = need;
    } else {
        int n_bands = (p.height + p.band_rows - 1) / p.band_rows;
        int full_bands_total = p.height / p.band_rows;           // bands with band_rows rows
        // own full bands: b = part, part + n_parts, ... < full_bands_total
        int own_full = full_bands_total > p.part ? (full_bands_total - p.part + p.n_parts - 1) / p.n_parts : 0;
        size_t band_bytes = row_bytes * (size_t)p.band_rows;
        if (own_full > 0) {
            CU(cudaMemcpy2DAsync(dst + (size_t)p.part * band_bytes, band_bytes * (size_t)p.n_parts, src, band_bytes,
                                 band_bytes, (size_t)own_full, cudaMemcpyDeviceToHost, sl.stream));
            total += band_bytes * (size_t)own_full;
        }
        // a partial last band, if this part owns it
        int last = n_bands - 1;
        if (n_bands > full_bands_total && last % p.n_parts == p.part) {
            size_t rows = (size_t)(p.height - last * p.band_rows);
            CU(cudaMemcpyAsync(dst + (size_t)last * band_bytes, src + (size_t)own_full * band_bytes, rows * row_bytes,
                               cudaMemcpyDeviceToHost, sl.stream));
            total += rows * row_bytes;
        }
    }
    if (bytes_out) *bytes_out = total;
    (void)s;
    return ERT_OK;
}

template <bool COUNT, bool TRI>
void launch_render(int accel, dim3 grid, cudaStream_t st, const DevScene &d, const FrameParams &fp)
{
    switch (accel) {
    case ERT_ACCEL_EXACT: render_free_kernel<1, COUNT><<<grid, 256, 0, st>>>(d, fp); break;    // the linear FP64 scan
    case ERT_ACCEL_LINEAR: render_tiled_kernel<COUNT, TRI><<<grid, 256, 2 * kTileSpheres * 16, st>>>(d, fp); break;
    default: render_free_kernel<3, COUNT, TRI><<<grid, 256, 0, st>>>(d, fp); break;   // BVH megakernel (also depth 0)
    }
}

template <bool TRI>
void launch_trace_rays(int accel, unsigned blocks, cudaStream_t st, const DevScene &d, long long n_rays, const double *rays,
                       int *ord, double *t)
{
    switch (accel) {
    case ERT_ACCEL_WARP: trace_rays_warp_kernel<TRI><<<(unsigned)((n_rays * 32 + 255) / 256), 256, 0, st>>>(d, n_rays, rays, ord, t); break;
    case ERT_ACCEL_EXACT: trace_rays_kernel<1><<<blocks, 256, 0, st>>>(d, n_rays, rays, ord, t); break;    // the linear FP64 scan
    case ERT_ACCEL_LINEAR: trace_rays_kernel<2, TRI><<<blocks, 256, 0, st>>>(d, n_rays, rays, ord, t); break;
    case ERT_ACCEL_BVH_MEGAKERNEL: trace_rays_kernel<3, TRI><<<blocks, 256, 0, st>>>(d, n_rays, rays, ord, t); break;
    case ERT_ACCEL_GRID: trace_rays_kernel<5, TRI><<<blocks, 256, 0, st>>>(d, n_rays, rays, ord, t); break;
    default: trace_rays_kernel<4, TRI><<<blocks, 256, 0, st>>>(d, n_rays, rays, ord, t); break;
    }
}

// ---- wavefront frame (ERT_ACCEL_BVH) ------------------------------------------------------
size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int wf_prepare(ert_scene *s, Slot &sl, const FrameParams &fp, WfBuf &wf, bool scan)
{
    int tiles_x = (fp.width + 7) / 8, tiles_y = (fp.local_rows + 3) / 4;
    size_t n_pad = (size_t)tiles_x * (size_t)tiles_y * 32;
    if (n_pad >= ((size_t)1 << 31)) return fail(ERT_ERR_BADARG, "frame part has more than 2^31 pixels");
    size_t L = (size_t)std::max(s->host.n_lights, 1);
    // layout: C[3] res_t[1] doubles | two path queues | hits, raw_hits records | res_hit[2] r_key ints |
    // lit bytes | sort histogram + block sums
    size_t off = 0;
    size_t o_dbl = off; off += align_up(n_pad * 4 * sizeof(double), 256);
    size_t o_path = off; off += align_up(n_pad * 2 * sizeof(PathRec), 256);
    size_t o_rec = off; off += align_up(n_pad * 2 * (sizeof(HitHead) + sizeof(HitTail)), 256);
    size_t o_int = off; off += align_up(n_pad * 3 * sizeof(int), 256);
    size_t o_lit = off; off += align_up(n_pad * L, 256);
    size_t o_hist = off; off += align_up(((size_t)kSortCells + kSortBlocks) * sizeof(unsigned int), 256);
    if (sl.wf_cap < off) {
        if (sl.wf_mem) CU(cudaFree(sl.wf_mem));
        sl.wf_mem = nullptr; sl.wf_cap = 0;
        cudaError_t e = cudaMalloc(&sl.wf_mem, off);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ERT_ERR_NOMEM, "out of device memory for the wavefront queues");
        }
        sl.wf_cap = off;
    }
    if (sl.wf_ctr_depth < fp.depth) {
        if (sl.wf_ctr) CU(cudaFree(sl.wf_ctr));
        sl.wf_ctr = nullptr; sl.wf_ctr_depth = 0;
        CU(cudaMalloc(&sl.wf_ctr, (size_t)fp.depth * kWfCtr * sizeof(unsigned int)));
        sl.wf_ctr_depth = fp.depth;
    }
    if (!sl.wf_ctr_host) CU(cudaMallocHost(&sl.wf_ctr_host, kWfCtr * sizeof(unsigned int)));
    if (!sl.wf_ctr_all_host) CU(cudaMallocHost(&sl.wf_ctr_all_host, ERT_MAX_BOUNCE_STATS * kWfCtr * sizeof(unsigned int)));
    unsigned char *base = (unsigned char *)sl.wf_mem;
    double *d = (double *)(base + o_dbl);
    int *i = (int *)(base + o_int);
    wf.n_pad = (int)n_pad;
    wf.tiles_x = tiles_x;
    wf.C = d; wf.res_t = d + 3 * n_pad;
    wf.q = (PathRec *)(base + o_path); wf.nq = wf.q + n_pad;
    wf.hit_head = (HitHead *)(base + o_rec); wf.raw_head = wf.hit_head + n_pad;
    wf.hit_tail = (HitTail *)(wf.raw_head + n_pad); wf.raw_tail = wf.hit_tail + n_pad;
    wf.res_hit = (int2 *)i; wf.r_key = (unsigned int *)(i + 2 * n_pad);
    wf.lit = base + o_lit;
    wf.hist = (unsigned int *)(base + o_hist);
    wf.sums = wf.hist + kSortCells;
    wf.ctr = sl.wf_ctr;
    wf.sp_best = nullptr; wf.sp_t = nullptr; wf.sp_occ = nullptr;
    if (scan) {
        // per path ray its nearest hit so far; per shadow ray the target's Distance and the occluded flag
        if (n_pad * L >= ((size_t)1 << 32)) return fail(ERT_ERR_BADARG, "frame part has more than 2^32 shadow rays per bounce");
        const size_t o_best = 0, o_t = align_up(n_pad * sizeof(ScanBest), 256);
        const size_t o_occ = o_t + align_up(n_pad * L * sizeof(double), 256);
        const size_t need = o_occ + align_up(n_pad * L, 256);
        if (sl.scan_cap < need) {
            if (sl.scan_mem) CU(cudaFree(sl.scan_mem));
            sl.scan_mem = nullptr; sl.scan_cap = 0;
            if (cudaMalloc(&sl.scan_mem, need) != cudaSuccess) {
                cudaGetLastError();
                return fail(ERT_ERR_NOMEM, "out of device memory for the results of the brute-force scan");
            }
            sl.scan_cap = need;
        }
        unsigned char *sb = (unsigned char *)sl.scan_mem;
        wf.sp_best = (ScanBest *)(sb + o_best); wf.sp_t = (double *)(sb + o_t); wf.sp_occ = sb + o_occ;
    }
    return ERT_OK;
}

template <bool COUNT, bool TRI>
int launch_wavefront(ert_scene *s, Slot &sl, const FrameParams &fp_in, bool unsorted, bool no_grid, bool timed,
                     bool scan, bool cells, uint64_t *launches)
{
    WfBuf wf{};
    int rc;
    const FrameParams &fp = fp_in;
    if ((rc = wf_prepare(s, sl, fp, wf, scan)) != ERT_OK) return rc;
    cudaStream_t st = sl.stream;
    FrameParams fps = fp;                           // shadow kernels count into the second counter set
    fps.counters = fp.counters + CNT_N;
    size_t n_ticks = 0;
    sl.tick_class.clear();
    auto tick = [&](int cls) -> int {              // cls < 0: the opening event
        if (!timed) return ERT_OK;
        if (n_ticks == sl.ticks.size()) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            sl.ticks.push_back(e);
        }
        CU(cudaEventRecord(sl.ticks[n_ticks++], st));
        if (cls >= 0) sl.tick_class.push_back(cls);
        return ERT_OK;
    };
#define TICK(cls) do { if ((rc = tick(cls)) != ERT_OK) return rc; } while (0)
    TICK(-1);
    const DevScene &d = s->dev;
    CU(cudaMemsetAsync(wf.ctr, 0, (size_t)fp.depth * kWfCtr * sizeof(unsigned int), st));
    // the brute-force scan starts from a cleared colour buffer; the path kernels of bounce 0 clear it themselves
    if (scan || fp.depth <= 0) CU(cudaMemsetAsync(wf.C, 0, (size_t)wf.n_pad * 3 * sizeof(double), st));
    uint64_t n = 0;
    // ERT_DEBUG_SYNC=1: synchronise after every launch and name the kernel that faulted
    static const bool debug_sync = getenv("ERT_DEBUG_SYNC") != nullptr;
    // Binning hits by location pays when shadow rays walk the BVH (coherent warps); with a direction
    // grid for every light it costs more than the path rays gain from it (measured on C4: 29.2 vs 27.8 ms).
    static const bool force_sort = getenv("ERT_WF_SORT") != nullptr;
    constexpr int cells_from = 0;                                  // first bounce whose path rays use the cell grid
    constexpr int cells_refill_from = ERT_WF_REFILL_FROM;          // ... and the refilling form of that kernel
    const bool shadows_walk = !no_grid ? d.lg_count < d.n_lights : true;
    const bool no_sort = unsorted || (!shadows_walk && !force_sort);
    // every light has a direction grid and the hits stay in arrival order: shadow rays and the light fold in one kernel
    static const bool env_no_fuse = getenv("ERT_WF_NO_FUSE") != nullptr;
    const bool fused_shade = !env_no_fuse && !scan && !shadows_walk && no_sort && d.n_lights <= kSsMaxLights;
#define WF_CHECK(what)                                                                 \
    do {                                                                               \
        if (debug_sync) {                                                              \
            cudaError_t e__ = cudaStreamSynchronize(st);                               \
            if (e__ != cudaSuccess) {                                                  \
                char buf__[128];                                                       \
                snprintf(buf__, sizeof buf__, "%s (bounce %d)", what, b);              \
                return cuda_fail(e__, buf__);                                          \
            }                                                                          \
        }                                                                              \
    } while (0)
    const WfBuf wf_even = wf;
    WfBuf wf_odd = wf;
    std::swap(wf_odd.q, wf_odd.nq);
    // Two chains per frame.  The reflection rays of bounce b+1 exist as soon as the hits of bounce b do (they do not
    // depend on the shadow rays), so `st` goes straight on to the next bounce's path rays while `st2` answers the
    // shadow rays of bounce b and folds its colours: the tails of the path launches, where a few long walks keep
    // most of the machine idle, fill with shadow rays.  The hit queue then alternates between its two buffer sets
    // (a bounce's records are read until its shading is done).  Not when the hits are binned (the second set is the
    // binning's), not for the brute-force scan (it shares its result arrays between the two kinds of ray), and not
    // when every launch is timed on its own.
    static const bool env_no_overlap = getenv("ERT_WF_NO_OVERLAP") != nullptr;
    const bool overlap = !env_no_overlap && !timed && !scan && no_sort && fp.depth > 1 && d.n_lights > 0 && !debug_sync;
    cudaStream_t st2 = overlap ? sl.stream2 : st;
    if (overlap) {
        std::swap(wf_odd.hit_head, wf_odd.raw_head);
        std::swap(wf_odd.hit_tail, wf_odd.raw_tail);
        while ((int)sl.ev_path.size() < fp.depth) {
            cudaEvent_t e1, e2;
            CU(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            sl.ev_path.push_back(e1);
            sl.ev_shade.push_back(e2);
        }
    }
    int last_shaded = -1;
    for (int b = 0; b < fp.depth; b++) {
        // bounce b reads the path queue the emitters of bounce b-1 wrote and writes the other one
        wf = (b & 1) ? wf_odd : wf_even;
        if (overlap && b >= 2) CU(cudaStreamWaitEvent(st, sl.ev_shade[(size_t)b - 2], 0));   // its hit buffers are free again
        if (b >= 8) {
            // deep recursions: stop launching once the path queue has run dry
            CU(cudaMemcpyAsync(sl.wf_ctr_host, wf.ctr + (size_t)(b - 1) * kWfCtr, kWfCtr * sizeof(unsigned int),
                               cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            if (sl.wf_ctr_host[WF_NNEXT] == 0) break;
        }
        const bool sort = b >= 1 && !no_sort && !scan;
        const bool grid_b = cells && b >= cells_from;
        const bool refill = b >= (grid_b ? cells_refill_from : ERT_WF_REFILL_FROM);
        // the path kernels emit their hit records themselves unless the hits are to be binned first
        const bool emitted = !scan && (b == 0 || !sort);
        if (scan) {
            // planes/triangles seed every ray's result (counted with the other kernels), then every ray meets every sphere
            if (b == 0) wf_scan_init<false, true, COUNT, TRI><<<s->wf_grid[3], 256, 0, st>>>(d, fp, wf, b);
            else wf_scan_init<false, false, COUNT, TRI><<<s->wf_grid[3], 256, 0, st>>>(d, fp, wf, b);
            n++;
            TICK(2);
            if (b == 0) wf_scan<false, true, COUNT><<<s->wf_grid_scan, kScanThreads, kScanSmem, st>>>(d, fp, wf, b);
            else wf_scan<false, false, COUNT><<<s->wf_grid_scan, kScanThreads, kScanSmem, st>>>(d, fp, wf, b);
        }
        else if (cells && b >= cells_from) {
            // path rays step through the cell grid (ERT_ACCEL_GRID)
            if (b == 0) wf_trace_path<true, COUNT, true, true, TRI><<<s->wf_grid[4], kWfThreads, 0, st>>>(d, fp, wf, b);
            else if (!refill && !emitted) wf_trace_path<false, COUNT, false, true, TRI><<<s->wf_grid[5], kWfThreads, 0, st>>>(d, fp, wf, b);
            else if (!refill) wf_trace_path<false, COUNT, true, true, TRI><<<s->wf_grid[5], kWfThreads, 0, st>>>(d, fp, wf, b);
            else if (!emitted) wf_trace_path_refill<COUNT, true, false, TRI><<<s->wf_grid[5], kWfThreads, 0, st>>>(d, fp, wf, b);
            else wf_trace_path_refill<COUNT, true, true, TRI><<<s->wf_grid[5], kWfThreads, 0, st>>>(d, fp, wf, b);
        }
        else if (b == 0) wf_trace_path<true, COUNT, true, false, TRI><<<s->wf_grid[0], kWfThreads, 0, st>>>(d, fp, wf, b);
        else if (!refill && !emitted) wf_trace_path<false, COUNT, false, false, TRI><<<s->wf_grid[1], kWfThreads, 0, st>>>(d, fp, wf, b);
        else if (!refill) wf_trace_path<false, COUNT, true, false, TRI><<<s->wf_grid[1], kWfThreads, 0, st>>>(d, fp, wf, b);
        else if (!emitted) wf_trace_path_refill<COUNT, false, false, TRI><<<s->wf_grid[1], kWfThreads, 0, st>>>(d, fp, wf, b);
        else wf_trace_path_refill<COUNT, false, true, TRI><<<s->wf_grid[1], kWfThreads, 0, st>>>(d, fp, wf, b);
        n++;
        TICK(0);
        WF_CHECK("wf_trace_path");
        if (d.n_lights == 0) break;          // the fold over no lights is black (erl:211-252)
        if (scan) {
            // results to the arrays the hit emission reads (counted with it)
            if (b == 0) wf_scan_finish<false, true><<<s->wf_grid[3], 256, 0, st>>>(d, wf, b);
            else wf_scan_finish<false, false><<<s->wf_grid[3], 256, 0, st>>>(d, wf, b);
            n++;
        }
        if (emitted) {
            n--;                                 // no separate launch
        } else if (b == 0) {
            wf_emit_hits<true, false><<<s->wf_grid[3], kWfThreads, 0, st>>>(d, fp, wf, b);
        } else if (!sort) {
            wf_emit_hits<false, false><<<s->wf_grid[3], kWfThreads, 0, st>>>(d, fp, wf, b);
        } else {
            CU(cudaMemsetAsync(wf.hist, 0, (size_t)kSortCells * sizeof(unsigned int), st));
            wf_emit_hits<false, true><<<s->wf_grid[3], kWfThreads, 0, st>>>(d, fp, wf, b);
            wf_bin_scan_a<<<kSortBlocks, 1024, 0, st>>>(wf);
            wf_bin_scan_b<<<1, kSortScanBThreads, 0, st>>>(wf);
            wf_bin_scatter<<<s->wf_grid[3], kWfThreads, 0, st>>>(wf, b);
            n += 3;
        }
        n++;
        TICK(2);
        WF_CHECK("wf_emit_hits / wf_bin_*");
        if (overlap) {
            // the hits and the next rays of this bounce exist: the other stream takes the shadow rays from here
            CU(cudaEventRecord(sl.ev_path[(size_t)b], st));
            CU(cudaStreamWaitEvent(st2, sl.ev_path[(size_t)b], 0));
        }
        if (scan) {
            wf_scan_init<true, false, COUNT, TRI><<<s->wf_grid[3], 256, 0, st2>>>(d, fps, wf, b);
            n++;
            TICK(2);
            wf_scan<true, false, COUNT><<<s->wf_grid_scan, kScanThreads, kScanSmem, st2>>>(d, fps, wf, b);
        }
        else if (fused_shade) wf_shadow_shade<COUNT, TRI><<<s->wf_grid[6], kWfThreads, 0, st2>>>(d, fps, wf, b);
        else if (no_grid) wf_trace_shadow<COUNT, false, TRI><<<s->wf_grid[2], kWfThreads, 0, st2>>>(d, fps, wf, b);
        else wf_trace_shadow<COUNT, true, TRI><<<s->wf_grid[2], kWfThreads, 0, st2>>>(d, fps, wf, b);
        TICK(1);
        WF_CHECK("wf_trace_shadow");
        if (scan) {
            wf_scan_finish<true, false><<<s->wf_grid[3], 256, 0, st2>>>(d, wf, b);
            n++;
        }
        if (!fused_shade) {
            wf_shade<<<s->wf_grid[3], kWfThreads, 0, st2>>>(d, fp, wf, b);
            n++;
        }
        if (overlap) CU(cudaEventRecord(sl.ev_shade[(size_t)b], st2));
        last_shaded = b;
        n++;
        TICK(2);
        WF_CHECK("wf_shade");
    }
    if (overlap && last_shaded >= 0) CU(cudaStreamWaitEvent(st, sl.ev_shade[(size_t)last_shaded], 0));
    wf_finalize<<<s->wf_grid_fin, kWfThreads, 0, st>>>(fp, wf);
    n++;
    TICK(2);
    sl.wf_levels = std::min(fp.depth, (int)ERT_MAX_BOUNCE_STATS);
    CU(cudaMemcpyAsync(sl.wf_ctr_all_host, wf.ctr, (size_t)sl.wf_levels * kWfCtr * sizeof(unsigned int),
                       cudaMemcpyDeviceToHost, st));
    CU(cudaGetLastError());
#undef WF_CHECK
#undef TICK
    *launches = n;
    return ERT_OK;
}

int finish_slot(ert_scene *s, Slot &sl)
{
    if (!sl.busy) return ERT_OK;
    cudaError_t e = cudaStreamSynchronize(sl.stream);
    sl.busy = false;
    if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
    float k = 0, t = 0;
    cudaEventElapsedTime(&k, sl.ev0, sl.ev1);
    cudaEventElapsedTime(&t, sl.ev0, sl.ev2);
    sl.stats.kernel_ms = k;
    sl.stats.total_ms = t;
    const unsigned long long *c0 = sl.counters_host, *c1 = sl.counters_host + CNT_N;
    sl.stats.rays = c0[CNT_RAYS] + c1[CNT_RAYS];
    sl.stats.sphere_filter_tests = c0[CNT_FILTER] + c1[CNT_FILTER];
    sl.stats.box_tests = c0[CNT_BOX] + c1[CNT_BOX];
    sl.stats.exact_sphere_tests = c0[CNT_EXACT_SPH] + c1[CNT_EXACT_SPH];
    sl.stats.exact_other_tests = c0[CNT_EXACT_OTHER] + c1[CNT_EXACT_OTHER];
    sl.stats.cell_steps = c0[CNT_CELL] + c1[CNT_CELL];
#ifdef ERT_PROBE
    fprintf(stderr, "PROBE path rays %llu filter %llu exact %llu cell %llu :", c0[CNT_RAYS], c0[CNT_FILTER], c0[CNT_EXACT_SPH], c0[CNT_CELL]);
    for (int k = 0; k < 8; k++) fprintf(stderr, " p%d=%llu", k, c0[CNT_PROBE + k]);
    {
        unsigned long long r[8];
        cudaMemcpyFromSymbol(r, g_sb_reason, sizeof r);
        fprintf(stderr, "\nPROBE triage open reasons: empty %llu rest-beyond-target %llu list-exhausted %llu tries-exhausted %llu (%llu)", r[0], r[1], r[2], r[3], r[4]);
        unsigned long long z[8] = {0};
        cudaMemcpyToSymbol(g_sb_reason, z, sizeof z);
    }
    fprintf(stderr, "\nPROBE shadow rays %llu filter %llu exact %llu :", c1[CNT_RAYS], c1[CNT_FILTER], c1[CNT_EXACT_SPH]);
    for (int k = 0; k < 8; k++) fprintf(stderr, " p%d=%llu", k, c1[CNT_PROBE + k]);
    fprintf(stderr, "\n");
#endif
    sl.stats.bounces_recorded = sl.wf_levels;
    for (int b = 0; b < sl.wf_levels; b++) {
        const unsigned int *c = sl.wf_ctr_all_host + (size_t)b * kWfCtr;
        sl.stats.bounce_hits[b] = c[WF_NHITS];
        sl.stats.bounce_path_rays[b] = b == 0 ? sl.stats.pixels : sl.wf_ctr_all_host[(size_t)(b - 1) * kWfCtr + WF_NNEXT];
    }
    sl.wf_levels = 0;
    sl.stats.has_cell_grid = s->host.cgrid.enabled ? 1 : 0;
    sl.stats.path_box_tests = c0[CNT_BOX]; sl.stats.path_filter_tests = c0[CNT_FILTER];
    sl.stats.shadow_box_tests = c1[CNT_BOX]; sl.stats.shadow_filter_tests = c1[CNT_FILTER];
    // per-class device time of the wavefront launches (ERT_FLAG_TIME_KERNELS)
    for (size_t i = 0; i + 1 < sl.tick_class.size() + 1 && i < sl.tick_class.size(); i++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, sl.ticks[i], sl.ticks[i + 1]) != cudaSuccess) { cudaGetLastError(); continue; }
        switch (sl.tick_class[i]) {
        case 0: sl.stats.path_ms += ms; sl.stats.path_launches++; break;
        case 1: sl.stats.shadow_ms += ms; sl.stats.shadow_launches++; break;
        default: sl.stats.other_ms += ms; break;
        }
    }
    sl.tick_class.clear();
    (void)s;
    return ERT_OK;
}

// ---- in-place update (ert_scene_update) ---------------------------------------------------------------------------

// the new element tables of an update in the staging buffer, and which of them differ from the scene's
struct UpdateTables { double *p[T_COUNT]; bool changed[T_COUNT]; };

// Checks desc against the scene's list shape and every value, writes the new tables into the staging buffer in the
// scene's element order and sets inf.changed.  Nothing of the scene is written.
int update_stage(ert_scene *s, const ert_scene_desc *d, UpdateTables &t, ert_update_info &inf)
{
    HostScene &h = s->host;
    SourceOrder src;
    std::string err = check_update(d, h.order, src);
    if (!err.empty()) return fail(ERT_ERR_BADARG, err);
    size_t off[T_COUNT + 1] = {0};
    for (int k = 0; k < T_COUNT; k++) off[k + 1] = off[k] + h.tab[k].size();
    if (s->staging_cap < off[T_COUNT] * sizeof(double)) {
        if (s->staging) CU(cudaFreeHost(s->staging));
        s->staging = nullptr;
        s->staging_cap = 0;
        if (cudaMallocHost(&s->staging, std::max<size_t>(off[T_COUNT], 1) * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            s->staging = nullptr;
            return fail(ERT_ERR_NOMEM, "out of pinned host memory for the update's staging buffer");
        }
        s->staging_cap = off[T_COUNT] * sizeof(double);
    }
    for (int k = 0; k < T_COUNT; k++) t.p[k] = (double *)s->staging + off[k];
    if (!(err = pack_tables(*d, src, t.p)).empty()) return fail(ERT_ERR_BADARG, err);
    for (int k = 0; k < T_COUNT; k++) {
        const size_t n = h.tab[k].size();
        t.changed[k] = s->broken || (n && memcmp(t.p[k], h.tab[k].data(), n * sizeof(double)) != 0);
        if (t.changed[k] && n) inf.changed |= kTables[k].changed;
    }
    for (int64_t i = 0; i < h.n_lights; i++)
        if (memcmp(&t.p[T_LIGHTS][i * 9 + 3], &h.tab[T_LIGHTS][(size_t)i * 9 + 3], 3 * sizeof(double)) != 0)
            inf.changed |= ERT_CHANGED_LIGHT_POS;
    if (memcmp(&d->camera, &h.camera, sizeof d->camera) != 0) inf.changed |= ERT_CHANGED_CAMERA;
    return ERT_OK;
}

int free_alloc(ert_scene *s, const void *p)
{
    auto it = std::find(s->allocs.begin(), s->allocs.end(), p);
    if (it == s->allocs.end()) return ERT_OK;
    s->allocs.erase(it);
    CU(cudaFree(const_cast<void *>(p)));
    return ERT_OK;
}

void drop_plan(RefitPlan &plan)
{
    if (plan.order) cudaFree(plan.order);
    plan.order = nullptr;
    plan.off.clear();
}

double tree_area(const std::vector<BvhNode> &nodes)
{
    double a = 0;
    for (const BvhNode &n : nodes) a += child_half_area(n, 0) + child_half_area(n, 1);
    return a;
}

// The refit schedule of a tree, made on its first refit, and its area at build (the host mirror still holds the
// built nodes then).
int ensure_plan(RefitPlan &plan, const std::vector<BvhNode> &nodes, double &build_area)
{
    if (plan.order) return ERT_OK;
    std::vector<int32_t> order;
    refit_levels(nodes, order, plan.off);
    CU(cudaMalloc(&plan.order, std::max<size_t>(order.size(), 1) * sizeof(int32_t)));
    CU(cudaMemcpy(plan.order, order.data(), order.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (build_area == 0) build_area = tree_area(nodes);
    return ERT_OK;
}

template <typename LeafBox>
void launch_refit(const RefitPlan &plan, BvhNode *nodes, const LeafBox &leaf_box, double *area, cudaStream_t st)
{
    for (int lvl = (int)plan.off.size() - 2; lvl >= 0; lvl--) {
        const int cnt = plan.off[(size_t)lvl + 1] - plan.off[(size_t)lvl];
        if (cnt > 0)
            upd_refit_level<<<(cnt + kUpdThreads - 1) / kUpdThreads, kUpdThreads, 0, st>>>(
                nodes, plan.order + plan.off[(size_t)lvl], cnt, leaf_box, area);
    }
}

// The arrays derived on the device by updates (filters, pairs, leaf filters, tree nodes, leaf vertices) from
// src's device into h.
int download_derived(const ert_scene *src, HostScene &h)
{
    const DevScene &d = src->dev;
    CU(cudaSetDevice(src->device));
    auto get = [](void *dst, const void *p, size_t bytes) -> int {
        if (bytes) CU(cudaMemcpy(dst, p, bytes, cudaMemcpyDeviceToHost));
        return ERT_OK;
    };
    int rc;
    if ((rc = get(h.sph_filter.data(), d.sph_filter, h.sph_filter.size() * sizeof(float))) != ERT_OK) return rc;
    if ((rc = get(h.sph_pairs.data(), d.sph_pairs, h.sph_pairs.size() * sizeof(float))) != ERT_OK) return rc;
    if ((rc = get(h.leaf_filter.data(), d.leaf_filter, h.leaf_filter.size() * sizeof(float))) != ERT_OK) return rc;
    if ((rc = get(h.bvh.nodes.data(), d.nodes, h.bvh.nodes.size() * sizeof(BvhNode))) != ERT_OK) return rc;
    if (h.has_tri_bvh) {
        if ((rc = get(h.tbvh.bvh.nodes.data(), d.tri_nodes, h.tbvh.bvh.nodes.size() * sizeof(BvhNode))) != ERT_OK) return rc;
        if ((rc = get(h.tbvh.leaf_tris.data(), d.tri_leaf, h.tbvh.leaf_tris.size() * sizeof(double))) != ERT_OK) return rc;
    }
    h.derived_stale = false;
    return ERT_OK;
}

// A tree triangle left the float range of the boxes (kTriAlwaysAbs): the triangle BVH is built again on the host.
int rebuild_tri_bvh(ert_scene *s)
{
    HostScene &h = s->host;
    DevScene &d = s->dev;
    TriBvh t;
    build_triangle_bvh(h.tab[T_TRIS].data(), h.n_tris, t);
    if (t.bvh.depth >= kBvhStack) return fail(ERT_ERR_BADARG, "triangle BVH is deeper than the traversal stack");
    int rc;
    const void *old[4] = {d.tri_nodes, d.tri_leaf, d.tri_leaf_id, d.tri_always};
    for (const void *p : old)
        if ((rc = free_alloc(s, p)) != ERT_OK) return rc;
    h.tbvh = std::move(t);
    const BvhNode *nodes; const double *leaf; const int *id; const int *always;
    if ((rc = upload(s, h.tbvh.bvh.nodes, &nodes)) != ERT_OK) return rc;
    if ((rc = upload(s, h.tbvh.leaf_tris, &leaf)) != ERT_OK) return rc;
    if ((rc = upload(s, h.tbvh.bvh.leaf_prim, &id)) != ERT_OK) return rc;
    if ((rc = upload(s, h.tbvh.always, &always)) != ERT_OK) return rc;
    d.tri_nodes = nodes; d.tri_leaf = leaf; d.tri_leaf_id = id; d.tri_always = always;
    d.n_tri_tree = (int)h.tbvh.bvh.leaf_prim.size();
    d.n_tri_always = (int)h.tbvh.always.size();
    drop_plan(s->plan_tri);
    h.tri_build_area = tree_area(h.tbvh.bvh.nodes);
    return ERT_OK;
}

// Builds on the device (grid_build.cuh), from the device's current spheres and filter spheres, the cell grid (cell)
// and the direction grids of the lights flagged in `need`; a light whose grid goes over its entry budget ends the
// run of grids.  Adds the H2D bytes (the LightGridDev array) to *h2d.
int build_grids_on_device(ert_scene *s, bool cell, const std::vector<char> &need, cudaStream_t st, uint64_t *h2d)
{
    HostScene &h = s->host;
    const DevScene &d = s->dev;
    if (cell) {
        double density;
        if (cell_grid_wanted(density))
            CU(build_cell_grid_device(d.sph_exact, d.sph_filter, h.n_spheres, h.sph_lo, h.sph_hi, h.abs_max, density,
                                      s->grid_tmp, s->cg_buf, st));
        else
            s->cg_buf.enabled = false;
        h.cgrid = CellGrid();
        h.cgrid.enabled = s->cg_buf.enabled;
        if (h.cgrid.enabled) cell_grid_set_geometry(h.cgrid, s->cg_buf.geo);
        h.cgrid_dev = h.cgrid.enabled;
        set_cell_desc(s);
    }
    if (!need.empty()) {
        const int res = light_grid_res();
        if (s->lg_buf.size() < need.size()) s->lg_buf.resize(need.size());
        size_t keep = 0;
        for (; keep < need.size(); keep++) {
            if (!need[keep]) continue;
            LightGridDevOut &o = s->lg_buf[keep];
            CU(build_light_grid_device(d.sph_exact, d.sph_filter, h.n_spheres, &h.tab[T_LIGHTS][keep * 9 + 3], res,
                                       kLightGridMaxEntries, s->grid_tmp, o, st));
            if (!o.ok) break;
        }
        h.lgrids.resize(keep);
        for (size_t g = 0; g < keep; g++)
            if (need[g]) {
                h.lgrids[g] = LightGrid();
                h.lgrids[g].res = res;
                h.lgrid_dev[g] = true;
            }
        int rc;
        if ((rc = write_light_desc(s, (int)keep, st, h2d)) != ERT_OK) return rc;
    }
    CU(cudaStreamSynchronize(st));
    return ERT_OK;
}

// ERT_UPDATE_REBUILD_GRIDS: the cell grid (cell) and the direction grids of `stale` lights, and any an earlier
// update dropped, built again on the device.
int rebuild_grids(ert_scene *s, bool cell, const std::vector<char> &stale, cudaStream_t st, ert_update_info &inf)
{
    HostScene &h = s->host;
    int rc;
    const int n_target = light_grid_target(h, light_grid_res());
    const size_t have = h.lgrids.size();
    std::vector<char> need((size_t)n_target, 0);
    int n_need = 0;
    for (int g = 0; g < n_target; g++)
        if ((size_t)g >= have || ((size_t)g < stale.size() && stale[(size_t)g])) {
            need[(size_t)g] = 1;
            n_need++;
        }
    const bool lights = n_need > 0 || have < (size_t)n_target;
    if (!lights) need.clear();
    CU(cudaEventRecord(s->upd_ev[0], st));
    if ((rc = build_grids_on_device(s, cell, need, st, &inf.h2d_bytes)) != ERT_OK) return rc;
    CU(cudaEventRecord(s->upd_ev[1], st));
    CU(cudaEventSynchronize(s->upd_ev[1]));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->upd_ev[0], s->upd_ev[1]));
    inf.device_ms += ms;
    if (cell) {
        h.cgrid_dropped = false;
        inf.done |= ERT_DID_REBUILD_CELL_GRID;
    }
    if (lights) {
        h.lgrids_dropped = false;
        inf.done |= ERT_DID_REBUILD_LIGHT_GRIDS;
        inf.light_grids_rebuilt = n_need;
    }
    return ERT_OK;
}

// Everything after the checks: the host mirror takes the staged tables, the changed ones go to the device, the
// kernels of ert_update.cuh recompute what create derived from them, and stale grids are dropped or rebuilt.
int update_apply(ert_scene *s, UpdateTables &t, const ert_camera &camera, uint32_t flags, ert_update_info &inf)
{
    HostScene &h = s->host;
    DevScene &d = s->dev;
    cudaStream_t st = s->slots[0].stream;
    int rc;
    const bool was_broken = s->broken;
    const bool sph_geo = t.changed[T_SPH_EXACT] && h.n_spheres > 0;
    const bool tri_geo = t.changed[T_TRIS] && h.has_tri_bvh && !h.tbvh.bvh.leaf_prim.empty();
    // lights whose direction grid went stale
    std::vector<char> lg_stale(h.lgrids.size(), 0);
    for (size_t g = 0; g < h.lgrids.size(); g++)
        lg_stale[g] = sph_geo || was_broken || memcmp(&t.p[T_LIGHTS][g * 9 + 3], &h.tab[T_LIGHTS][g * 9 + 3], 3 * sizeof(double)) != 0;
    s->broken = true;                 // until every step below has succeeded
    h.camera = camera;
    if (!s->upd_dev) CU(cudaMalloc(&s->upd_dev, sizeof(UpdateScalars)));
    if (!s->upd_host) CU(cudaMallocHost(&s->upd_host, sizeof(UpdateScalars)));
    if (sph_geo && (rc = ensure_plan(s->plan_sph, h.bvh.nodes, h.sph_build_area)) != ERT_OK) return rc;
    if (tri_geo && (rc = ensure_plan(s->plan_tri, h.tbvh.bvh.nodes, h.tri_build_area)) != ERT_OK) return rc;

    CU(cudaEventRecord(s->upd_ev[0], st));
    for (int k = 0; k < T_COUNT; k++) {
        if (!t.changed[k] || h.tab[k].empty()) continue;
        const size_t bytes = h.tab[k].size() * sizeof(double);
        memcpy(h.tab[k].data(), t.p[k], bytes);
        CU(cudaMemcpyAsync(const_cast<double *>(s->tab_dev[k]), t.p[k], bytes, cudaMemcpyHostToDevice, st));
        inf.h2d_bytes += bytes;
    }
    UpdateScalars &u = *s->upd_host;
    memset(&u, 0, sizeof u);
    for (int a = 0; a < 3; a++) u.lo[a] = ~0ull;
    CU(cudaMemcpyAsync(s->upd_dev, &u, sizeof u, cudaMemcpyHostToDevice, st));
    if (sph_geo) {
        const int n = h.n_spheres;
        upd_spheres<<<(n + kUpdThreads - 1) / kUpdThreads, kUpdThreads, 0, st>>>(
            d.sph_exact, d.leaf_sph, n, const_cast<float4 *>(d.sph_filter), const_cast<float *>((const float *)d.sph_pairs),
            const_cast<float4 *>(d.leaf_filter), s->upd_dev);
        launch_refit(s->plan_sph, const_cast<BvhNode *>(d.nodes), SphereLeafBox{d.sph_exact, d.leaf_sph},
                     &s->upd_dev->area_sph, st);
    }
    if (tri_geo) {
        const int n = d.n_tri_tree;
        upd_triangles<<<(n + kUpdThreads - 1) / kUpdThreads, kUpdThreads, 0, st>>>(d.tris, d.tri_leaf_id, n,
                                                                                   const_cast<double *>(d.tri_leaf), s->upd_dev);
        launch_refit(s->plan_tri, const_cast<BvhNode *>(d.tri_nodes), TriangleLeafBox{d.tri_leaf}, &s->upd_dev->area_tri, st);
    }
    CU(cudaGetLastError());
    CU(cudaEventRecord(s->upd_ev[1], st));
    CU(cudaMemcpyAsync(&u, s->upd_dev, sizeof u, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->upd_ev[0], s->upd_ev[1]));
    inf.device_ms = ms;

    if (sph_geo) {
        // the constants flatten() folds over the spheres, from the same per-sphere values (max and min do not
        // depend on the order)
        memcpy(&h.r_max, &u.r_max, 4); memcpy(&h.pad_c_max, &u.pad_c_max, 4);
        memcpy(&h.eta_c_max, &u.eta_c_max, 4); memcpy(&h.abs_max, &u.abs_max, 4);
        double lo[3], hi[3];
        for (int a = 0; a < 3; a++) { lo[a] = dkey_value(u.lo[a]); hi[a] = dkey_value(u.hi[a]); }
        set_sort_grid(h, lo, hi);
        for (int a = 0; a < 3; a++) { h.sph_lo[a] = lo[a]; h.sph_hi[a] = hi[a]; }
        h.derived_stale = true;
        inf.done |= ERT_DID_REFIT_SPHERES;
        if (h.sph_build_area > 0) inf.sphere_area_ratio = u.area_sph / h.sph_build_area;
    }
    if (tri_geo) {
        double e, m;
        memcpy(&e, &u.tri_edge, 8);
        memcpy(&m, &u.tri_abs, 8);
        if (!(m <= kTriAlwaysAbs)) {
            // the builder's admission rule: a box of float cannot hold this triangle
            if ((rc = rebuild_tri_bvh(s)) != ERT_OK) return rc;
            inf.done |= ERT_DID_REBUILD_TRI_BVH;
        } else {
            h.tbvh.edge_max = e * (1.0 + 1.0 / 1099511627776.0);   // as build_triangle_bvh rounds it up
            h.tbvh.abs_max = m;
            h.derived_stale = true;
            inf.done |= ERT_DID_REFIT_TRIANGLES;
            if (h.tri_build_area > 0) inf.triangle_area_ratio = u.area_tri / h.tri_build_area;
        }
    }
    set_constants(s);

    // grids: the cell grid and the direction grids hold copies of filter spheres, a direction grid its light
    const bool cell_stale = sph_geo && h.cgrid.enabled;
    bool lg_any = false;
    for (char c : lg_stale) lg_any = lg_any || c;
    if (flags & ERT_UPDATE_REBUILD_GRIDS) {
        // a grid the spheres refused (a knot of more than kCellGridMaxCount) is tried again when they move
        const bool cell = cell_stale || h.cgrid_dropped || (sph_geo && h.n_spheres >= kCellGridMinSpheres);
        if ((cell || lg_any || h.lgrids_dropped) && (rc = rebuild_grids(s, cell, lg_stale, st, inf)) != ERT_OK) return rc;
    } else {
        if (cell_stale) {
            h.cgrid.enabled = false;
            d.cg.enabled = 0;
            h.cgrid_dropped = true;
            inf.done |= ERT_DID_DROP_CELL_GRID;
        }
        if (lg_any) {
            size_t keep = 0;
            while (keep < lg_stale.size() && !lg_stale[keep]) keep++;
            h.lgrids.resize(keep);
            d.lg_count = (int)keep;
            h.lgrids_dropped = true;
            inf.done |= ERT_DID_DROP_LIGHT_GRIDS;
        }
    }
    s->broken = false;
    return ERT_OK;
}

// ERT_UPDATE_REBUILD: the create path into the scene's handle
int update_rebuild(ert_scene *s, const ert_scene_desc *desc, ert_update_info &inf)
{
    HostScene h;
    int rc = flatten(desc, h);
    if (rc != ERT_OK) return rc;
    s->broken = true;
    CU(cudaEventRecord(s->upd_ev[0], 0));
    for (void *p : s->allocs) cudaFree(p);
    s->allocs.clear();
    drop_plan(s->plan_sph);
    drop_plan(s->plan_tri);
    s->host = std::move(h);
    s->host.sph_build_area = tree_area(s->host.bvh.nodes);
    if (s->host.has_tri_bvh) s->host.tri_build_area = tree_area(s->host.tbvh.bvh.nodes);
    const uint64_t before = s->uploaded;
    if ((rc = upload_tables(s)) != ERT_OK) return rc;
    CU(cudaEventRecord(s->upd_ev[1], 0));
    CU(cudaEventSynchronize(s->upd_ev[1]));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->upd_ev[0], s->upd_ev[1]));
    inf.device_ms = ms;
    inf.h2d_bytes = s->uploaded - before;
    inf.done |= ERT_DID_REBUILD;
    s->broken = false;
    return ERT_OK;
}

}  // namespace

extern "C" {

int ert_abi_version(void) { return ERT_ABI_VERSION; }

const char *ert_last_error(void) { return g_err.c_str(); }

int ert_device_count(int *count)
{
    if (!count) return fail(ERT_ERR_BADARG, "count is NULL");
    *count = 0;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    *count = n;
    return ERT_OK;
}

static int check_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    if (n <= 0) return fail(ERT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU fallback");
    if (device < 0 || device >= n) return fail(ERT_ERR_BADARG, "device index out of range");
    return ERT_OK;
}

int ert_scene_create(const ert_scene_desc *desc, int device, ert_scene **out)
{
    if (!out) return fail(ERT_ERR_BADARG, "out is NULL");
    *out = nullptr;
    ert_scene *s = new (std::nothrow) ert_scene();
    if (!s) return fail(ERT_ERR_NOMEM, "out of host memory");
    s->device = device;
    int rc;
    try {
        rc = flatten(desc, s->host);
    } catch (const std::bad_alloc &) {
        delete s;
        return fail(ERT_ERR_NOMEM, "out of host memory while flattening the scene");
    } catch (const std::exception &e) {
        delete s;
        return fail(ERT_ERR_NOMEM, std::string("scene build failed: ") + e.what());
    }
    if (rc != ERT_OK) { delete s; return rc; }
    if ((rc = check_device(device)) != ERT_OK) { delete s; return rc; }
    try {
        rc = upload_scene(s);
    } catch (const std::exception &e) {
        g_err = std::string("out of host memory while uploading the scene: ") + e.what();
        rc = ERT_ERR_NOMEM;
    }
    if (rc != ERT_OK) {
        std::string keep = g_err;
        destroy(s);
        g_err = keep;
        return rc;
    }
    *out = s;
    return ERT_OK;
}

int ert_scene_clone(const ert_scene *src, int device, ert_scene **out)
{
    if (!src || !out) return fail(ERT_ERR_BADARG, "NULL argument");
    *out = nullptr;
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    ert_scene *s = new (std::nothrow) ert_scene();
    if (!s) return fail(ERT_ERR_NOMEM, "out of host memory");
    s->device = device;
    {
        // an updated source's filters and trees are current on its device only
        std::lock_guard<std::mutex> lock(const_cast<ert_scene *>(src)->mu);
        if (src->broken) {
            delete s;
            return fail(ERT_ERR_CUDA, "the source scene's last update failed");
        }
        try {
            s->host = src->host;
            rc = s->host.derived_stale ? download_derived(src, s->host) : ERT_OK;
        } catch (const std::exception &) {
            delete s;
            return fail(ERT_ERR_NOMEM, "out of host memory");
        }
        if (rc != ERT_OK) { delete s; return rc; }
    }
    try {
        rc = upload_scene(s);
        // grids built on the source's device: the same builders on this one, from the same tables
        HostScene &h = s->host;
        std::vector<char> need(h.lgrids.size(), 0);
        bool any = h.cgrid_dev;
        for (size_t g = 0; g < need.size(); g++) any |= (need[g] = h.lgrid_dev[g] ? 1 : 0) != 0;
        if (rc == ERT_OK && any) {
            const size_t n_grids = h.lgrids.size();
            rc = build_grids_on_device(s, h.cgrid_dev, need, s->slots[0].stream, nullptr);
            if (rc == ERT_OK && h.lgrids.size() != n_grids) rc = fail(ERT_ERR_CUDA, "a direction grid of the source failed to build again");
        }
    } catch (const std::exception &e) {
        g_err = std::string("out of host memory while uploading the scene: ") + e.what();
        rc = ERT_ERR_NOMEM;
    }
    if (rc != ERT_OK) {
        std::string keep = g_err;
        destroy(s);
        g_err = keep;
        return rc;
    }
    *out = s;
    return ERT_OK;
}

int ert_scene_destroy(ert_scene *scene)
{
    if (!scene) return ERT_OK;
    destroy(scene);
    return ERT_OK;
}

int ert_scene_update(ert_scene *scene, const ert_scene_desc *desc, uint32_t flags, ert_update_info *info)
{
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene) return fail(ERT_ERR_BADARG, "scene is NULL");
    if (flags & ~(ERT_UPDATE_REBUILD_GRIDS | ERT_UPDATE_REBUILD)) return fail(ERT_ERR_BADARG, "unknown update flags");
    std::lock_guard<std::mutex> lock(scene->mu);
    CU(cudaSetDevice(scene->device));
    ert_update_info inf{};
    inf.sphere_area_ratio = inf.triangle_area_ratio = 1.0;
    UpdateTables t{};
    int rc;
    try {
        rc = update_stage(scene, desc, t, inf);
    } catch (const std::exception &) {
        return fail(ERT_ERR_NOMEM, "out of host memory while checking the update");
    }
    if (rc != ERT_OK) return rc;
    // frames already queued render the scene they were queued with
    for (Slot &sl : scene->slots)
        if ((rc = finish_slot(scene, sl)) != ERT_OK) return rc;
    if (!scene->upd_ev[0]) CU(cudaEventCreate(&scene->upd_ev[0]));
    if (!scene->upd_ev[1]) CU(cudaEventCreate(&scene->upd_ev[1]));
    try {
        rc = (flags & ERT_UPDATE_REBUILD) ? update_rebuild(scene, desc, inf) : update_apply(scene, t, desc->camera, flags, inf);
    } catch (const std::exception &e) {
        scene->broken = true;
        rc = fail(ERT_ERR_NOMEM, std::string("scene update failed: ") + e.what());
    }
    if (rc != ERT_OK) return rc;
    inf.has_cell_grid = scene->host.cgrid.enabled ? 1 : 0;
    inf.light_grids = (int32_t)scene->host.lgrids.size();
    inf.host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (info) *info = inf;
    return ERT_OK;
}

int ert_render_async(ert_scene *scene, const ert_render_params *params, int slot, void *host_frame,
                     size_t host_frame_bytes)
{
    if (!scene) return fail(ERT_ERR_BADARG, "scene is NULL");
    int rc;
    if ((rc = check_params(params)) != ERT_OK) return rc;
    if (slot < 0 || slot >= ERT_MAX_SLOTS) return fail(ERT_ERR_BADARG, "slot out of range");
    std::lock_guard<std::mutex> lock(scene->mu);
    if (scene->broken) return fail(ERT_ERR_CUDA, "the scene's last update failed: update it again or destroy it");
    CU(cudaSetDevice(scene->device));
    Slot &sl = scene->slots[slot];
    if ((rc = finish_slot(scene, sl)) != ERT_OK) return rc;

    const ert_render_params &p = *params;
    const ert_camera &cam = p.camera ? *p.camera : scene->host.camera;
    if (const std::string err = check_camera(cam); !err.empty()) return fail(ERT_ERR_BADARG, err);

    FrameParams fp{};
    fp.width = p.width; fp.height = p.height; fp.depth = p.depth; fp.format = p.format;
    fp.band_rows = p.band_rows; fp.n_parts = p.n_parts <= 1 ? 1 : p.n_parts; fp.part = p.part;
    if (fp.n_parts == 1 || p.band_rows <= 0) { fp.n_parts = 1; fp.part = 0; fp.band_rows = 0; }
    fp.local_rows = local_rows_of(p);
    fp.cam[0] = cam.location[0]; fp.cam[1] = cam.location[1]; fp.cam[2] = cam.location[2];
    // focal_length/2 (erl:483-484) with the host libm's tan, as BEAM's math:tan would
    fp.focal = cam.screen_width / (2 * tan(cam.fov * (M_PI / 180) / 2));
    fp.screen_w = cam.screen_width; fp.screen_h = cam.screen_height;

    size_t fb_bytes = (size_t)std::max(fp.local_rows, 1) * (size_t)p.width * 3 * bytes_per_channel(p.format);
    if (sl.fb_cap < fb_bytes) {
        if (sl.fb) CU(cudaFree(sl.fb));
        sl.fb = nullptr; sl.fb_cap = 0;
        CU(cudaMalloc(&sl.fb, fb_bytes));
        sl.fb_cap = fb_bytes;
    }
    fp.out = sl.fb;
    fp.counters = sl.counters_dev;

    sl.params = p;
    sl.params.camera = nullptr;
    sl.local_rows = fp.local_rows;
    sl.stats = ert_stats{};
    int accel = pick_accel(scene, p.accel);
    sl.stats.accel_used = accel;
    sl.stats.pixels = (uint64_t)fp.local_rows * (uint64_t)p.width;
    sl.stats.h2d_bytes = sizeof(DevScene) + sizeof(FrameParams);   // kernel parameters of this frame

    CU(cudaMemsetAsync(sl.counters_dev, 0, kCounterSets * CNT_N * sizeof(unsigned long long), sl.stream));
    CU(cudaEventRecord(sl.ev0, sl.stream));
    // the wavefront serves the BVH strategy and, past one resident tile of spheres, the brute-force scan
    const bool wf_scan = accel == ERT_ACCEL_LINEAR && scene->host.n_spheres > kWfScanFrom;
    const bool wf_cells = accel == ERT_ACCEL_GRID;
    if (fp.local_rows > 0 && (accel == ERT_ACCEL_BVH || wf_cells || wf_scan) && fp.depth > 0) {
        uint64_t n = 0;
        const bool unsorted = (p.flags & ERT_FLAG_WF_UNSORTED) != 0;
        const bool no_grid = (p.flags & ERT_FLAG_NO_LIGHT_GRID) != 0;
        const bool timed = (p.flags & ERT_FLAG_TIME_KERNELS) != 0;
        const bool count = (p.flags & ERT_FLAG_COUNT_TESTS) != 0;
        if (scene->host.has_tri_bvh)
            rc = count ? launch_wavefront<true, true>(scene, sl, fp, unsorted, no_grid, timed, wf_scan, wf_cells, &n)
                       : launch_wavefront<false, true>(scene, sl, fp, unsorted, no_grid, timed, wf_scan, wf_cells, &n);
        else
            rc = count ? launch_wavefront<true, false>(scene, sl, fp, unsorted, no_grid, timed, wf_scan, wf_cells, &n)
                       : launch_wavefront<false, false>(scene, sl, fp, unsorted, no_grid, timed, wf_scan, wf_cells, &n);
        if (rc != ERT_OK) return rc;
        sl.stats.gpu_launches = n;
    } else if (fp.local_rows > 0) {
        dim3 grid((unsigned)((p.width + 31) / 32), (unsigned)((fp.local_rows + 7) / 8));
        const bool count = (p.flags & ERT_FLAG_COUNT_TESTS) != 0;
        if (scene->host.has_tri_bvh) {
            if (count) launch_render<true, true>(accel, grid, sl.stream, scene->dev, fp);
            else launch_render<false, true>(accel, grid, sl.stream, scene->dev, fp);
        } else {
            if (count) launch_render<true, false>(accel, grid, sl.stream, scene->dev, fp);
            else launch_render<false, false>(accel, grid, sl.stream, scene->dev, fp);
        }
        CU(cudaGetLastError());
        sl.stats.gpu_launches = 1;
    }
    CU(cudaEventRecord(sl.ev1, sl.stream));
    CU(cudaMemcpyAsync(sl.counters_host, sl.counters_dev, kCounterSets * CNT_N * sizeof(unsigned long long),
                       cudaMemcpyDeviceToHost, sl.stream));
    sl.has_frame = true;
    sl.busy = true;
    if (host_frame && fp.local_rows > 0) {
        uint64_t bytes = 0;
        if ((rc = copy_part_to_host(scene, sl, p, host_frame, host_frame_bytes, &bytes)) != ERT_OK) {
            std::string keep = g_err;
            cudaStreamSynchronize(sl.stream);
            sl.busy = false;
            g_err = keep;
            return rc;
        }
        sl.stats.d2h_bytes = bytes;
    }
    CU(cudaEventRecord(sl.ev2, sl.stream));
    return ERT_OK;
}

int ert_wait(ert_scene *scene, int slot)
{
    if (!scene) return fail(ERT_ERR_BADARG, "scene is NULL");
    if (slot < 0 || slot >= ERT_MAX_SLOTS) return fail(ERT_ERR_BADARG, "slot out of range");
    std::lock_guard<std::mutex> lock(scene->mu);
    CU(cudaSetDevice(scene->device));
    return finish_slot(scene, scene->slots[slot]);
}

int ert_render(ert_scene *scene, const ert_render_params *params, void *host_frame, size_t host_frame_bytes)
{
    if (!host_frame) return fail(ERT_ERR_BADARG, "host_frame is NULL");
    int rc = ert_render_async(scene, params, 0, host_frame, host_frame_bytes);
    if (rc != ERT_OK) return rc;
    return ert_wait(scene, 0);
}

int ert_download(ert_scene *scene, int slot, void *host_frame, size_t host_frame_bytes)
{
    if (!scene || !host_frame) return fail(ERT_ERR_BADARG, "NULL argument");
    if (slot < 0 || slot >= ERT_MAX_SLOTS) return fail(ERT_ERR_BADARG, "slot out of range");
    std::lock_guard<std::mutex> lock(scene->mu);
    CU(cudaSetDevice(scene->device));
    Slot &sl = scene->slots[slot];
    int rc;
    if ((rc = finish_slot(scene, sl)) != ERT_OK) return rc;
    if (!sl.has_frame) return fail(ERT_ERR_BADARG, "nothing has been rendered on this slot");
    uint64_t bytes = 0;
    if (sl.local_rows > 0) {
        if ((rc = copy_part_to_host(scene, sl, sl.params, host_frame, host_frame_bytes, &bytes)) != ERT_OK) return rc;
    }
    CU(cudaStreamSynchronize(sl.stream));
    sl.stats.d2h_bytes = bytes;
    return ERT_OK;
}

int ert_get_stats(ert_scene *scene, int slot, ert_stats *out)
{
    if (!scene || !out) return fail(ERT_ERR_BADARG, "NULL argument");
    if (slot < 0 || slot >= ERT_MAX_SLOTS) return fail(ERT_ERR_BADARG, "slot out of range");
    std::lock_guard<std::mutex> lock(scene->mu);
    *out = scene->slots[slot].stats;
    return ERT_OK;
}

int ert_trace_rays(ert_scene *scene, int64_t n_rays, const double *rays6, int accel, int32_t *order_out,
                   double *t_out)
{
    if (!scene || (n_rays > 0 && (!rays6 || !order_out || !t_out))) return fail(ERT_ERR_BADARG, "NULL argument");
    if (n_rays < 0) return fail(ERT_ERR_BADARG, "negative ray count");
    if (accel < ERT_ACCEL_AUTO || accel > ERT_ACCEL_WARP) return fail(ERT_ERR_BADARG, "unknown accel");
    if (n_rays == 0) return ERT_OK;
    std::lock_guard<std::mutex> lock(scene->mu);
    if (scene->broken) return fail(ERT_ERR_CUDA, "the scene's last update failed: update it again or destroy it");
    CU(cudaSetDevice(scene->device));
    accel = pick_accel(scene, accel);
    double *d_rays = nullptr, *d_t = nullptr;
    int *d_ord = nullptr;
    cudaStream_t st = scene->slots[0].stream;
    int rc = ERT_OK;
    bool timed = false;
    cudaError_t e;
#define TRY(call)                                         \
    do {                                                  \
        if ((e = (call)) != cudaSuccess) {                \
            rc = cuda_fail(e, #call);                     \
            goto done;                                    \
        }                                                 \
    } while (0)
    TRY(cudaMalloc(&d_rays, (size_t)n_rays * 6 * sizeof(double)));
    TRY(cudaMalloc(&d_t, (size_t)n_rays * sizeof(double)));
    TRY(cudaMalloc(&d_ord, (size_t)n_rays * sizeof(int)));
    TRY(cudaMemcpyAsync(d_rays, rays6, (size_t)n_rays * 6 * sizeof(double), cudaMemcpyHostToDevice, st));
    {
        unsigned blocks = (unsigned)((n_rays + 255) / 256);
        // the kernel's device time is left in slot 0's stats.kernel_ms (unless a frame is in flight there: its
        // events are not touched)
        Slot &sl0 = scene->slots[0];
        timed = !sl0.busy;
        if (timed) TRY(cudaEventRecord(sl0.ev0, st));
        if (accel == ERT_ACCEL_WARP && n_rays > (1ll << 26)) {
            rc = fail(ERT_ERR_BADARG, "ERT_ACCEL_WARP takes at most 2^26 rays per call");
            goto done;
        }
        if (scene->host.has_tri_bvh) launch_trace_rays<true>(accel, blocks, st, scene->dev, n_rays, d_rays, d_ord, d_t);
        else launch_trace_rays<false>(accel, blocks, st, scene->dev, n_rays, d_rays, d_ord, d_t);
    }
    TRY(cudaGetLastError());
    if (timed) TRY(cudaEventRecord(scene->slots[0].ev1, st));
    TRY(cudaMemcpyAsync(order_out, d_ord, (size_t)n_rays * sizeof(int), cudaMemcpyDeviceToHost, st));
    TRY(cudaMemcpyAsync(t_out, d_t, (size_t)n_rays * sizeof(double), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    if (timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, scene->slots[0].ev0, scene->slots[0].ev1) == cudaSuccess) scene->slots[0].stats.kernel_ms = ms;
    }
#undef TRY
done:
    if (d_rays) cudaFree(d_rays);
    if (d_t) cudaFree(d_t);
    if (d_ord) cudaFree(d_ord);
    return rc;
}

int ert_host_alloc(size_t bytes, void **out)
{
    if (!out) return fail(ERT_ERR_BADARG, "out is NULL");
    *out = nullptr;
    CU(cudaMallocHost(out, std::max<size_t>(bytes, 1)));
    return ERT_OK;
}
int ert_host_free(void *p)
{
    if (p) CU(cudaFreeHost(p));
    return ERT_OK;
}
int ert_host_register(void *p, size_t bytes)
{
    if (!p) return fail(ERT_ERR_BADARG, "pointer is NULL");
    CU(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return ERT_OK;
}
int ert_host_unregister(void *p)
{
    if (p) CU(cudaHostUnregister(p));
    return ERT_OK;
}

int ert_fp32_peak(int device, double *lane_instr_per_s)
{
    if (!lane_instr_per_s) return fail(ERT_ERR_BADARG, "out is NULL");
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    int blocks = prop.multiProcessorCount * 8;
    float *out = nullptr;
    CU(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(float)));
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    const int iters = 4096;
    double best = 0;
    for (int rep = 0; rep < 6; rep++) {
        CU(cudaEventRecord(a));
        fp32_peak_kernel<<<blocks, 256>>>(out, iters, 1.0f + rep);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        double rate = (double)blocks * 256.0 * iters * kPeakFfmaPerIter / (ms * 1e-3);
        if (rep > 0) best = std::max(best, rate);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(out);
    *lane_instr_per_s = best;
    return ERT_OK;
}

int ert_fp32_peak_rrr(int device, double *lane_instr_per_s)
{
    if (!lane_instr_per_s) return fail(ERT_ERR_BADARG, "out is NULL");
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    int blocks = prop.multiProcessorCount * 8;
    float *out = nullptr, *in = nullptr;
    CU(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(float)));
    CU(cudaMalloc(&in, 8 * sizeof(float)));
    const float host_in[8] = {1.0f, 0.9999f, 0.99991f, 0.0001f, 0.00011f, 0, 0, 0};
    CU(cudaMemcpy(in, host_in, sizeof host_in, cudaMemcpyHostToDevice));
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    const int iters = 4096;
    double best = 0;
    for (int rep = 0; rep < 6; rep++) {
        CU(cudaEventRecord(a));
        fp32_peak_rrr_kernel<<<blocks, 256>>>(out, iters, in);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        double rate = (double)blocks * 256.0 * iters * kPeakFfmaPerIter / (ms * 1e-3);
        if (rep > 0) best = std::max(best, rate);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(out);
    cudaFree(in);
    *lane_instr_per_s = best;
    return ERT_OK;
}

int ert_fp64_peak(int device, double *lane_instr_per_s)
{
    if (!lane_instr_per_s) return fail(ERT_ERR_BADARG, "out is NULL");
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    int blocks = prop.multiProcessorCount * 8;
    double *out = nullptr, *in = nullptr;
    CU(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(double)));
    CU(cudaMalloc(&in, 8 * sizeof(double)));
    const double host_in[8] = {1.0, 0.9999, 0.99991, 0.0001, 0.00011, 0, 0, 0};
    CU(cudaMemcpy(in, host_in, sizeof host_in, cudaMemcpyHostToDevice));
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    const int iters = 2048;
    double best = 0;
    for (int rep = 0; rep < 6; rep++) {
        CU(cudaEventRecord(a));
        fp64_peak_kernel<<<blocks, 256>>>(out, iters, in);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        double rate = (double)blocks * 256.0 * iters * kPeakFfmaPerIter / (ms * 1e-3);
        if (rep > 0) best = std::max(best, rate);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(out);
    cudaFree(in);
    *lane_instr_per_s = best;
    return ERT_OK;
}

int ert_d2h_peak(int device, size_t bytes, double *gb_per_s)
{
    if (!gb_per_s) return fail(ERT_ERR_BADARG, "out is NULL");
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    CU(cudaSetDevice(device));
    bytes = std::max<size_t>(bytes, 1 << 20);
    void *dev = nullptr, *host = nullptr;
    CU(cudaMalloc(&dev, bytes));
    if (cudaMallocHost(&host, bytes) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(dev);
        return fail(ERT_ERR_NOMEM, "out of pinned host memory");
    }
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(a));
        CU(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, 0));
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        if (rep > 0) best = std::max(best, (double)bytes / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFreeHost(host);
    cudaFree(dev);
    *gb_per_s = best;
    return ERT_OK;
}

int ert_l2_flush(int device)
{
    int rc;
    if ((rc = check_device(device)) != ERT_OK) return rc;
    CU(cudaSetDevice(device));
    // one buffer per device for the life of the process, whatever thread calls
    static void *buf[16] = {nullptr};
    static std::mutex buf_mu;
    const size_t bytes = (size_t)256 << 20;
    if (device >= 16) return fail(ERT_ERR_BADARG, "device index too large for the flush buffers");
    std::lock_guard<std::mutex> lock(buf_mu);
    if (!buf[device]) CU(cudaMalloc(&buf[device], bytes));
    l2_flush_kernel<<<1184, 256>>>((uint4 *)buf[device], bytes / 16);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    return ERT_OK;
}

}  // extern "C"
