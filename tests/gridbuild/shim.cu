// Test-only C shim: the device grid builders (eraytracer_b200/csrc/grid_build.cuh) next to the host builders of
// host_shim.cpp, on the same sphere table, so tests/test_gpu_grid_build.py can compare their bytes.  Built with
// nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false, like the library.
#include "host_shim.cpp"
#include "../../eraytracer_b200/csrc/grid_build.cuh"

namespace {

struct DevCell {
    int enabled = 0;
    CellGridGeom geo;
    std::vector<CellBlock> blocks;
    std::vector<float> over_filter;
    std::vector<int> over_sph, big;
};
struct DevLight {
    int ok = 0;
    std::vector<unsigned> cell_off;
    std::vector<LightGridCand> cand, head;
    std::vector<int> always;
};

// the sphere table and its filter spheres (as flatten / upd_spheres make them) on the device
struct DevSpheres {
    Spheres S;
    double4 *sph = nullptr;
    float4 *filter = nullptr;
    int err = 0;
    DevSpheres(const double *s, long long n) : S(s, n)
    {
        err |= cudaMalloc(&sph, std::max<size_t>((size_t)n, 1) * 32) != cudaSuccess;
        err |= cudaMalloc(&filter, std::max<size_t>((size_t)n, 1) * 16) != cudaSuccess;
        if (!err && n) {
            err |= cudaMemcpy(sph, s, (size_t)n * 32, cudaMemcpyHostToDevice) != cudaSuccess;
            err |= cudaMemcpy(filter, S.filter.data(), (size_t)n * 16, cudaMemcpyHostToDevice) != cudaSuccess;
        }
    }
    ~DevSpheres()
    {
        cudaFree(sph);
        cudaFree(filter);
    }
};

template <typename T>
bool fetch(std::vector<T> &v, const DevBuf &b, size_t count)
{
    v.resize(count);
    return count == 0 || cudaMemcpy(v.data(), b.p, count * sizeof(T), cudaMemcpyDeviceToHost) == cudaSuccess;
}

}  // namespace

extern "C" {

// nullptr on a CUDA error
void *gd_cell(const double *sph, long long n, double density)
{
    DevSpheres D(sph, n);
    if (D.err) return nullptr;
    double lo[3], hi[3];
    sphere_bounds(D.S.centers.data(), D.S.radii.data(), n, lo, hi);
    GridScratch t;
    CellGridDevOut out;
    DevCell *c = new DevCell();
    bool ok = build_cell_grid_device(D.sph, D.filter, (int)n, lo, hi, D.S.abs_max, density, t, out, 0) == cudaSuccess &&
              cudaDeviceSynchronize() == cudaSuccess;
    if (ok && out.enabled) {
        c->enabled = 1;
        c->geo = out.geo;
        ok = fetch(c->blocks, out.blocks, (size_t)out.geo.n_cells * kCellGridBlocks) &&
             fetch(c->over_filter, out.over_filter, out.n_over * 4) && fetch(c->over_sph, out.over_sph, out.n_over) &&
             fetch(c->big, out.big, (size_t)out.n_big);
    }
    t.release();
    out.release();
    if (!ok) { delete c; return nullptr; }
    return c;
}
void gd_cell_free(void *p) { delete (DevCell *)p; }
int gd_cell_enabled(void *p) { return ((DevCell *)p)->enabled; }
void gd_cell_geometry(void *p, int *res, float *lo, float *hi, float *cs)
{
    const CellGridGeom &g = ((DevCell *)p)->geo;
    for (int a = 0; a < 3; a++) { res[a] = g.res[a]; lo[a] = g.lo[a]; hi[a] = g.hi[a]; }
    cs[0] = g.cs; cs[1] = g.inv_cs; cs[2] = g.eps;
}
long long gd_cell_n_blocks(void *p) { return (long long)((DevCell *)p)->blocks.size(); }
long long gd_cell_n_over(void *p) { return (long long)((DevCell *)p)->over_sph.size(); }
long long gd_cell_n_big(void *p) { return (long long)((DevCell *)p)->big.size(); }
const void *gd_cell_blocks(void *p) { return ((DevCell *)p)->blocks.data(); }
const void *gd_cell_over_filter(void *p) { return ((DevCell *)p)->over_filter.data(); }
const void *gd_cell_over_sph(void *p) { return ((DevCell *)p)->over_sph.data(); }
const void *gd_cell_big(void *p) { return ((DevCell *)p)->big.data(); }

// budget: the largest entry count the light may have (the library uses kLightGridMaxEntries); nullptr on a CUDA error
void *gd_light(const double *sph, long long n, const double *light, int res, unsigned long long budget)
{
    DevSpheres D(sph, n);
    if (D.err) return nullptr;
    GridScratch t;
    LightGridDevOut out;
    DevLight *g = new DevLight();
    bool ok = build_light_grid_device(D.sph, D.filter, (int)n, light, res, budget, t, out, 0) == cudaSuccess &&
              cudaDeviceSynchronize() == cudaSuccess;
    if (ok && out.ok) {
        const size_t n_cells = (size_t)6 * res * res;
        g->ok = 1;
        ok = fetch(g->cell_off, out.cell_off, n_cells + 1) && fetch(g->cand, out.cand, out.n_entries) &&
             fetch(g->head, out.head, n_cells) && fetch(g->always, out.always, (size_t)out.n_always);
    }
    t.release();
    out.release();
    if (!ok) { delete g; return nullptr; }
    return g;
}
void gd_light_free(void *p) { delete (DevLight *)p; }
int gd_light_ok(void *p) { return ((DevLight *)p)->ok; }
long long gd_light_n_entries(void *p) { return (long long)((DevLight *)p)->cand.size(); }
long long gd_light_n_always(void *p) { return (long long)((DevLight *)p)->always.size(); }
const void *gd_light_cell_off(void *p) { return ((DevLight *)p)->cell_off.data(); }
const void *gd_light_cand(void *p) { return ((DevLight *)p)->cand.data(); }
const void *gd_light_head(void *p) { return ((DevLight *)p)->head.data(); }
const void *gd_light_always(void *p) { return ((DevLight *)p)->always.data(); }

}
