// Test-only C shim around the host grid builders (eraytracer_b200/csrc/cell_grid.cpp, light_grid.cpp): the cell grid
// and the direction grids of a sphere table {cx, cy, cz, r}, with the filter spheres and abs_max made as flatten()
// makes them.  tests/test_grid_build_host.py pins their bytes; shim.cu adds the device builders next to them.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "../../eraytracer_b200/csrc/cell_grid.h"
#include "../../eraytracer_b200/csrc/light_grid.h"
#include "../../eraytracer_b200/csrc/scene_math.h"

using namespace ert;

namespace {
struct Spheres {
    std::vector<double> centers, radii;
    std::vector<float> filter;
    float abs_max = 0;
    Spheres(const double *sph, long long n) : centers((size_t)n * 3), radii((size_t)n), filter((size_t)n * 4)
    {
        for (long long k = 0; k < n; k++) {
            const double *s = sph + 4 * k;
            float pad_c, eta_c;
            make_filter_sphere(s, s[3], &filter[(size_t)k * 4], pad_c, eta_c);
            for (int a = 0; a < 3; a++) {
                centers[(size_t)k * 3 + a] = s[a];
                abs_max = std::max(abs_max, f_round_up(std::fabs(s[a]) + std::fabs(s[3])));
            }
            radii[(size_t)k] = s[3];
        }
    }
};
}  // namespace

extern "C" {

void gh_filter(const double *sph, long long n, float *filter_out, float *abs_max_out)
{
    Spheres S(sph, n);
    memcpy(filter_out, S.filter.data(), S.filter.size() * sizeof(float));
    *abs_max_out = S.abs_max;
}

void *gh_cell(const double *sph, long long n, double density)
{
    Spheres S(sph, n);
    CellGrid *g = new CellGrid();
    build_cell_grid(S.centers.data(), S.radii.data(), S.filter.data(), n, S.abs_max, density, *g);
    return g;
}
void gh_cell_free(void *p) { delete (CellGrid *)p; }
int gh_cell_enabled(void *p) { return ((CellGrid *)p)->enabled ? 1 : 0; }
// res[3], lo[3], hi[3], {cs, inv_cs, eps}
void gh_cell_geometry(void *p, int *res, float *lo, float *hi, float *cs)
{
    const CellGrid &g = *(CellGrid *)p;
    for (int a = 0; a < 3; a++) { res[a] = g.res[a]; lo[a] = g.lo[a]; hi[a] = g.hi[a]; }
    cs[0] = g.cs; cs[1] = g.inv_cs; cs[2] = g.eps;
}
long long gh_cell_n_blocks(void *p) { return (long long)((CellGrid *)p)->blocks.size(); }
long long gh_cell_n_over(void *p) { return (long long)((CellGrid *)p)->over_sph.size(); }
long long gh_cell_n_big(void *p) { return (long long)((CellGrid *)p)->big.size(); }
const void *gh_cell_blocks(void *p) { return ((CellGrid *)p)->blocks.data(); }
const void *gh_cell_over_filter(void *p) { return ((CellGrid *)p)->over_filter.data(); }
const void *gh_cell_over_sph(void *p) { return ((CellGrid *)p)->over_sph.data(); }
const void *gh_cell_big(void *p) { return ((CellGrid *)p)->big.data(); }

void *gh_light(const double *sph, long long n, const double *light, int res)
{
    Spheres S(sph, n);
    LightGrid *g = new LightGrid();
    if (!build_light_grid(S.centers.data(), S.radii.data(), S.filter.data(), n, light, res, *g)) { delete g; return nullptr; }
    return g;
}
void gh_light_free(void *p) { delete (LightGrid *)p; }
long long gh_light_n_cells(void *p) { return (long long)((LightGrid *)p)->cell_off.size() - 1; }
long long gh_light_n_entries(void *p) { return (long long)((LightGrid *)p)->entries.size(); }
long long gh_light_n_always(void *p) { return (long long)((LightGrid *)p)->always.size(); }
const void *gh_light_cell_off(void *p) { return ((LightGrid *)p)->cell_off.data(); }
const void *gh_light_entries(void *p) { return ((LightGrid *)p)->entries.data(); }
const void *gh_light_fs(void *p) { return ((LightGrid *)p)->fs.data(); }
const void *gh_light_always(void *p) { return ((LightGrid *)p)->always.data(); }
// the layout the shadow kernels walk (pack_light_grid): cand [n_entries], head [n_cells], 32 bytes each
void gh_light_packed(void *p, void *cand_out, void *head_out)
{
    std::vector<LightGridCand> cand, head;
    pack_light_grid(*(LightGrid *)p, cand, head);
    memcpy(cand_out, cand.data(), cand.size() * sizeof(LightGridCand));
    memcpy(head_out, head.data(), head.size() * sizeof(LightGridCand));
}
long long gh_light_cell(const double *d, int res) { return light_grid_cell(d, res); }
long long gh_light_cell_f32(const float *d, int res) { return light_grid_cell_f32(d, res); }

}
