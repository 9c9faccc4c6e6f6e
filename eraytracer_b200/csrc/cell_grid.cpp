// Builder of the uniform cell grid over the spheres.  See cell_grid.h.
#include "cell_grid.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>

#include "grid_math.h"

namespace ert {

void cell_grid_range(const CellGrid &g, int axis, double a, double b, int &i0, int &i1)
{
    cell_range(g.lo, g.cs, g.eps, g.res, axis, a, b, i0, i1);
}

void cell_grid_set_geometry(CellGrid &g, const CellGridGeom &geo)
{
    for (int a = 0; a < 3; a++) { g.res[a] = geo.res[a]; g.lo[a] = geo.lo[a]; g.hi[a] = geo.hi[a]; }
    g.cs = geo.cs; g.inv_cs = geo.inv_cs; g.eps = geo.eps;
}

void sphere_bounds(const double *centers, const double *radii, int64_t n, double lo[3], double hi[3])
{
    for (int a = 0; a < 3; a++) { lo[a] = DBL_MAX; hi[a] = -DBL_MAX; }
    for (int64_t k = 0; k < n; k++) {
        const double r = std::fabs(radii[k]);
        for (int a = 0; a < 3; a++) {
            lo[a] = std::min(lo[a], centers[k * 3 + a] - r);
            hi[a] = std::max(hi[a], centers[k * 3 + a] + r);
        }
    }
}

void build_cell_grid(const double *centers, const double *radii, const float *filter, int64_t n, float abs_max,
                     double density, CellGrid &out)
{
    out = CellGrid();
    if (n < kCellGridMinSpheres || !(density > 0) || !std::isfinite(abs_max) || abs_max > 1e6f) return;
    double lo[3], hi[3];
    sphere_bounds(centers, radii, n, lo, hi);
    CellGridGeom geo;
    const bool ok = cell_grid_geometry(lo, hi, n, abs_max, density, kCellGridMinSpheres, kCellGridMaxRes, geo);
    cell_grid_set_geometry(out, geo);
    if (!ok) return;
    const size_t n_cells = (size_t)geo.n_cells;
    const double eps = geo.eps_d;

    // pass 1: counts
    std::vector<uint32_t> count(n_cells, 0);
    std::vector<uint8_t> is_big((size_t)n, 0);
    uint64_t refs = 0;
    auto range = [&](int64_t k, int (&i0)[3], int (&i1)[3]) {
        const double r = std::fabs(radii[k]);
        for (int a = 0; a < 3; a++) cell_grid_range(out, a, centers[k * 3 + a] - r, centers[k * 3 + a] + r, i0[a], i1[a]);
    };
    const size_t sx = 1, sy = (size_t)out.res[0], sz = (size_t)out.res[0] * (size_t)out.res[1];
    auto reaches = [&](int64_t k, int x, int y, int z) {
        return cell_reaches(out.lo, out.cs, eps, &centers[k * 3], radii[k], x, y, z);
    };
    for (int64_t k = 0; k < n; k++) {
        int i0[3], i1[3];
        range(k, i0, i1);
        uint64_t cells = (uint64_t)(i1[0] - i0[0] + 1) * (uint64_t)(i1[1] - i0[1] + 1) * (uint64_t)(i1[2] - i0[2] + 1);
        if (cells > (uint64_t)kCellGridBigCells) {
            is_big[(size_t)k] = 1;
            out.big.push_back((int32_t)k);
            if ((int)out.big.size() > kCellGridMaxBig) { out = CellGrid(); return; }
            continue;
        }
        for (int z = i0[2]; z <= i1[2]; z++)
            for (int y = i0[1]; y <= i1[1]; y++)
                for (int x = i0[0]; x <= i1[0]; x++)
                    if (reaches(k, x, y, z)) { count[x * sx + y * sy + z * sz]++; refs++; }
        if (refs >= kCellGridMaxRefs) { out = CellGrid(); return; }
    }
    // pass 2: offsets, packed cell words
    out.cells.resize(n_cells);
    std::vector<uint32_t> cursor(n_cells);
    uint32_t run = 0;
    for (size_t c = 0; c < n_cells; c++) {
        if (count[c] > (uint32_t)kCellGridMaxCount) { out = CellGrid(); return; }
        out.cells[c] = (run << 7) | count[c];
        cursor[c] = run;
        // every cell's list is stored in whole groups of kCellGridPad entries: the filter loop of the walk reads
        // a group at a time without looking at the count (the padding is a sphere that never passes)
        run += (count[c] + (uint32_t)kCellGridPad - 1) / (uint32_t)kCellGridPad * (uint32_t)kCellGridPad;
        if (run >= kCellGridMaxRefs) { out = CellGrid(); return; }
    }
    // pass 3: fill, spheres in list order inside a cell
    run += (uint32_t)kCellGridPad;                   // the loop may fetch one group past the last list
    out.ref_filter.assign((size_t)run * 4, 0.f);
    for (size_t k = 0; k < (size_t)run; k++) out.ref_filter[k * 4 + 3] = -3.0e38f;
    out.ref_sph.assign((size_t)run, -1);
    for (int64_t k = 0; k < n; k++) {
        if (is_big[(size_t)k]) continue;
        int i0[3], i1[3];
        range(k, i0, i1);
        for (int z = i0[2]; z <= i1[2]; z++)
            for (int y = i0[1]; y <= i1[1]; y++)
                for (int x = i0[0]; x <= i1[0]; x++) {
                    if (!reaches(k, x, y, z)) continue;
                    uint32_t slot = cursor[x * sx + y * sy + z * sz]++;
                    memcpy(&out.ref_filter[(size_t)slot * 4], &filter[(size_t)k * 4], 16);
                    out.ref_sph[slot] = (int32_t)k;
                }
    }
    out.enabled = true;
    pack_cell_blocks(out);
}

void pack_cell_blocks(CellGrid &g)
{
    const size_t n_cells = g.cells.size();
    constexpr uint32_t kIn = (uint32_t)(kCellGridInline * kCellGridBlocks);
    CellBlock empty;
    for (int k = 0; k < kCellGridInline; k++) {
        empty.f[k][0] = empty.f[k][1] = empty.f[k][2] = 0.f;
        empty.f[k][3] = -3.0e38f;
        empty.sph[k] = -1;
    }
    empty.cnt = 0; empty.more = 0;
    g.blocks.assign(n_cells * kCellGridBlocks, empty);
    auto padded = [](uint32_t cnt) { return cnt > kIn ? ((size_t)(cnt - kIn) + kCellGridPad - 1) / kCellGridPad * kCellGridPad : 0; };
    size_t n_over = 0;
    for (size_t c = 0; c < n_cells; c++) n_over += padded(g.cells[c] & 127u);
    n_over += kCellGridPad;                          // the walk's loop may fetch one group past the last list
    g.over_filter.assign(n_over * 4, 0.f);
    for (size_t k = 0; k < n_over; k++) g.over_filter[k * 4 + 3] = -3.0e38f;
    g.over_sph.assign(n_over, -1);
    size_t run = 0;
    for (size_t c = 0; c < n_cells; c++) {
        const uint32_t cnt = g.cells[c] & 127u, first = g.cells[c] >> 7;
        CellBlock *b = &g.blocks[c * kCellGridBlocks];
        b[0].cnt = cnt;
        b[0].more = (uint32_t)run;
        for (uint32_t k = 0; k < cnt; k++) {
            const size_t slot = (size_t)first + k;
            if (k < kIn) {
                CellBlock &bb = b[k / kCellGridInline];
                memcpy(bb.f[k % kCellGridInline], &g.ref_filter[slot * 4], 16);
                bb.sph[k % kCellGridInline] = g.ref_sph[slot];
            } else {
                const size_t o = run + (k - kIn);
                memcpy(&g.over_filter[o * 4], &g.ref_filter[slot * 4], 16);
                g.over_sph[o] = g.ref_sph[slot];
            }
        }
        run += padded(cnt);
    }
}

}  // namespace ert
