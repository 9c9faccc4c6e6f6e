// Uniform cell grid over the spheres (host-side builder).
//
// nearest_object_intersecting_ray/2 (raytracer.erl:300-346) tests a ray against every object
// of the list.  For scenes of many small spheres a regular grid of cells, each listing the
// spheres whose (slightly inflated) bounding box overlaps it, lets a ray visit only the cells
// it passes through, front to back (3-D DDA), and stop at the first cell that starts behind
// its nearest hit so far.  A cell step costs a third of a BVH node visit and scattered
// reflection rays need a third as many of them, which is why the path rays of the wavefront
// use the grid when the scene has one.  Like the BVH it only prunes: a listed sphere still
// goes through the FP32 filter and the literal FP64 test with the (t, order) comparison of
// erl:319, and every sphere the ray can touch is listed in a cell the walk visits (DESIGN.md
// "Cell grid"), so the result is the linear scan's.
#pragma once
#include <cstdint>
#include <vector>

namespace ert {

constexpr double kCellGridDensity = 0.35;    // default: cells per sphere (ERT_CELL_GRID_DENSITY)
constexpr int kCellGridMinSpheres = 256;     // smaller scenes do not get one
constexpr int kCellGridMaxRes = 1024;        // cells per axis (the walk keeps plane indices as floats)
constexpr int kCellGridMaxCount = 127;       // spheres per cell (7 bits of the packed cell word)
constexpr int kCellGridPad = 4;              // a cell's list is stored in whole groups of this many entries
constexpr int kCellGridInline = 6;           // spheres held in one 128-byte block (what the device walks)
constexpr int kCellGridBlocks = 2;           // blocks per cell: lists of up to 12 spheres need no dependent fetch
constexpr uint32_t kCellGridMaxRefs = 1u << 25;
constexpr int kCellGridBigCells = 512;       // a sphere overlapping more cells than this goes to the `big` list
constexpr int kCellGridMaxBig = 32;          // more of those than this: no grid for the scene

// What the device walks: kCellGridBlocks 128-byte blocks per cell, their address pure arithmetic on the cell id (no
// dependent fetch between the 3-D DDA and the spheres), each holding kCellGridInline filter spheres and their
// indices; a list that fits the first block leaves the second untouched.  Longer lists continue in over_filter /
// over_sph from entry `more` on, in whole groups of kCellGridPad.  `cnt` and `more` are those of the first block.
struct alignas(16) CellBlock {
    float f[kCellGridInline][4];              // filter spheres (padding: R = -3e38, never passes)
    int32_t sph[kCellGridInline];             // sphere indices (padding: -1)
    uint32_t cnt;                             // spheres listed in the cell, inline ones included
    uint32_t more;                            // first overflow entry of this cell
};
static_assert(sizeof(CellBlock) == 128, "one cell is one 128-byte line");

struct CellGrid {
    bool enabled = false;
    int res[3] = {0, 0, 0};
    float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};   // bounds of the grid (outward of every inflated sphere box)
    float cs = 0, inv_cs = 0;                     // edge of a cell
    float eps = 0;                                // inflation of the sphere boxes; rays need 4m <= eps
    std::vector<uint32_t> cells;                  // [rx*ry*rz] (first_ref << 7) | count
    std::vector<float> ref_filter;                // [n_refs][4] filter spheres in cell order (padding: R = -3e38)
    std::vector<int32_t> ref_sph;                 // [n_refs] sphere index (padding: -1)
    std::vector<int32_t> big;                     // spheres tested by every ray
    // the same lists in the layout the device walks (pack_cell_blocks); cells / ref_* above stay on the host
    std::vector<CellBlock> blocks;                // [rx*ry*rz][kCellGridBlocks]
    std::vector<float> over_filter;               // [n_over][4]
    std::vector<int32_t> over_sph;                // [n_over]
};

// Fills blocks / over_* from cells / ref_* (called by build_cell_grid; separate so that the tests can check it).
void pack_cell_blocks(CellGrid &g);

// centers: n*3, radii: n, filter: n*4 (the scene's FP32 filter spheres), abs_max: largest
// |coordinate| of any sphere box.  Leaves out.enabled false when the scene does not suit a grid.
void build_cell_grid(const double *centers, const double *radii, const float *filter, int64_t n, float abs_max,
                     double density, CellGrid &out);

// Cell range [i0, i1] of the interval [a, b] along one axis (shared with the tests).
void cell_grid_range(const CellGrid &g, int axis, double a, double b, int &i0, int &i1);

// The double bounds [min (c - |r|), max (c + |r|)] of the sphere boxes, the input of the grid's geometry
// (cell_grid_geometry in grid_math.h).
void sphere_bounds(const double *centers, const double *radii, int64_t n, double lo[3], double hi[3]);

// Copies res, lo, hi, cs, inv_cs and eps of geo into g.
struct CellGridGeom;
void cell_grid_set_geometry(CellGrid &g, const CellGridGeom &geo);

}  // namespace ert
