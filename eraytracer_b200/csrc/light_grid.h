// Per-light direction grid for shadow queries (host-side builder).
//
// shadow_factor/4 (raytracer.erl:256-267) shoots every shadow ray of a light from the SAME
// origin, the light's location.  Seen from there a sphere covers a small patch of directions;
// a cube map of direction cells around the light, each listing the spheres whose patch
// overlaps the cell (nearest first), answers "can anything be in the way of this ray?" with a
// handful of candidates instead of a walk through the sphere BVH.  Like the BVH it only
// prunes: every candidate still goes through the FP32 filter and the literal FP64 test, and a
// sphere the ray can touch is always listed, so the result is the linear scan's.
#pragma once
#include <cstdint>
#include <vector>

namespace ert {

constexpr int kLightGridRes = 128;          // default cells per cube-face edge
constexpr int kMaxLightGrids = 8;           // lights beyond this use the BVH for their shadow rays
constexpr int kLightGridMinSpheres = 64;    // smaller scenes do not need one
constexpr uint64_t kLightGridMaxEntries = 1ull << 27;   // (cell, sphere) entries per light: 4 GB of candidates

struct LightGridEntry {          // 8 bytes next to a 16-byte filter sphere
    int32_t sphere;              // sphere index (list order among spheres)
    float dmin;                  // lower bound of the distance from the light to the sphere
};

// One entry of a light's direction grid on the device: 32 bytes, one 256-bit load.
struct alignas(32) LightGridCand {
    float cx, cy, cz, R;         // filter sphere
    int sphere;                  // sphere index
    float dmin;                  // lower bound of the distance light -> sphere
    int pad[2];
};

struct LightGrid {
    int res = 0;                             // cells per cube-face edge
    std::vector<uint32_t> cell_off;          // [6*res*res + 1] offsets into the entry arrays
    std::vector<float> fs;                   // [n_entries][4] filter spheres {cx, cy, cz, R}
    std::vector<LightGridEntry> entries;     // [n_entries]
    std::vector<int32_t> always;             // spheres that (nearly) contain the light: candidates of every ray
};

// centers: n*3, radii: n, filter: n*4 (the scene's FP32 filter spheres), light: xyz.
// Returns false (and leaves `out` empty) when the grid would need more than kLightGridMaxEntries entries.
bool build_light_grid(const double *centers, const double *radii, const float *filter, int64_t n,
                      const double light[3], int res, LightGrid &out);

// The layout the shadow kernels walk (LightGridDev in ert_device.cuh): every entry with its filter sphere (cand), and
// per cell its nearest candidate (head) with pad[] = the range [first + 1, end) of the others in cand; an empty cell's
// head has R = -3e38, sphere -1, dmin = +inf.
void pack_light_grid(const LightGrid &g, std::vector<LightGridCand> &cand, std::vector<LightGridCand> &head);

// Face/cell of a direction, shared by the builder's tests and (re-stated) by the device code:
// major axis m = first axis of largest |d|, face = 2*m + (d[m] < 0), u = d[(m+1)%3]/|d[m]|,
// v = d[(m+2)%3]/|d[m]|, cell = (face*res + iv)*res + iu with i = floor((x+1)*res/2) clamped.
int64_t light_grid_cell(const double d[3], int res);
// The same in FP32, operation for operation what the shadow kernel does with the filter ray's direction.
int64_t light_grid_cell_f32(const float d[3], int res);

}  // namespace ert
