// Builder of the per-light direction grids.  See light_grid.h.
#include "light_grid.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>

#include "grid_math.h"
#include "host_threads.h"

namespace ert {
namespace {

struct Rect { int32_t sphere; uint8_t face; uint16_t u0, u1, v0, v1; };

}  // namespace

int64_t light_grid_cell(const double d[3], int res)
{
    double ax = std::fabs(d[0]), ay = std::fabs(d[1]), az = std::fabs(d[2]);
    int m = 0;
    double am = ax;
    if (ay > am) { m = 1; am = ay; }
    if (az > am) { m = 2; am = az; }
    int face = 2 * m + (d[m] < 0.0 ? 1 : 0);
    double u = d[(m + 1) % 3] / am, v = d[(m + 2) % 3] / am;
    return ((int64_t)face * res + cell_index(v, res)) * res + cell_index(u, res);
}

// The cell a shadow ray looks in, as the device computes it (same IEEE operations: wf_trace_shadow).
int64_t light_grid_cell_f32(const float d[3], int res)
{
    const float ax = std::fabs(d[0]), ay = std::fabs(d[1]), az = std::fabs(d[2]);
    int m = 0;
    float am = ax;
    if (ay > am) { m = 1; am = ay; }
    if (az > am) { m = 2; am = az; }
    const int face = 2 * m + (d[m] < 0.0f ? 1 : 0);
    const float inv = 1.0f / am;
    const float u = d[(m + 1) % 3] * inv, v = d[(m + 2) % 3] * inv;
    const float half = 0.5f * (float)res;
    int iu = (int)std::floor((u + 1.0f) * half), iv = (int)std::floor((v + 1.0f) * half);
    iu = std::min(std::max(iu, 0), res - 1);
    iv = std::min(std::max(iv, 0), res - 1);
    return ((int64_t)face * res + iv) * res + iu;
}

bool build_light_grid(const double *centers, const double *radii, const float *filter, int64_t n,
                      const double light[3], int res, LightGrid &out)
{
    out.res = res;
    out.always.clear();
    const size_t n_cells = (size_t)6 * res * res;
    out.cell_off.assign(n_cells + 1, 0);

    // pass 1: the cell rectangle of every (sphere, face) pair, in parallel over sphere ranges
    unsigned n_thr = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (n < 20000) n_thr = 1;
    std::vector<std::vector<Rect>> rects(n_thr);
    std::vector<std::vector<int32_t>> always(n_thr);
    auto work = [&](unsigned t) {
        int64_t i0 = n * t / n_thr, i1 = n * (t + 1) / n_thr;
        auto &rv = rects[t];
        rv.reserve((size_t)(i1 - i0) * 3 / 2);
        for (int64_t i = i0; i < i1; i++) {
            LightRect lr[6];
            const int nr = light_rects(&centers[3 * i], radii[i], light, res, lr);
            if (nr < 0) { always[t].push_back((int32_t)i); continue; }
            for (int j = 0; j < nr; j++) {
                Rect q;
                q.sphere = (int32_t)i;
                q.face = (uint8_t)lr[j].face;
                q.u0 = (uint16_t)lr[j].u0; q.u1 = (uint16_t)lr[j].u1;
                q.v0 = (uint16_t)lr[j].v0; q.v1 = (uint16_t)lr[j].v1;
                rv.push_back(q);
            }
        }
    };
    parallel_threads(n_thr, work);
    for (auto &v : always) out.always.insert(out.always.end(), v.begin(), v.end());

    // pass 2: counting sort of (cell, sphere) pairs
    for (auto &rv : rects)
        for (const Rect &q : rv)
            for (int v = q.v0; v <= q.v1; v++) {
                uint32_t *row = &out.cell_off[((size_t)q.face * res + v) * res];
                for (int u = q.u0; u <= q.u1; u++) row[u]++;
            }
    uint64_t total = 0;
    for (size_t k = 0; k < n_cells; k++) total += out.cell_off[k];
    if (total > kLightGridMaxEntries) {
        // many spheres close to the light: the grid would cost more memory than it saves walks (and its 32-bit
        // offsets would wrap past 2^32); this light's shadow rays walk the BVH instead
        out = LightGrid{};
        return false;
    }
    total = 0;
    for (size_t k = 0; k < n_cells; k++) { uint32_t c = out.cell_off[k]; out.cell_off[k] = (uint32_t)total; total += c; }
    out.cell_off[n_cells] = (uint32_t)total;
    out.entries.assign((size_t)total, LightGridEntry{0, 0.f});
    std::vector<uint32_t> cursor(out.cell_off.begin(), out.cell_off.end() - 1);
    for (auto &rv : rects)
        for (const Rect &q : rv) {
            double c[3] = {centers[3 * (size_t)q.sphere] - light[0], centers[3 * (size_t)q.sphere + 1] - light[1],
                           centers[3 * (size_t)q.sphere + 2] - light[2]};
            const float dmin = light_dmin(c, radii[q.sphere]);
            for (int v = q.v0; v <= q.v1; v++)
                for (int u = q.u0; u <= q.u1; u++) {
                    size_t cell = ((size_t)q.face * res + v) * res + u;
                    out.entries[cursor[cell]++] = LightGridEntry{q.sphere, dmin};
                }
        }
    // nearest first inside every cell (ties by sphere index keep the order deterministic)
    auto sort_range = [&](size_t k0, size_t k1) {
        for (size_t k = k0; k < k1; k++) {
            auto b = out.entries.begin() + out.cell_off[k], e = out.entries.begin() + out.cell_off[k + 1];
            if (e - b > 1)
                std::sort(b, e, [](const LightGridEntry &x, const LightGridEntry &y) {
                    return x.dmin < y.dmin || (x.dmin == y.dmin && x.sphere < y.sphere);
                });
        }
    };
    parallel_threads(n_thr, [&](unsigned t) { sort_range(n_cells * t / n_thr, n_cells * (t + 1) / n_thr); });
    out.fs.resize((size_t)total * 4);
    for (size_t e = 0; e < (size_t)total; e++) memcpy(&out.fs[4 * e], filter + 4 * (size_t)out.entries[e].sphere, 16);
    return true;
}

void pack_light_grid(const LightGrid &G, std::vector<LightGridCand> &cand, std::vector<LightGridCand> &head)
{
    cand.resize(G.entries.size());
    for (size_t e = 0; e < cand.size(); e++) {
        LightGridCand &c = cand[e];
        c.cx = G.fs[4 * e]; c.cy = G.fs[4 * e + 1]; c.cz = G.fs[4 * e + 2]; c.R = G.fs[4 * e + 3];
        c.sphere = G.entries[e].sphere; c.dmin = G.entries[e].dmin; c.pad[0] = c.pad[1] = 0;
    }
    // per-cell heads: the nearest candidate inline, the rest by range
    const size_t n_cells = G.cell_off.empty() ? 0 : G.cell_off.size() - 1;
    head.resize(n_cells);
    for (size_t c = 0; c < n_cells; c++) {
        const uint32_t e0 = G.cell_off[c], e1 = G.cell_off[c + 1];
        LightGridCand &hd = head[c];
        if (e0 < e1) {
            hd = cand[e0];
            hd.pad[0] = (int)(e0 + 1); hd.pad[1] = (int)e1;
        } else {
            hd.cx = hd.cy = hd.cz = 0.f; hd.R = -3.0e38f; hd.sphere = -1; hd.dmin = INFINITY;
            hd.pad[0] = hd.pad[1] = 0;
        }
    }
}

}  // namespace ert
