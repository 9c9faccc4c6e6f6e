// Device builders of the cell grid and of the direction grids (ert_scene_update with ERT_UPDATE_REBUILD_GRIDS).
//
// After an update the spheres, their filter spheres and the scene constants are current on the device, so the grids
// that hold copies of them are built there too, from sph_exact / sph_filter.  The builders produce the bytes the host
// builders (cell_grid.cpp, light_grid.cpp) produce from the same tables: the per-element arithmetic is the shared code
// of grid_math.h, every list is put in the host's order (spheres ascending inside a cell, (dmin, sphere) ascending
// inside a direction cell, the big and always lists in sphere order), and every "no grid" decision is taken on the
// totals the host's monotone incremental checks end with.  Counting, scans, fills and sorts are plain kernels: no
// CUB, no Thrust.  One read-back of a few scalars per grid sizes the output arrays.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>

#include "cell_grid.h"
#include "grid_math.h"
#include "light_grid.h"

namespace ert {

constexpr int kGbThreads = 256;
constexpr int kGbScanThreads = 1024;
constexpr int kGbScanTile = 4 * kGbScanThreads;     // elements per block of the scan

// A device array that keeps its allocation across builds and grows only when asked for more (a cudaFree in every
// update would synchronise the device).
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes)
    {
        if (bytes < 16) bytes = 16;
        if (bytes <= cap) return cudaSuccess;
        if (p) {
            cudaError_t e = cudaFree(p);
            p = nullptr;
            cap = 0;
            if (e != cudaSuccess) return e;
        }
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = bytes;
        return cudaSuccess;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return (T *)p; }
};

// Temporary arrays of the builders, shared by every grid of a scene (the builds run one after another on one stream).
struct GridScratch {
    DevBuf count, cur, over, tmp, flags, scan, rects, dmin, scalars;
    void release()
    {
        for (DevBuf *b : {&count, &cur, &over, &tmp, &flags, &scan, &rects, &dmin, &scalars}) b->release();
    }
};

// A cell grid on the device, in the layout of CellGrid::blocks / over_filter / over_sph / big.
struct CellGridDevOut {
    DevBuf blocks, over_filter, over_sph, big;
    bool enabled = false;
    CellGridGeom geo;
    int n_big = 0;
    size_t n_over = 0;       // entries of over_* (the trailing group included)
    void release()
    {
        for (DevBuf *b : {&blocks, &over_filter, &over_sph, &big}) b->release();
    }
};

// A direction grid on the device: cell_off, cand, head and always of LightGridDev.
struct LightGridDevOut {
    DevBuf cell_off, cand, head, always;
    bool ok = false;
    int res = 0, n_always = 0;
    size_t n_entries = 0;
    void release()
    {
        for (DevBuf *b : {&cell_off, &cand, &head, &always}) b->release();
    }
};

struct GridScalars {
    unsigned long long refs, n_big, max_cnt, run, n_over;   // cell grid
    unsigned long long entries, n_always;                   // direction grid
    unsigned n_long;                                        // direction cells sorted by gb_light_sort_long
};

// ---- exclusive scan of unsigned words ------------------------------------------------------------------------------

// Scans every tile of kGbScanTile words in place and writes each tile's total to sums[tile].
__global__ void __launch_bounds__(kGbScanThreads) gb_scan_tiles(unsigned *data, size_t n, unsigned *sums)
{
    __shared__ unsigned warp_off[32];
    const size_t base = (size_t)blockIdx.x * kGbScanTile + (size_t)threadIdx.x * 4;
    unsigned v[4], s = 0;
    for (int j = 0; j < 4; j++) {
        v[j] = base + j < n ? data[base + j] : 0u;
        s += v[j];
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned x = s;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_off[w] = x;
    __syncthreads();
    if (w == 0) {
        const unsigned t = warp_off[lane];
        unsigned z = t;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, z, o);
            if (lane >= o) z += y;
        }
        warp_off[lane] = z - t;
        if (lane == 31) sums[blockIdx.x] = z;
    }
    __syncthreads();
    unsigned run = warp_off[w] + x - s;
    for (int j = 0; j < 4; j++) {
        if (base + j < n) data[base + j] = run;
        run += v[j];
    }
}

__global__ void __launch_bounds__(kGbThreads) gb_scan_add(unsigned *data, size_t n, const unsigned *sums)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) data[i] += sums[i / kGbScanTile];
}

// words of scratch scan_u32 needs for n elements
inline size_t scan_scratch_words(size_t n)
{
    size_t w = 0;
    do {
        n = (n + kGbScanTile - 1) / kGbScanTile;
        w += n;
    } while (n > 1);
    return w;
}

// Exclusive scan of data[0 .. n) in place (totals below 2^32).  A trailing zero element receives the total.
inline void scan_u32(unsigned *data, size_t n, unsigned *scratch, cudaStream_t st)
{
    const size_t nb = (n + kGbScanTile - 1) / kGbScanTile;
    gb_scan_tiles<<<(unsigned)nb, kGbScanThreads, 0, st>>>(data, n, scratch);
    if (nb > 1) {
        scan_u32(scratch, nb, scratch + nb, st);
        gb_scan_add<<<(unsigned)((n + kGbThreads - 1) / kGbThreads), kGbThreads, 0, st>>>(data, n, scratch);
    }
}

// out[scan[k]] = k for every k < n with scan[k + 1] != scan[k]: the flagged indices in ascending order.
__global__ void __launch_bounds__(kGbThreads) gb_compact(const unsigned *scan, int n, int *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n && scan[k + 1] != scan[k]) out[scan[k]] = k;
}

__device__ inline unsigned long long gb_warp_sum(unsigned long long v)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- cell grid -----------------------------------------------------------------------------------------------------

__device__ inline void gb_sphere_range(const CellGridGeom &g, const double4 &s, int i0[3], int i1[3])
{
    const double c[3] = {s.x, s.y, s.z};
    const double r = fabs(s.w);
    for (int a = 0; a < 3; a++) cell_range(g.lo, g.cs, g.eps, g.res, a, c[a] - r, c[a] + r, i0[a], i1[a]);
}

// Pass 1 of build_cell_grid: per sphere its cell range, its `big` flag, and one count per cell it reaches.
__global__ void __launch_bounds__(kGbThreads) gb_cell_count(const double4 *__restrict__ sph, int n, CellGridGeom g,
                                                            unsigned *count, unsigned *big, GridScalars *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long refs = 0, nb = 0;
    if (k < n) {
        const double4 s = sph[k];
        const double c[3] = {s.x, s.y, s.z};
        int i0[3], i1[3];
        gb_sphere_range(g, s, i0, i1);
        const uint64_t cells = (uint64_t)(i1[0] - i0[0] + 1) * (uint64_t)(i1[1] - i0[1] + 1) * (uint64_t)(i1[2] - i0[2] + 1);
        const size_t sy = (size_t)g.res[0], sz = (size_t)g.res[0] * (size_t)g.res[1];
        if (cells > (uint64_t)kCellGridBigCells) {
            nb = 1;
        } else {
            for (int z = i0[2]; z <= i1[2]; z++)
                for (int y = i0[1]; y <= i1[1]; y++)
                    for (int x = i0[0]; x <= i1[0]; x++)
                        if (cell_reaches(g.lo, g.cs, g.eps_d, c, s.w, x, y, z)) {
                            atomicAdd(&count[x + y * sy + z * sz], 1u);
                            refs++;
                        }
        }
        big[k] = (unsigned)nb;
    }
    refs = gb_warp_sum(refs);
    nb = gb_warp_sum(nb);
    if ((threadIdx.x & 31) == 0) {
        if (refs) atomicAdd(&out->refs, refs);
        if (nb) atomicAdd(&out->n_big, nb);
    }
}

__device__ inline unsigned gb_over_padded(unsigned cnt)
{
    constexpr unsigned kIn = (unsigned)(kCellGridInline * kCellGridBlocks);
    return cnt > kIn ? (cnt - kIn + kCellGridPad - 1) / kCellGridPad * kCellGridPad : 0u;
}

// Pass 2's totals: the largest count, the padded reference total, and each cell's padded overflow (over[c]).
__global__ void __launch_bounds__(kGbThreads) gb_cell_totals(const unsigned *count, size_t n_cells, unsigned *over,
                                                             GridScalars *out)
{
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned cnt = 0;
    unsigned long long run = 0, ov = 0;
    if (c < n_cells) {
        cnt = count[c];
        run = (cnt + kCellGridPad - 1) / kCellGridPad * kCellGridPad;
        ov = gb_over_padded(cnt);
        over[c] = (unsigned)ov;
    } else if (c == n_cells) {
        over[c] = 0;
    }
    cnt = __reduce_max_sync(0xffffffffu, cnt);
    run = gb_warp_sum(run);
    ov = gb_warp_sum(ov);
    if ((threadIdx.x & 31) == 0) {
        if (cnt) atomicMax(&out->max_cnt, (unsigned long long)cnt);
        if (run) atomicAdd(&out->run, run);
        if (ov) atomicAdd(&out->n_over, ov);
    }
}

// Pass 3: every sphere into the cells it reaches (cur: the cells' first slots, advanced as they fill).
__global__ void __launch_bounds__(kGbThreads) gb_cell_fill(const double4 *__restrict__ sph, int n, CellGridGeom g,
                                                           const unsigned *big, unsigned *cur, unsigned *ref)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || big[k]) return;
    const double4 s = sph[k];
    const double c[3] = {s.x, s.y, s.z};
    int i0[3], i1[3];
    gb_sphere_range(g, s, i0, i1);
    const size_t sy = (size_t)g.res[0], sz = (size_t)g.res[0] * (size_t)g.res[1];
    for (int z = i0[2]; z <= i1[2]; z++)
        for (int y = i0[1]; y <= i1[1]; y++)
            for (int x = i0[0]; x <= i1[0]; x++)
                if (cell_reaches(g.lo, g.cs, g.eps_d, c, s.w, x, y, z)) ref[atomicAdd(&cur[x + y * sy + z * sz], 1u)] = (unsigned)k;
}

__device__ inline uint4 gb_bits(float4 f)
{
    return make_uint4(__float_as_uint(f.x), __float_as_uint(f.y), __float_as_uint(f.z), __float_as_uint(f.w));
}

// One cell: its list sorted by sphere index, then written as pack_cell_blocks writes it (both blocks, padding
// included, and the cell's padded overflow from more[c] on).  Thread n_cells writes the trailing padding group.
__global__ void __launch_bounds__(kGbThreads) gb_cell_write(const unsigned *count, const unsigned *cur,
                                                            const unsigned *more, unsigned *ref,
                                                            const float4 *__restrict__ filter, size_t n_cells,
                                                            uint4 *blocks, float4 *over_filter, int *over_sph,
                                                            size_t n_over)
{
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const float4 pad_f = make_float4(0.f, 0.f, 0.f, -3.0e38f);
    if (c == n_cells) {
        for (int j = 0; j < kCellGridPad; j++) {
            over_filter[n_over - kCellGridPad + j] = pad_f;
            over_sph[n_over - kCellGridPad + j] = -1;
        }
    }
    if (c >= n_cells) return;
    const unsigned cnt = count[c];
    unsigned *l = ref + (cur[c] - cnt);
    for (unsigned i = 1; i < cnt; i++) {            // insertion sort: at most kCellGridMaxCount entries
        const unsigned v = l[i];
        unsigned j = i;
        for (; j > 0 && l[j - 1] > v; j--) l[j] = l[j - 1];
        l[j] = v;
    }
    const unsigned m = more[c];
    for (int b = 0; b < kCellGridBlocks; b++) {
        int sph[kCellGridInline];
        uint4 *o = blocks + (c * kCellGridBlocks + b) * 8;
        for (int i = 0; i < kCellGridInline; i++) {
            const unsigned k = (unsigned)(b * kCellGridInline + i);
            float4 f = pad_f;
            sph[i] = -1;
            if (k < cnt) {
                sph[i] = (int)l[k];
                f = filter[sph[i]];
            }
            o[i] = gb_bits(f);
        }
        o[6] = make_uint4((unsigned)sph[0], (unsigned)sph[1], (unsigned)sph[2], (unsigned)sph[3]);
        o[7] = make_uint4((unsigned)sph[4], (unsigned)sph[5], b == 0 ? cnt : 0u, b == 0 ? m : 0u);
    }
    constexpr unsigned kIn = (unsigned)(kCellGridInline * kCellGridBlocks);
    const unsigned padded = gb_over_padded(cnt);
    for (unsigned k = 0; k < padded; k++) {
        const unsigned e = kIn + k;
        if (e < cnt) {
            over_filter[m + k] = filter[l[e]];
            over_sph[m + k] = (int)l[e];
        } else {
            over_filter[m + k] = pad_f;
            over_sph[m + k] = -1;
        }
    }
}

// The cell grid of the n spheres sph (filter spheres `filter`) whose boxes span the double bounds [lo, hi], as
// build_cell_grid builds it.  out.enabled is false where the host builder gives no grid.
inline cudaError_t build_cell_grid_device(const double4 *sph, const float4 *filter, int n, const double lo[3],
                                          const double hi[3], float abs_max, double density, GridScratch &t,
                                          CellGridDevOut &out, cudaStream_t st)
{
    cudaError_t e;
#define GB_TRY(call)                                 \
    do {                                             \
        if ((e = (call)) != cudaSuccess) return e;   \
    } while (0)
    out.enabled = false;
    out.n_big = 0;
    out.n_over = 0;
    if (!cell_grid_geometry(lo, hi, n, abs_max, density, kCellGridMinSpheres, kCellGridMaxRes, out.geo)) return cudaSuccess;
    const CellGridGeom &g = out.geo;
    const size_t n_cells = (size_t)g.n_cells;
    GB_TRY(t.count.reserve(n_cells * 4));
    GB_TRY(t.over.reserve((n_cells + 1) * 4));
    GB_TRY(t.flags.reserve(((size_t)n + 1) * 4));
    GB_TRY(t.scalars.reserve(sizeof(GridScalars)));
    GB_TRY(cudaMemsetAsync(t.count.p, 0, n_cells * 4, st));
    GB_TRY(cudaMemsetAsync(t.flags.p, 0, ((size_t)n + 1) * 4, st));
    GB_TRY(cudaMemsetAsync(t.scalars.p, 0, sizeof(GridScalars), st));
    GridScalars *sc = t.scalars.as<GridScalars>();
    const unsigned nb_sph = (unsigned)((n + kGbThreads - 1) / kGbThreads);
    const unsigned nb_cell = (unsigned)((n_cells + 1 + kGbThreads - 1) / kGbThreads);
    gb_cell_count<<<nb_sph, kGbThreads, 0, st>>>(sph, n, g, t.count.as<unsigned>(), t.flags.as<unsigned>(), sc);
    gb_cell_totals<<<nb_cell, kGbThreads, 0, st>>>(t.count.as<unsigned>(), n_cells, t.over.as<unsigned>(), sc);
    GB_TRY(cudaGetLastError());
    GridScalars h;
    GB_TRY(cudaMemcpyAsync(&h, sc, sizeof h, cudaMemcpyDeviceToHost, st));
    GB_TRY(cudaStreamSynchronize(st));
    // the host's checks, all monotone in the sphere / cell loops, on their totals
    if (h.n_big > (unsigned long long)kCellGridMaxBig || h.refs >= kCellGridMaxRefs ||
        h.max_cnt > (unsigned long long)kCellGridMaxCount || h.run >= kCellGridMaxRefs)
        return cudaSuccess;
    out.n_big = (int)h.n_big;
    out.n_over = (size_t)h.n_over + kCellGridPad;
    GB_TRY(out.blocks.reserve(n_cells * kCellGridBlocks * sizeof(CellBlock)));
    GB_TRY(out.over_filter.reserve(out.n_over * 16));
    GB_TRY(out.over_sph.reserve(out.n_over * 4));
    GB_TRY(out.big.reserve((size_t)out.n_big * 4));
    GB_TRY(t.cur.reserve((n_cells + 1) * 4));
    GB_TRY(t.tmp.reserve(std::max<size_t>((size_t)h.refs, 1) * 4));
    GB_TRY(t.scan.reserve(scan_scratch_words(std::max<size_t>(n_cells, (size_t)n) + 1) * 4));
    unsigned *cur = t.cur.as<unsigned>(), *scan = t.scan.as<unsigned>();
    GB_TRY(cudaMemcpyAsync(cur, t.count.p, n_cells * 4, cudaMemcpyDeviceToDevice, st));
    GB_TRY(cudaMemsetAsync(cur + n_cells, 0, 4, st));
    scan_u32(cur, n_cells + 1, scan, st);
    scan_u32(t.over.as<unsigned>(), n_cells + 1, scan, st);
    gb_cell_fill<<<nb_sph, kGbThreads, 0, st>>>(sph, n, g, t.flags.as<unsigned>(), cur, t.tmp.as<unsigned>());
    gb_cell_write<<<nb_cell, kGbThreads, 0, st>>>(t.count.as<unsigned>(), cur, t.over.as<unsigned>(), t.tmp.as<unsigned>(),
                                                  filter, n_cells, out.blocks.as<uint4>(), out.over_filter.as<float4>(),
                                                  out.over_sph.as<int>(), out.n_over);
    if (out.n_big > 0) {
        scan_u32(t.flags.as<unsigned>(), (size_t)n + 1, scan, st);
        gb_compact<<<nb_sph, kGbThreads, 0, st>>>(t.flags.as<unsigned>(), n, out.big.as<int>());
    }
    GB_TRY(cudaGetLastError());
    out.enabled = true;
    return cudaSuccess;
}

// ---- direction grids -----------------------------------------------------------------------------------------------

constexpr unsigned kGbNoRect = 0xFFFFFFFFu;

// Per sphere: the always flag, the dmin bound, and its rectangle on each of the six faces (rects[6k + face]:
// u0 | u1 << 16, v0 | v1 << 16; kGbNoRect where it covers none).
__global__ void __launch_bounds__(kGbThreads) gb_light_rects(const double4 *__restrict__ sph, int n, double3 light,
                                                             int res, uint2 *rects, float *dmin, unsigned *always,
                                                             GridScalars *out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long entries = 0, n_always = 0;
    if (k < n) {
        const double4 s = sph[k];
        const double c[3] = {s.x, s.y, s.z}, L[3] = {light.x, light.y, light.z};
        LightRect lr[6];
        const int nr = light_rects(c, s.w, L, res, lr);
        uint2 r6[6];
        for (int f = 0; f < 6; f++) r6[f] = make_uint2(kGbNoRect, kGbNoRect);
        for (int j = 0; j < nr; j++) {
            const LightRect &q = lr[j];
            r6[q.face] = make_uint2((unsigned)q.u0 | ((unsigned)q.u1 << 16), (unsigned)q.v0 | ((unsigned)q.v1 << 16));
            entries += (unsigned long long)(q.u1 - q.u0 + 1) * (unsigned long long)(q.v1 - q.v0 + 1);
        }
        for (int f = 0; f < 6; f++) rects[(size_t)k * 6 + f] = r6[f];
        n_always = nr < 0 ? 1 : 0;
        always[k] = (unsigned)n_always;
        float dm = 0.f;
        if (nr >= 0) {
            const double cl[3] = {c[0] - L[0], c[1] - L[1], c[2] - L[2]};
            dm = light_dmin(cl, s.w);
        }
        dmin[k] = dm;
    }
    entries = gb_warp_sum(entries);
    n_always = gb_warp_sum(n_always);
    if ((threadIdx.x & 31) == 0) {
        if (entries) atomicAdd(&out->entries, entries);
        if (n_always) atomicAdd(&out->n_always, n_always);
    }
}

// order-preserving key of a float (dmin is never NaN: only spheres with d2 > r'^2 get one)
__device__ inline unsigned gb_fkey(float x)
{
    const unsigned b = __float_as_uint(x);
    return (b >> 31) ? ~b : (b | 0x80000000u);
}

// One warp per sphere, its lanes spread over the cells of its rectangles (a sphere near the light covers whole
// faces).  FILL false: one count per cell; FILL true: the entry key (dmin, sphere) into the cell's next slot.
template <bool FILL>
__global__ void __launch_bounds__(kGbThreads) gb_light_cells(const uint2 *__restrict__ rects,
                                                             const float *__restrict__ dmin, int n, int res,
                                                             unsigned *cnt, unsigned long long *keys)
{
    const size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= (size_t)n) return;
    const int k = (int)w;
    unsigned long long key = 0;
    if (FILL) key = ((unsigned long long)gb_fkey(dmin[k]) << 32) | (unsigned)k;
    for (int f = 0; f < 6; f++) {
        const uint2 r = rects[(size_t)k * 6 + f];
        if (r.x == kGbNoRect) continue;
        const int u0 = (int)(r.x & 0xFFFFu), u1 = (int)(r.x >> 16), v0 = (int)(r.y & 0xFFFFu), v1 = (int)(r.y >> 16);
        const int wu = u1 - u0 + 1, area = wu * (v1 - v0 + 1);
        for (int i = lane; i < area; i += 32) {
            const size_t cell = ((size_t)f * res + (size_t)(v0 + i / wu)) * res + (size_t)(u0 + i % wu);
            if (FILL)
                keys[atomicAdd(&cnt[cell], 1u)] = key;
            else
                atomicAdd(&cnt[cell], 1u);
        }
    }
}

__device__ inline void gb_store_cand(LightGridCand *dst, float4 f, int sphere, float dmin, int p0, int p1)
{
    uint4 *o = reinterpret_cast<uint4 *>(dst);
    o[0] = gb_bits(f);
    o[1] = make_uint4((unsigned)sphere, __float_as_uint(dmin), (unsigned)p0, (unsigned)p1);
}

// An entry of a direction cell at its place `rank` in the (dmin, sphere) order; the nearest one also goes to head with
// the range of the others.
__device__ inline void gb_put_entry(unsigned long long key, unsigned e0, unsigned len, unsigned rank, size_t c,
                                    const float *__restrict__ dmin, const float4 *__restrict__ filter,
                                    LightGridCand *cand, LightGridCand *head)
{
    const int sphere = (int)(unsigned)(key & 0xFFFFFFFFull);
    const float4 f = filter[sphere];
    const float dm = dmin[sphere];
    gb_store_cand(&cand[e0 + rank], f, sphere, dm, 0, 0);
    if (rank == 0) gb_store_cand(&head[c], f, sphere, dm, (int)(e0 + 1), (int)(e0 + len));
}

constexpr unsigned kGbLongCell = 512;      // longer direction cells are sorted by a block (gb_light_sort_long)
constexpr int kGbSortThreads = 1024;
constexpr int kGbLongBlocks = 256;         // blocks of gb_light_sort_long, each taking long cells in turn

// One warp per cell: the cell's entries ranked by key (unique: a sphere is listed once per cell), which is the host's
// (dmin, sphere) order.  Cells longer than kGbLongCell go to the list `long_cells` instead.
__global__ void __launch_bounds__(kGbThreads) gb_light_sort(const unsigned *__restrict__ cell_off,
                                                            const unsigned long long *__restrict__ keys,
                                                            const float *__restrict__ dmin,
                                                            const float4 *__restrict__ filter, size_t n_cells,
                                                            LightGridCand *cand, LightGridCand *head,
                                                            unsigned *long_cells, GridScalars *sc)
{
    const size_t c = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= n_cells) return;
    const unsigned e0 = cell_off[c], len = cell_off[c + 1] - e0;
    if (len == 0) {
        if (lane == 0) gb_store_cand(&head[c], make_float4(0.f, 0.f, 0.f, -3.0e38f), -1, INFINITY, 0, 0);
        return;
    }
    if (len > kGbLongCell) {
        if (lane == 0) long_cells[atomicAdd(&sc->n_long, 1u)] = (unsigned)c;
        return;
    }
    const unsigned long long *kc = keys + e0;
    for (unsigned bi = 0; bi < len; bi += 32) {
        const unsigned i = bi + lane;
        const unsigned long long mine = i < len ? kc[i] : ~0ull;
        unsigned rank = 0;
        for (unsigned bj = 0; bj < len; bj += 32) {
            const unsigned long long other = bj + lane < len ? kc[bj + lane] : ~0ull;
            for (int t = 0; t < 32; t++) rank += __shfl_sync(0xffffffffu, other, t) < mine ? 1u : 0u;
        }
        if (i < len) gb_put_entry(mine, e0, len, rank, c, dmin, filter, cand, head);
    }
}

// The long direction cells (a light far from a crowd of spheres sees most of them in a few cells): one block per cell,
// a stable LSD radix sort of its 64-bit keys, 8 bits per pass, between keys and alt (same offsets); the block's
// tiles of kGbSortThreads keys are ranked per digit with __match_any_sync and per-warp counts.
__global__ void __launch_bounds__(kGbSortThreads, 1) gb_light_sort_long(const unsigned *__restrict__ cell_off,
                                                                     unsigned long long *keys, unsigned long long *alt,
                                                                     const unsigned *__restrict__ long_cells,
                                                                     const GridScalars *sc,
                                                                     const float *__restrict__ dmin,
                                                                     const float4 *__restrict__ filter,
                                                                     LightGridCand *cand, LightGridCand *head)
{
    __shared__ unsigned base[256], tile[256];
    __shared__ unsigned wcnt[kGbSortThreads / 32][256];
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned n_long = sc->n_long;
    for (unsigned li = blockIdx.x; li < n_long; li += gridDim.x) {
        const unsigned c = long_cells[li];
        const unsigned e0 = cell_off[c], len = cell_off[c + 1] - e0;
        unsigned long long *src = keys + e0, *dst = alt + e0;
        for (int shift = 0; shift < 64; shift += 8) {
            if (tid < 256) tile[tid] = 0;
            __syncthreads();
            for (unsigned i = tid; i < len; i += kGbSortThreads) atomicAdd(&tile[(unsigned)(src[i] >> shift) & 255u], 1u);
            __syncthreads();
            if (tid == 0) {
                unsigned r = 0;
                for (int b = 0; b < 256; b++) { base[b] = r; r += tile[b]; }
            }
            __syncthreads();
            for (unsigned t0 = 0; t0 < len; t0 += kGbSortThreads) {
                const unsigned i = t0 + tid;
                const bool valid = i < len;
                const unsigned long long k = valid ? src[i] : 0ull;
                const unsigned d = valid ? ((unsigned)(k >> shift) & 255u) : 256u;
                for (unsigned j = tid; j < (kGbSortThreads / 32) * 256; j += kGbSortThreads) (&wcnt[0][0])[j] = 0;
                __syncthreads();
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                const unsigned below = __popc(peers & ((1u << lane) - 1u));
                if (valid && below == 0) wcnt[w][d] = __popc(peers);
                __syncthreads();
                if (tid < 256) {
                    unsigned r = 0;
                    for (int ww = 0; ww < kGbSortThreads / 32; ww++) {
                        const unsigned x = wcnt[ww][tid];
                        wcnt[ww][tid] = r;
                        r += x;
                    }
                    tile[tid] = r;
                }
                __syncthreads();
                if (valid) dst[base[d] + wcnt[w][d] + below] = k;
                __syncthreads();
                if (tid < 256) base[tid] += tile[tid];
                __syncthreads();
            }
            unsigned long long *t = src;
            src = dst;
            dst = t;
        }
        for (unsigned i = tid; i < len; i += kGbSortThreads) gb_put_entry(src[i], e0, len, i, c, dmin, filter, cand, head);
        __syncthreads();
    }
}

// The direction grid of `light` at res cells per face edge, as build_light_grid builds it.  out.ok is false (and the
// light gets no grid) when its entries would exceed `budget` (kLightGridMaxEntries for the scene).
inline cudaError_t build_light_grid_device(const double4 *sph, const float4 *filter, int n, const double light[3],
                                           int res, uint64_t budget, GridScratch &t, LightGridDevOut &out,
                                           cudaStream_t st)
{
    cudaError_t e;
    out.ok = false;
    out.res = res;
    out.n_always = 0;
    out.n_entries = 0;
    const size_t n_cells = (size_t)6 * res * res;
    GB_TRY(out.cell_off.reserve((n_cells + 1) * 4));
    GB_TRY(t.rects.reserve((size_t)n * 6 * sizeof(uint2)));
    GB_TRY(t.dmin.reserve((size_t)n * 4));
    GB_TRY(t.flags.reserve(((size_t)n + 1) * 4));
    GB_TRY(t.scalars.reserve(sizeof(GridScalars)));
    unsigned *off = out.cell_off.as<unsigned>();
    GB_TRY(cudaMemsetAsync(off, 0, (n_cells + 1) * 4, st));
    GB_TRY(cudaMemsetAsync(t.flags.as<unsigned>() + n, 0, 4, st));
    GB_TRY(cudaMemsetAsync(t.scalars.p, 0, sizeof(GridScalars), st));
    GridScalars *sc = t.scalars.as<GridScalars>();
    const unsigned nb_sph = (unsigned)((n + kGbThreads - 1) / kGbThreads);
    const unsigned nb_warp_sph = (unsigned)(((size_t)n * 32 + kGbThreads - 1) / kGbThreads);
    gb_light_rects<<<nb_sph, kGbThreads, 0, st>>>(sph, n, make_double3(light[0], light[1], light[2]), res,
                                                  t.rects.as<uint2>(), t.dmin.as<float>(), t.flags.as<unsigned>(), sc);
    gb_light_cells<false><<<nb_warp_sph, kGbThreads, 0, st>>>(t.rects.as<uint2>(), t.dmin.as<float>(), n, res, off, nullptr);
    GB_TRY(cudaGetLastError());
    GridScalars h;
    GB_TRY(cudaMemcpyAsync(&h, sc, sizeof h, cudaMemcpyDeviceToHost, st));
    GB_TRY(cudaStreamSynchronize(st));
    if (h.entries > budget) return cudaSuccess;
    out.n_entries = (size_t)h.entries;
    out.n_always = (int)h.n_always;
    GB_TRY(out.cand.reserve(out.n_entries * sizeof(LightGridCand)));
    GB_TRY(out.head.reserve(n_cells * sizeof(LightGridCand)));
    GB_TRY(out.always.reserve((size_t)out.n_always * 4));
    GB_TRY(t.cur.reserve(n_cells * 4));
    GB_TRY(t.tmp.reserve(std::max<size_t>(out.n_entries, 1) * 16));      // the keys, and the radix sort's copy
    GB_TRY(t.scan.reserve(scan_scratch_words(std::max(n_cells, (size_t)n) + 1) * 4));
    unsigned *scan = t.scan.as<unsigned>();
    scan_u32(off, n_cells + 1, scan, st);
    GB_TRY(cudaMemcpyAsync(t.cur.p, off, n_cells * 4, cudaMemcpyDeviceToDevice, st));
    gb_light_cells<true><<<nb_warp_sph, kGbThreads, 0, st>>>(t.rects.as<uint2>(), t.dmin.as<float>(), n, res,
                                                             t.cur.as<unsigned>(), t.tmp.as<unsigned long long>());
    unsigned long long *keys = t.tmp.as<unsigned long long>();
    gb_light_sort<<<(unsigned)((n_cells * 32 + kGbThreads - 1) / kGbThreads), kGbThreads, 0, st>>>(
        off, keys, t.dmin.as<float>(), filter, n_cells, out.cand.as<LightGridCand>(), out.head.as<LightGridCand>(),
        t.cur.as<unsigned>(), sc);
    gb_light_sort_long<<<kGbLongBlocks, kGbSortThreads, 0, st>>>(off, keys, keys + out.n_entries, t.cur.as<unsigned>(),
                                                                 sc, t.dmin.as<float>(), filter,
                                                                 out.cand.as<LightGridCand>(), out.head.as<LightGridCand>());
    if (out.n_always > 0) {
        scan_u32(t.flags.as<unsigned>(), (size_t)n + 1, scan, st);
        gb_compact<<<nb_sph, kGbThreads, 0, st>>>(t.flags.as<unsigned>(), n, out.always.as<int>());
    }
    GB_TRY(cudaGetLastError());
    out.ok = true;
    return cudaSuccess;
#undef GB_TRY
}

}  // namespace ert
