// Wavefront form of the eraytracer hot path for large sphere counts (ERT_ACCEL_BVH, ERT_ACCEL_GRID).
//
// The per-pixel recursion of raytracer.erl:186-252 is cut into queues that live in HBM, so
// that every traversal warp is full of live rays of ONE kind:
//
//   bounce b:  wf_trace_path[_refill]  path queue -> nearest hit (erl:300-346) -> hit record (compacted) AND the
//                                      reflection ray of bounce b+1 (erl:219-221), written by the same warp
//              wf_shadow_shade         hit queue x lights -> shadow_factor (erl:256-267: FP32 triage, then the literal
//                                      path for the pairs it leaves open) -> light fold into the pixel (erl:209-252);
//                                      on a second stream, beside the path rays of bounce b+1
//   end:       wf_finalize             colour -> framebuffer (quantisation of erl:678-680 fused)
//
// (wf_emit_hits, wf_bin_*, wf_trace_shadow and wf_shade are the same stages as separate launches: used when the
// hits are binned by location or a light has no direction grid.)
//
// The arithmetic is the megakernel's (ert_device.cuh): FP64 in the literal operation order for
// everything that feeds a decision or a colour, FP32 only in conservative filters and in proofs with explicit
// margins (shadow_blocked).  All forms produce bit-identical frames (tests/test_gpu_parity.py, test_gpu_edges.py,
// test_gpu_cell_grid.py).
#pragma once

#include <limits.h>

#include "ert_device.cuh"

#ifdef ERT_WF_DEBUG
#include <cstdio>
#define WF_ASSERT(cond, ...)                                            \
    do {                                                                \
        if (!(cond)) {                                                  \
            printf("WF_ASSERT %s:%d " #cond " : ", __FILE__, __LINE__); \
            printf(__VA_ARGS__);                                        \
            printf("\n");                                               \
            __trap();                                                   \
        }                                                               \
    } while (0)
#else
#define WF_ASSERT(cond, ...) do { } while (0)
#endif

namespace ert {

// One hit of a path ray, in two records: the shadow stage streams only the 32-byte heads
// (dense, every fetched byte used), the shade stage reads both.
struct alignas(32) HitHead {
    double P[3];                // hit location
    int obj, order;             // object code, list position
};
struct alignas(32) HitTail {
    double N[3];                // normal
    int pid, pad0;              // pixel of the path
    double D[3];                // direction of the ray that hit
    double W;                   // weight of the path up to this hit: product of (lights * reflectivity) of earlier bounces
};
static_assert(sizeof(HitHead) == 32 && sizeof(HitTail) == 64, "hit records are 32 + 64 bytes");

// One ray of the path queue: two 256-bit transactions to write, two to read.
struct alignas(32) PathRec {
    double O[3];                // origin
    double W;                   // weight of the path: product of (lights * reflectivity) of earlier bounces
    double D[3];                // direction
    int pid, pad0;              // pixel of the path
};
static_assert(sizeof(PathRec) == 64, "a path ray is 64 bytes");

// nearest hit of one path ray of the brute-force scan: 16 bytes, one 128-bit compare-and-swap
struct alignas(16) ScanBest {
    double t;
    int order, obj;
};

struct WfBuf {
    int n_pad;                  // pixels of this part padded to whole 8x4 tiles: tiles * 32
    int tiles_x;                // tiles per row of tiles
    double *C;                  // [3][n_pad] colour so far, by pixel
    // path queue of the bounce being traced (read) and of the next one (written by whoever emits the hits): two
    // buffer sets that swap every bounce, so that the next rays exist as soon as their hits do — the reflection
    // (erl:219-221) does not depend on the shadow rays, only the colour does
    PathRec *q;                 // [n_pad] rays of the bounce being traced
    PathRec *nq;                // [n_pad] rays of the next bounce
    double *res_t;              // nearest hit of each path ray: Distance,
    int2 *res_hit;              //   (object code or -1, list position)
    HitHead *hit_head;          // hit queue the shadow and shade stages read
    HitTail *hit_tail;
    HitHead *raw_head;          // hit queue in arrival order (before binning, when hits are binned)
    HitTail *raw_tail;
    unsigned int *r_key;        // cell of each raw hit (Morton order)
    unsigned char *lit;         // [n_lights][n_pad] shadow factor of (light, hit)
    unsigned int *ctr;          // [depth][kWfCtr] queue lengths and work cursors
    unsigned int *hist;         // [kSortCells] cell histogram -> offsets -> scatter cursors
    unsigned int *sums;         // [kSortBlocks] per-block totals of the histogram scan
    // brute-force scan (ert_scan.cuh), allocated for ERT_ACCEL_LINEAR frames only
    ScanBest *sp_best;      // [n_pad] nearest hit of each path ray while candidates fold into it
    double *sp_t;               // [n_pad * lights] Distance of each shadow ray's target
    unsigned char *sp_occ;      // [n_pad * lights] 1: something is nearer than the target (or the target is missed)
};
enum WfCtr : int { WF_NHITS = 0, WF_NNEXT = 1, WF_FETCH_PATH = 2 /* 64-bit */, WF_FETCH_SHADOW = 4 /* 64-bit */, kWfCtr = 8 };
constexpr int kWfThreads = 256;
#ifndef ERT_WF_LDG256
#define ERT_WF_LDG256 1             /* 64-byte BVH nodes fetched as two 256-bit loads */
#endif
#ifndef ERT_WF_MINBLOCKS
#define ERT_WF_MINBLOCKS 4          /* resident blocks per SM the traversal kernels are compiled for */
#endif
#ifndef ERT_SHADE_MINBLOCKS
#define ERT_SHADE_MINBLOCKS 3       /* wf_shade */
#endif
#ifndef ERT_SHADOW_MINBLOCKS
#define ERT_SHADOW_MINBLOCKS 4      /* the shadow kernel */
#endif
#ifndef ERT_GRID_MINBLOCKS
#define ERT_GRID_MINBLOCKS 3        /* the path kernels that walk the cell grid: 85 registers without spills beat
                                       64 with (C4 path walks 8.2 vs 9.0 ms) */
#endif
#ifndef ERT_WF_SORT_BITS
#define ERT_WF_SORT_BITS 8
#endif
constexpr int kSortBits = ERT_WF_SORT_BITS;                   // per axis
constexpr int kSortCells = 1 << (3 * kSortBits);              // bins of the counting sort (16 Mi)
constexpr int kSortScanBlock = 4096;                          // bins scanned by one block
constexpr int kSortBlocks = kSortCells / kSortScanBlock;
constexpr int kSortScanBThreads = kSortBlocks < 1024 ? kSortBlocks : 1024;
constexpr int kSortScanBItems = kSortBlocks / kSortScanBThreads;
static_assert(kSortBlocks % 32 == 0 && kSortBlocks <= 8192, "scan phase B is one block");
// ------------------------------------------------------------------ slim ray for the traversal
// Same bounds as FRay (DESIGN.md "Filter bounds"); the slab constants are written so that the
// near/far choice needs no select: with m the absolute margin,
//     ta = lo*inv - (o+m)*inv,  tb = hi*inv - (o-m)*inv,  t_enter = min(ta,tb), t_exit = max(ta,tb)
// pushes the entered plane outward by m and the left plane outward by m for either sign of inv.
struct SRay {
    float ox, oy, oz;
    float dx, dy, dz;
    float ix, iy, iz;
    float klx, kly, klz;
    float khx, khy, khz;
    float theta, bcull, pad2, m4;
};
// The FP64 ray (origin, direction, a = D.D, 1/sqrt(a)) is needed only by the rare literal tests:
// it lives in shared memory, one column per thread, so the walk keeps it out of registers.
struct RaySlot {
    double *p;                                           // &slots[0][threadIdx.x], stride kWfThreads
    __device__ __forceinline__ double get(int k) const { return p[k * kWfThreads]; }
    __device__ __forceinline__ void put(d3 O, d3 D, double, double)
    {
        p[0] = O.x; p[kWfThreads] = O.y; p[2 * kWfThreads] = O.z;
        p[3 * kWfThreads] = D.x; p[4 * kWfThreads] = D.y; p[5 * kWfThreads] = D.z;
    }
    __device__ __forceinline__ d3 O() const { return mk(get(0), get(1), get(2)); }
    __device__ __forceinline__ d3 D() const { return mk(get(3), get(4), get(5)); }
    // a = D.D and 1/sqrt(a) are recomputed where the rare literal tests need them (same expressions
    // as make_sray), which keeps the slot at 48 bytes per thread: shared memory here is L1 lost
    __device__ __forceinline__ double a() const
    {
        const d3 d = D();
        return d.x * d.x + d.y * d.y + d.z * d.z;
    }
    __device__ __forceinline__ double inv_sqrt_a() const
    {
        const double aa = a();
        return (fabs(aa - 1.0) <= 1e-9) ? (1.5 - 0.5 * aa) : 1.0 / sqrt(aa);
    }
};
constexpr int kRaySlotDoubles = 6;
#define ERT_KAPPA 1.00006103515625f   /* 1 + 2^-14 >= (1+2^-16)/(1-2^-16): slab slack as one factor */

// Returns false for a ray beyond the filter's range (kFilterRange, as make_fray); its constants are then left as
// they are, and the callers do not filter with them: a walk decides every sphere with scan_spheres_instead instead,
// and wf_scan passes every sphere through stage 1.  (Its m4 exceeds every cell grid's eps, see grid_begin.)
__device__ __forceinline__ bool make_sray(const DevScene &sc, d3 O, d3 D, SRay &f, double &a_out, double &inv_out)
{
    const double a = D.x * D.x + D.y * D.y + D.z * D.z;
    // 1/sqrt(a): directions are unit vectors up to rounding except after a bounce off an
    // un-normalised plane normal; 1.5 - a/2 is 1/sqrt(a) to 4e-19 relative for |a-1| <= 1e-9
    // (this value only scales the FP32 filter ray and the cull distance, both with 2^-16 slack)
    double inv = (fabs(a - 1.0) <= 1e-9) ? (1.5 - 0.5 * a) : 1.0 / sqrt(a);
    a_out = a;
    inv_out = inv;
    f.ox = (float)O.x; f.oy = (float)O.y; f.oz = (float)O.z;
    double k = inv * ERT_KD;
    f.dx = (float)(D.x * k); f.dy = (float)(D.y * k); f.dz = (float)(D.z * k);
    float eo = 2.0f * fmaxf(fmaxf(fabsf((float)(O.x - (double)f.ox)), fabsf((float)(O.y - (double)f.oy))),
                            fabsf((float)(O.z - (double)f.oz)));
    eo *= 1.0001f;
    f.theta = 16.0f * sc.r_max * eo + 8.0f * eo * (eo / ERT_U);
    f.bcull = 2.0f * (5.0f * ERT_U * sc.r_max + 2.0f * eo + 2.0f * sc.eta_c_max);
    f.pad2 = 2.0f * (f.theta + sc.pad_c_max) + 1e-30f;
    float oabs = fmaxf(fmaxf(fabsf(f.ox), fabsf(f.oy)), fabsf(f.oz));
    float m = eo + 32.0f * ERT_U * (oabs + sc.abs_max);
    f.m4 = 4.0f * m;
    // approximate reciprocals (2 ulp): a relative error of the slope scales every slab distance
    // of that axis alike and is covered by kappa and the 2^-16 slack of the cull distance
    f.ix = __frcp_rn(clamp_dir(f.dx)); f.iy = __frcp_rn(clamp_dir(f.dy)); f.iz = __frcp_rn(clamp_dir(f.dz));
    f.klx = -(f.ox + m) * f.ix; f.kly = -(f.oy + m) * f.iy; f.klz = -(f.oz + m) * f.iz;
    f.khx = -(f.ox - m) * f.ix; f.khy = -(f.oy - m) * f.iy; f.khz = -(f.oz - m) * f.iz;
    return oabs + sc.abs_max < kFilterRange;                // false for NaN and Inf as well
}

__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void ldg256(const void *p, float (&v)[8])
{
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}

// 6 FFMA + 6 FMNMX + 2 FMNMX3 + FMNMX + FMUL + FMNMX + compare.  `cullk` already carries kappa.
__device__ __forceinline__ bool slab_test(const SRay &f, float lox, float hix, float loy, float hiy, float loz,
                                          float hiz, float cullk, float &tnear)
{
    float ax = __fmaf_rn(lox, f.ix, f.klx), bx = __fmaf_rn(hix, f.ix, f.khx);
    float ay = __fmaf_rn(loy, f.iy, f.kly), by = __fmaf_rn(hiy, f.iy, f.khy);
    float az = __fmaf_rn(loz, f.iz, f.klz), bz = __fmaf_rn(hiz, f.iz, f.khz);
    float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
    float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    tnear = fmaxf(tn, 0.f);
    return tnear <= fminf(tf * ERT_KAPPA, cullk);
}

// reference Distance of the incumbent -> filter-space cull distance (upper bound), kappa included
__device__ __forceinline__ float cullk_from(const SRay &f, double inv_sqrt_a, const Hit &best)
{
    if (best.obj < 0) return __int_as_float(0x7f800000);
    float sf = __double2float_ru(best.t * inv_sqrt_a);
    return (sf + fabsf(sf) * ERT_REL16 + f.m4) * ERT_KAPPA;
}

// One leaf sphere: FP32 filter, then the literal FP64 test on survivors (rare).
template <bool COUNT>
__device__ __forceinline__ void leaf_sphere(const DevScene &sc, const SRay &f, const RaySlot &ray, float4 fs,
                                            const int *__restrict__ slot_sph, int slot, int skip_obj, Hit &best,
                                            float &cullk, Tally<COUNT> &tl)
{
    float b, v;
    TALLY(filter);
    if (!filter_stage1(f, fs, b, v)) return;
    if (!filter_stage2(f, fs, b, v, cullk)) return;
    int sph = __ldg(slot_sph + slot);
    int code = obj_code(OBJ_SPHERE, sph);
    if (code == skip_obj) return;
    double t;
    TALLY(exact_sph);
    if (sphere_exact(ray.O(), ray.D(), ray.a(), ld_sphere(sc.sph_exact + sph), t)) {
        int ord = sc.sph_order[sph];
        if (better(t, ord, best)) {
            best.t = t; best.order = ord; best.obj = code;
            cullk = cullk_from(f, ray.inv_sqrt_a(), best);
        }
    }
}

// ------------------------------------------------------------------ resumable traversal
// The state of one ray's walk.  trav_step() runs inner nodes until the ray holds a leaf,
// processes that leaf and pops (while-while: the lanes of a warp meet again at every leaf).
// Handing new rays to finished lanes in mid-walk (persistent lanes with dynamic fetch) was
// measured and lost: the set-up of a few lanes at a time costs more than the idle lanes do.
// ANY: the search ends at the first improvement of the incumbent (shadow rays).
constexpr int kTravDone = INT_MIN;
template <bool ANY>
struct Trav {
    int node, sp;
    float cullk;
};
// The stack is a separate local array (passed as `stack`): as a member it would drag node, sp and
// cullk into local memory with it wherever the state outlives a loop iteration.

template <bool ANY>
__device__ __forceinline__ void trav_start(Trav<ANY> &tr, int *stack, const SRay &f, double inv_sqrt_a, const Hit &best)
{
    stack[0] = kTravDone;
    tr.sp = 1;
    tr.node = 0;
    tr.cullk = cullk_from(f, inv_sqrt_a, best);
}

// A popped subtree is re-tested against the current cull distance when it is visited.  Tagging stack
// entries with their entry distance to skip them at the pop was measured and cost more (a second
// local-memory array competing with the tree for L1: path walks 18.2 vs 16.3 ms on C4) than the
// 6 % of box tests it saved.  (A triangle incumbent can have t < 0, erl:402-455 has no t >= 0 test:
// then cullk is negative and every box test fails, which is right — no sphere has t < 0.)
template <bool ANY>
__device__ __forceinline__ void trav_pop(Trav<ANY> &tr, const int *stack)
{
    --tr.sp;
    WF_ASSERT(tr.sp >= 0, "sp %d", tr.sp);
    tr.node = stack[tr.sp];
}

// returns true when the search is over
template <bool ANY, bool COUNT>
__device__ __forceinline__ bool trav_step(Trav<ANY> &tr, int *stack, const DevScene &sc, const RaySlot &ray, const SRay &f,
                                          Hit &best, int skip_obj, int seed_obj, Tally<COUNT> &tl)
{
    while (tr.node >= 0) {
        WF_ASSERT(tr.node < sc.n_nodes, "node %d of %d sp %d", tr.node, sc.n_nodes, tr.sp);
        // one 64-byte node = two 256-bit loads (LDG.E.256): half the L1 wavefronts of four 128-bit ones
        float n0[8], n1[8];
#if ERT_WF_LDG256
        ldg256(sc.nodes + tr.node, n0);
        ldg256(reinterpret_cast<const char *>(sc.nodes + tr.node) + 32, n1);
#else
        {
            const float4 *np4 = reinterpret_cast<const float4 *>(sc.nodes + tr.node);
            float4 q0 = __ldg(np4), q1 = __ldg(np4 + 1), q2 = __ldg(np4 + 2);
            float2 q3 = __ldg(reinterpret_cast<const float2 *>(np4 + 3));
            n0[0] = q0.x; n0[1] = q0.y; n0[2] = q0.z; n0[3] = q0.w; n0[4] = q1.x; n0[5] = q1.y; n0[6] = q1.z; n0[7] = q1.w;
            n1[0] = q2.x; n1[1] = q2.y; n1[2] = q2.z; n1[3] = q2.w; n1[4] = q3.x; n1[5] = q3.y; n1[6] = 0.f; n1[7] = 0.f;
        }
#endif
        int2 ch = make_int2(__float_as_int(n1[4]), __float_as_int(n1[5]));
        float tn0, tn1;
        if constexpr (COUNT) tl.box += 2;
        bool h0 = slab_test(f, n0[0], n0[1], n0[2], n0[3], n1[0], n1[1], tr.cullk, tn0);
        bool h1 = slab_test(f, n0[4], n0[5], n0[6], n0[7], n1[2], n1[3], tr.cullk, tn1);
        if (h0 && h1) {
            bool swap = tn1 < tn0;
            tr.node = swap ? ch.y : ch.x;
            if (tr.sp < kBvhStack) {                     // always true: ert_scene_create rejects trees of depth >= kBvhStack
                stack[tr.sp] = swap ? ch.x : ch.y;
                tr.sp++;
            }
        } else if (h0) {
            tr.node = ch.x;
        } else if (h1) {
            tr.node = ch.y;
        } else {
            trav_pop(tr, stack);
        }
    }
    if (tr.node == kTravDone) return true;
    {
        int code = ~tr.node;
        int first = code >> 3, cnt = (code & 7) + 1;
        WF_ASSERT(first >= 0 && first + cnt <= sc.n_spheres, "leaf first %d cnt %d", first, cnt);
#pragma unroll 1
        for (int k = 0; k < cnt; k++) {
            float4 fs = __ldg(sc.leaf_filter + first + k);
            leaf_sphere<COUNT>(sc, f, ray, fs, sc.leaf_sph, first + k, skip_obj, best, tr.cullk, tl);
        }
    }
    if constexpr (ANY) {
        if (best.obj != seed_obj) return true;
    }
    trav_pop(tr, stack);
    return tr.node == kTravDone;
}

// ------------------------------------------------------------------ cell-grid walk (3-D DDA)
// Path rays of scenes that have a cell grid (cell_grid.h) visit the cells along the ray front to
// back instead of walking the BVH.  Plane k of an axis sits at lo + k*cs; the ray reaches it at
// t = k*A + B with A = cs/d, B = (lo - o)/d — one FFMA from the integer-valued float k, so errors do
// not accumulate and t is monotone in k.  The walk therefore visits exactly the cells of SOME
// sequence of plane crossings each within a few ulps (of position) of the true one, i.e. at every
// parameter the true ray is within m/2 of the cell the walk is in (m: the margin of make_sray).
// The builder lists a sphere in every cell its box inflated by eps overlaps and a ray uses the grid
// only if 4m <= eps, so every sphere the ray touches is listed in a visited cell; the walk ends
// when the next cell starts beyond the cull distance of the incumbent (an upper bound, as in the
// BVH walk) or outside the grid.  Every step moves one plane index towards its end, so the loop
// ends whatever the float values are.
#ifndef ERT_GRID_RAY_SMEM
#define ERT_GRID_RAY_SMEM 1          /* the six DDA constants of a ray live in shared memory, not registers */
#endif
struct GridRay {
#if ERT_GRID_RAY_SMEM
    float *p;                        // column of this thread, stride kWfThreads: A[3], B[3]
    __device__ __forceinline__ void bind()
    {
        __shared__ float gslots[6][kWfThreads];
        p = &gslots[0][threadIdx.x];
    }
    __device__ __forceinline__ float A(int k) const { return p[k * kWfThreads]; }
    __device__ __forceinline__ float B(int k) const { return p[(3 + k) * kWfThreads]; }
    __device__ __forceinline__ void set(int k, float a, float b) { p[k * kWfThreads] = a; p[(3 + k) * kWfThreads] = b; }
#else
    float a_[3], b_[3];
    __device__ __forceinline__ void bind() { }
    __device__ __forceinline__ float A(int k) const { return a_[k]; }
    __device__ __forceinline__ float B(int k) const { return b_[k]; }
    __device__ __forceinline__ void set(int k, float a, float b) { a_[k] = a; b_[k] = b; }
#endif
    int sgn;                         // bit k set: the ray runs towards +k
};
struct GridWalk {
    float nbx, nby, nbz;             // index of the next plane along each axis (integer-valued)
    float tx, ty, tz;                // ray parameter there
    int id;                          // linear id of the cell the walk looks at next; < 0: the walk is over
    float cullk;
};
constexpr int kOrderUnknown = INT_MIN;          // Hit::order of a sphere whose list position has not been fetched yet

// list position of the incumbent (the grid walk fetches it only when a tie asks for it)
__device__ __forceinline__ int hit_order(const DevScene &sc, const Hit &best)
{
    return best.order != kOrderUnknown ? best.order : object_order(sc, best.obj);
}

__device__ __forceinline__ void grid_start(GridWalk &g, GridRay &r, const DevScene &sc, const SRay &f, float cullk)
{
    const DevScene::CellGridDev &cg = sc.cg;
    g.cullk = cullk;
    g.id = -1;
    float t0;
    if (!slab_test(f, cg.lo[0], cg.hi[0], cg.lo[1], cg.hi[1], cg.lo[2], cg.hi[2], cullk, t0)) return;
    const float inv_cs = 1.0f / cg.cs;
    r.bind();
    const float Ax = cg.cs * f.ix, Ay = cg.cs * f.iy, Az = cg.cs * f.iz;
    const float Bx = __fmaf_rn(cg.lo[0], f.ix, -(f.ox * f.ix));
    const float By = __fmaf_rn(cg.lo[1], f.iy, -(f.oy * f.iy));
    const float Bz = __fmaf_rn(cg.lo[2], f.iz, -(f.oz * f.iz));
    r.set(0, Ax, Bx); r.set(1, Ay, By); r.set(2, Az, Bz);
    float cx = floorf((__fmaf_rn(f.dx, t0, f.ox) - cg.lo[0]) * inv_cs);
    float cy = floorf((__fmaf_rn(f.dy, t0, f.oy) - cg.lo[1]) * inv_cs);
    float cz = floorf((__fmaf_rn(f.dz, t0, f.oz) - cg.lo[2]) * inv_cs);
    cx = fminf(fmaxf(cx, 0.f), (float)(cg.rx - 1));
    cy = fminf(fmaxf(cy, 0.f), (float)(cg.ry - 1));
    cz = fminf(fmaxf(cz, 0.f), (float)(cg.rz - 1));
    const bool px = f.ix >= 0.f, py = f.iy >= 0.f, pz = f.iz >= 0.f;
    g.nbx = cx + (px ? 1.f : 0.f); g.nby = cy + (py ? 1.f : 0.f); g.nbz = cz + (pz ? 1.f : 0.f);
    g.tx = __fmaf_rn(g.nbx, Ax, Bx); g.ty = __fmaf_rn(g.nby, Ay, By); g.tz = __fmaf_rn(g.nbz, Az, Bz);
    const int sy = cg.rx, sz = cg.rx * cg.ry;
    r.sgn = (px ? 1 : 0) | (py ? 2 : 0) | (pz ? 4 : 0);
    g.id = (int)cx + sy * (int)cy + sz * (int)cz;
}

// Moves the walk to the next cell (id < 0 when that is outside the grid) and returns the ray
// parameter at which the cell just left ends, i.e. where the next one starts.
__device__ __forceinline__ float grid_advance(GridWalk &g, const GridRay &r, const DevScene::CellGridDev &cg)
{
    const float te = fminf(fminf(g.tx, g.ty), g.tz);
    if (g.tx == te) {
        const bool pos = (r.sgn & 1) != 0;
        g.nbx += pos ? 1.f : -1.f;
        g.tx = __fmaf_rn(g.nbx, r.A(0), r.B(0));
        g.id += pos ? 1 : -1;
        if (g.nbx == (pos ? (float)(cg.rx + 1) : -1.f)) g.id = -1;
    } else if (g.ty == te) {
        const bool pos = (r.sgn & 2) != 0;
        g.nby += pos ? 1.f : -1.f;
        g.ty = __fmaf_rn(g.nby, r.A(1), r.B(1));
        g.id += pos ? cg.rx : -cg.rx;
        if (g.nby == (pos ? (float)(cg.ry + 1) : -1.f)) g.id = -1;
    } else {
        const bool pos = (r.sgn & 4) != 0;
        g.nbz += pos ? 1.f : -1.f;
        g.tz = __fmaf_rn(g.nbz, r.A(2), r.B(2));
        g.id += pos ? cg.rx * cg.ry : -(cg.rx * cg.ry);
        if (g.nbz == (pos ? (float)(cg.rz + 1) : -1.f)) g.id = -1;
    }
    return te;
}

// The spheres listed in one cell, in two phases.  The filter phase runs stage 1 of the FP32 filter and the
// behind-the-origin cull over up to 32 of them (survivors as a bit mask: bits 0-5 the spheres inside the cell's
// block, bits 6.. the overflow entries from `obase` on), grid_exact the literal FP64 tests of the survivors: callers
// put the second phase where the lanes of a warp meet again, so that they enter the expensive part together
// instead of one at a time.  A sphere is listed in every cell it overlaps, so the incumbent itself comes by again:
// it is skipped.  The beyond-the-incumbent cull waits for grid_exact, where it sees the newest cull distance.
// (The sphere a reflected ray leaves passes stage 1 in every cell that lists it — the origin lies on it — and was
// a third of all survivors before the behind-the-origin cull moved into the mask.)
__device__ __forceinline__ unsigned int stage1_bit(const SRay &f, float4 s, float nth, float nbc)
{
    float b, v;
    filter_stage1(f, s, b, v);
    return (v < nth || b < nbc) ? 0u : 1u;
}
constexpr int kGridInline = kCellGridInline * kCellGridBlocks;      // mask bits 0..11: the spheres in the cell's two blocks
constexpr int kGridOverChunk = 20;                                  // overflow entries per survivor mask (bits 12..31)
constexpr int kBlockU4 = 8 * kCellGridBlocks;                       // uint4 per cell
static_assert(kCellGridInline == 6 && kCellGridBlocks == 2 && kCellGridPad == 4 && kGridOverChunk % kCellGridPad == 0 &&
              kGridInline + kGridOverChunk <= 32, "mask layout");

// stage 1 over `cnt` overflow entries from `e0` on (whole groups of four; the padding never passes)
__device__ __forceinline__ unsigned int grid_filter_over(const DevScene &sc, const SRay &f, unsigned int e0, int cnt)
{
    const float4 *fp4 = sc.cg.over_filter + e0;
    const float nth = -f.theta, nbc = -f.bcull;
    unsigned int surv = 0u;
    float p[8], q[8];
    ldg256(fp4, p); ldg256(fp4 + 2, q);                  // groups of four are 64-byte aligned: two 256-bit loads
    float4 s0 = make_float4(p[0], p[1], p[2], p[3]), s1 = make_float4(p[4], p[5], p[6], p[7]);
    float4 s2 = make_float4(q[0], q[1], q[2], q[3]), s3 = make_float4(q[4], q[5], q[6], q[7]);
#pragma unroll 1
    for (int k = 0; k < cnt; k += 4) {
        // the next group is in flight while this one is tested (one group past the list at the end: it exists)
        ldg256(fp4 + k + 4, p); ldg256(fp4 + k + 6, q);
        const float4 n0 = make_float4(p[0], p[1], p[2], p[3]), n1 = make_float4(p[4], p[5], p[6], p[7]);
        const float4 n2 = make_float4(q[0], q[1], q[2], q[3]), n3 = make_float4(q[4], q[5], q[6], q[7]);
        const unsigned int m = stage1_bit(f, s0, nth, nbc) | (stage1_bit(f, s1, nth, nbc) << 1) |
                               (stage1_bit(f, s2, nth, nbc) << 2) | (stage1_bit(f, s3, nth, nbc) << 3);
        surv |= m << (kGridInline + k);
        s0 = n0; s1 = n1; s2 = n2; s3 = n3;
    }
    return surv;
}

template <bool COUNT>
__device__ __forceinline__ void grid_exact(const DevScene &sc, const SRay &f, const RaySlot &ray, int cell,
                                           unsigned int obase, unsigned int surv, int skip_obj, Hit &best, float &cullk,
                                           Tally<COUNT> &tl)
{
    const DevScene::CellGridDev &cg = sc.cg;
    const uint4 *blk = cg.blocks + (size_t)cell * kBlockU4;
    WF_ASSERT(cell >= 0 && cell < cg.rx * cg.ry * cg.rz, "cell %d of %d", cell, cg.rx * cg.ry * cg.rz);
    PROBE(0, surv ? 1 : 0);
    PROBE(1, __popc(surv));
    while (surv) {
        const int k = __ffs((int)surv) - 1;
        surv &= surv - 1u;
        int sph;
        float4 fs;
        if (k < kGridInline) {
            const int half = k >= kCellGridInline ? 1 : 0, j = k - half * kCellGridInline;
            sph = __ldg(reinterpret_cast<const int *>(blk + 8 * half) + 4 * kCellGridInline + j);
            fs = __ldg(reinterpret_cast<const float4 *>(blk + 8 * half) + j);
        } else {
            const unsigned int e = obase + (unsigned int)(k - kGridInline);
            sph = __ldg(cg.over_sph + e);
            fs = __ldg(cg.over_filter + e);
        }
        if (sph < 0) continue;                           // padding (only a NaN ray gets here)
        WF_ASSERT(sph < sc.n_spheres, "sphere %d of %d (cell %d, bit %d)", sph, sc.n_spheres, cell, k);
        const int code = obj_code(OBJ_SPHERE, sph);
        if (code == skip_obj || code == best.obj) { PROBE(2, 1); continue; }
        // the FP64 sphere is asked for before the cull decides whether it is needed (nine times of ten it is): the
        // whole warp waits for this phase, so its longest latency starts as early as the index is known
        const double4 es = ld_sphere(sc.sph_exact + sph);
        {
            float b, v;
            filter_stage1(f, fs, b, v);
            if (!filter_stage2(f, fs, b, v, cullk)) { PROBE(4, 1); continue; }
        }
        double t;
        TALLY(exact_sph);
        if (sphere_exact(ray.O(), ray.D(), ray.a(), es, t)) {
            PROBE(5, 1);
            // better() of erl:319 with the list positions fetched only for a tie
            bool win = best.obj < 0 || t < best.t;
            int ord = kOrderUnknown;
            if (!win && t == best.t) {
                ord = sc.sph_order[sph];
                best.order = hit_order(sc, best);
                win = ord < best.order;
            }
            if (win) {
                PROBE(6, 1);
                best.t = t; best.order = ord; best.obj = code;
                cullk = cullk_from(f, ray.inv_sqrt_a(), best);
            }
        }
    }
}

// Runs empty cells until the ray holds a cell with spheres and filters those (while-while, like
// trav_step).  A cell's block sits at an address the DDA computes: no dependent fetch stands between
// the step and the spheres.  (Prefetching the next cell's block — to L1 or L2, one block or both — is
// within 0.4 % of not prefetching at all: DESIGN.md "dropped".)  Returns false when the walk is over
// (the next cell starts beyond the cull distance, or outside the grid); otherwise `surv` marks the filter survivors of cell `cell`
// (overflow entries counted from `obase`) and `te` is where the cell ends: grid_exact on the
// survivors and grid_leave complete the step.
template <bool COUNT>
__device__ __forceinline__ bool grid_find(GridWalk &g, const GridRay &r, const DevScene &sc, const RaySlot &ray,
                                          const SRay &f, Hit &best, int skip_obj, Tally<COUNT> &tl, unsigned int &surv,
                                          int &cell, unsigned int &obase, float &te)
{
    const DevScene::CellGridDev &cg = sc.cg;
    surv = 0u;
    const uint4 *blk;
    uint2 hd;
    float4 s0, s1, s2, s3, s4, s5;
    for (;;) {
        if (g.id < 0) return false;
        WF_ASSERT(g.id < cg.rx * cg.ry * cg.rz, "cell %d of %d", g.id, cg.rx * cg.ry * cg.rz);
        cell = g.id;
        blk = cg.blocks + (size_t)cell * kBlockU4;
        // one 128-byte line: count and overflow word, six filter spheres
        hd = __ldg(reinterpret_cast<const uint2 *>(blk) + 15);
        {
            float p[8];
            ldg256(blk, p);     s0 = make_float4(p[0], p[1], p[2], p[3]); s1 = make_float4(p[4], p[5], p[6], p[7]);
            ldg256(blk + 2, p); s2 = make_float4(p[0], p[1], p[2], p[3]); s3 = make_float4(p[4], p[5], p[6], p[7]);
            ldg256(blk + 4, p); s4 = make_float4(p[0], p[1], p[2], p[3]); s5 = make_float4(p[4], p[5], p[6], p[7]);
        }
        TALLY(cell);
        te = grid_advance(g, r, cg);
        if (hd.x) break;
        if (te > g.cullk) { g.id = -1; return false; }
    }
    const float nth = -f.theta, nbc = -f.bcull;
    int cnt = (int)hd.x;
    obase = hd.y;
    if constexpr (COUNT) tl.filter += cnt;
    surv = stage1_bit(f, s0, nth, nbc) | (stage1_bit(f, s1, nth, nbc) << 1) | (stage1_bit(f, s2, nth, nbc) << 2) |
           (stage1_bit(f, s3, nth, nbc) << 3) | (stage1_bit(f, s4, nth, nbc) << 4) | (stage1_bit(f, s5, nth, nbc) << 5);
    if (cnt > kCellGridInline) {
        // the second block of the cell (asked for a step ago, like the first)
        {
            float p[8];
            ldg256(blk + 8, p);  s0 = make_float4(p[0], p[1], p[2], p[3]); s1 = make_float4(p[4], p[5], p[6], p[7]);
            ldg256(blk + 10, p); s2 = make_float4(p[0], p[1], p[2], p[3]); s3 = make_float4(p[4], p[5], p[6], p[7]);
            ldg256(blk + 12, p); s4 = make_float4(p[0], p[1], p[2], p[3]); s5 = make_float4(p[4], p[5], p[6], p[7]);
        }
        surv |= (stage1_bit(f, s0, nth, nbc) << 6) | (stage1_bit(f, s1, nth, nbc) << 7) | (stage1_bit(f, s2, nth, nbc) << 8) |
                (stage1_bit(f, s3, nth, nbc) << 9) | (stage1_bit(f, s4, nth, nbc) << 10) | (stage1_bit(f, s5, nth, nbc) << 11);
        cnt -= kGridInline;
        if (cnt > 0) {
            while (cnt > kGridOverChunk) {
                // rare: more than one mask's worth of spheres in the cell; all but the last chunk are finished here
                const unsigned int sv = surv | grid_filter_over(sc, f, obase, kGridOverChunk);
                grid_exact<COUNT>(sc, f, ray, cell, obase, sv, skip_obj, best, g.cullk, tl);
                surv = 0u;
                obase += kGridOverChunk; cnt -= kGridOverChunk;
            }
            surv |= grid_filter_over(sc, f, obase, cnt);
        }
    }
    return true;
}
__device__ __forceinline__ bool grid_leave(GridWalk &g, float te)
{
    if (te > g.cullk) g.id = -1;
    return g.id < 0;
}

// one whole step for callers that do not separate the phases; returns true when the search is over
template <bool COUNT>
__device__ __forceinline__ bool grid_step(GridWalk &g, const GridRay &r, const DevScene &sc, const RaySlot &ray,
                                          const SRay &f, Hit &best, int skip_obj, Tally<COUNT> &tl)
{
    unsigned int surv, obase;
    int cell;
    float te;
    if (!grid_find<COUNT>(g, r, sc, ray, f, best, skip_obj, tl, surv, cell, obase, te)) return true;
    grid_exact<COUNT>(sc, f, ray, cell, obase, surv, skip_obj, best, g.cullk, tl);
    return grid_leave(g, te);
}

// spheres too large for the cells: every ray tests them before its walk
template <bool COUNT>
__device__ __forceinline__ void grid_big_spheres(const DevScene &sc, const SRay &f, const RaySlot &ray, int skip_obj,
                                                 Hit &best, float &cullk, Tally<COUNT> &tl)
{
    for (int k = 0; k < sc.cg.n_big; k++) {
        float4 fs = __ldg(sc.sph_filter + __ldg(sc.cg.big + k));
        leaf_sphere<COUNT>(sc, f, ray, fs, sc.cg.big, k, skip_obj, best, cullk, tl);
    }
}

// A ray whose margin is too large for the grid (origin far outside the scene) walks the BVH
// instead, and a ray beyond the filter's range tests every sphere.  Rare, so it is a call: the
// walk state of the BVH stays out of the callers' registers.
__device__ __forceinline__ void walk_bvh_instead(const DevScene *scp, double *slot, int skip_obj, Hit *best_io)
{
    const DevScene &sc = *scp;
    RaySlot ray;
    ray.p = slot;
    SRay f;
    double a, inv;
    if (!make_sray(sc, ray.O(), ray.D(), f, a, inv)) {
        *best_io = scan_spheres_instead(scp, ray.O(), ray.D(), *best_io, skip_obj, false, -1);
        return;
    }
    Hit best = *best_io;
    Tally<false> tl;
    Trav<false> tr;
    int stack[kBvhStack];
    trav_start(tr, stack, f, inv, best);
    while (!trav_step<false, false>(tr, stack, sc, ray, f, best, skip_obj, -1, tl)) { }
    *best_io = best;
}

// Sets a ray up for the grid: the spheres too large for the cells, then the start of the walk.
// Returns false when there is no walk to make (also for rays that had to walk the BVH instead).
template <bool COUNT>
__device__ __forceinline__ bool grid_begin(GridWalk &g, GridRay &r, const DevScene &sc, const RaySlot &ray, const SRay &f,
                                           double inv_sqrt_a, int skip_obj, Hit &best, Tally<COUNT> &tl)
{
    g.id = -1;
    if (!(f.m4 <= sc.cg.eps)) {
        Hit tmp = best;
        walk_bvh_instead(&sc, ray.p, skip_obj, &tmp);
        best = tmp;
        return false;
    }
    float cullk = cullk_from(f, inv_sqrt_a, best);
    grid_big_spheres<COUNT>(sc, f, ray, skip_obj, best, cullk, tl);
    grid_start(g, r, sc, f, cullk);
    return g.id >= 0;
}

template <bool COUNT>
__device__ __forceinline__ void grid_trace(const DevScene &sc, const RaySlot &ray, const SRay &f, double inv_sqrt_a,
                                           int skip_obj, Hit &best, Tally<COUNT> &tl)
{
    GridWalk g;
    GridRay r;
    if (!grid_begin<COUNT>(g, r, sc, ray, f, inv_sqrt_a, skip_obj, best, tl)) return;
    while (!grid_step<COUNT>(g, r, sc, ray, f, best, skip_obj, tl)) { }
    best.order = hit_order(sc, best);
}

// one ray through the cell grid, no persistence (ert_trace_rays with ERT_ACCEL_GRID)
__device__ void trace_ray_grid(const DevScene &sc, d3 O, d3 D, Hit &best)
{
    __shared__ double slots[kRaySlotDoubles][kWfThreads];
    RaySlot ray;
    ray.p = &slots[0][threadIdx.x];
    SRay f;
    Tally<false> tl;
    double a, inv;
    make_sray(sc, O, D, f, a, inv);
    ray.put(O, D, a, inv);
    grid_trace<false>(sc, ray, f, inv, -1, best, tl);
}

// one ray, no persistence (ert_trace_rays); the FP64 ray sits in a local column
__device__ void trace_ray_wavefront(const DevScene &sc, d3 O, d3 D, Hit &best)
{
    __shared__ double slots[kRaySlotDoubles][kWfThreads];
    RaySlot ray;
    ray.p = &slots[0][threadIdx.x];
    SRay f;
    Tally<false> tl;
    Trav<false> tr;
    int stack[kBvhStack];
    double a, inv;
    if (!make_sray(sc, O, D, f, a, inv)) {
        best = scan_spheres_instead(&sc, O, D, best, -1, false, -1);
        return;
    }
    ray.put(O, D, a, inv);
    trav_start(tr, stack, f, inv, best);
    while (!trav_step<false, false>(tr, stack, sc, ray, f, best, -1, -1, tl)) { }
}

// ------------------------------------------------------------------ pixel <-> queue index
// Pixel i of the part: 8x4 tile (i >> 5), lane (i & 31) inside it, tiles row-major.
__device__ __forceinline__ void pixel_of_index(const FrameParams &fp, const WfBuf &wf, int i, int &X, int &local_y,
                                               int &Y, bool &inside)
{
    int tile = i >> 5, lane = i & 31;
    int ty = tile / wf.tiles_x, tx = tile - ty * wf.tiles_x;
    X = tx * 8 + (lane & 7);
    local_y = ty * 4 + (lane >> 3);
    if (fp.n_parts > 1 && fp.band_rows > 0) {
        int j = local_y / fp.band_rows;
        Y = (fp.part + j * fp.n_parts) * fp.band_rows + (local_y - j * fp.band_rows);
    } else {
        Y = local_y;
    }
    inside = X < fp.width && local_y < fp.local_rows && Y < fp.height;
}

__device__ __forceinline__ double path_weight_of_index(const WfBuf &wf, bool first, unsigned int i)
{
    return first ? 1.0 : __ldcs(&wf.q[i].W);
}
__device__ __forceinline__ void path_ray_of_index(const FrameParams &fp, const WfBuf &wf, bool first, unsigned int i,
                                                  d3 &O, d3 &D, int &pid, bool &valid, double *W_out = nullptr)
{
    if (first) {
        int X, ly, Y;
        pixel_of_index(fp, wf, (int)i, X, ly, Y, valid);
        pid = (int)i;
        if (valid) primary_ray(fp, X, Y, O, D);                 // erl:486-511
        if (W_out) *W_out = 1.0;
    } else {
        valid = true;
        // queue traffic is read once: streaming loads keep it from evicting the scene
        const double4 a = ld_rec32_cs(wf.q + i), b = ld_rec32_cs(reinterpret_cast<const char *>(wf.q + i) + 32);
        O = mk(a.x, a.y, a.z);
        D = mk(b.x, b.y, b.z);
        pid = (int)(__double_as_longlong(b.w) & 0xffffffffll);
        if (W_out) *W_out = a.w;
    }
}

// ------------------------------------------------------------------ binning hits by location
// Rays that leave a curved surface scatter: the hits of bounce >= 1 arrive in an order that
// has little to do with where they are, and a warp of their shadow rays walks 32 unrelated
// parts of the tree.  A counting sort by the Morton cell of the hit location (a uniform grid
// over the sphere bounds) restores the coherence bounce 0 has for free.  The order of a queue
// never changes a pixel (every record carries its pixel), so this is purely a schedule.
__device__ __forceinline__ unsigned int part1by2(unsigned int x)
{
    x &= 0x3ffu;
    x = (x | (x << 16)) & 0x30000ffu;
    x = (x | (x << 8)) & 0x300f00fu;
    x = (x | (x << 4)) & 0x30c30c3u;
    x = (x | (x << 2)) & 0x9249249u;
    return x;
}
// (Measured and dropped: a grid narrowed to mean +- k sigma of the previous bounce's hits; the octant of
// the reflected direction as the leading key bits.  7 -> 8 bits per axis was worth 9 % on C4.)
__device__ __forceinline__ unsigned int sort_cell(const DevScene &sc, d3 P)
{
    const float top = (float)((1 << kSortBits) - 1);
    float fx = fminf(fmaxf(((float)P.x - sc.grid_lo[0]) * sc.grid_scale[0], 0.f), top);
    float fy = fminf(fmaxf(((float)P.y - sc.grid_lo[1]) * sc.grid_scale[1], 0.f), top);
    float fz = fminf(fmaxf(((float)P.z - sc.grid_lo[2]) * sc.grid_scale[2], 0.f), top);
    return part1by2((unsigned int)fx) | (part1by2((unsigned int)fy) << 1) | (part1by2((unsigned int)fz) << 2);
}

// exclusive scan of the histogram, phase A: each block scans kSortScanBlock cells in place
__global__ void __launch_bounds__(1024) wf_bin_scan_a(const __grid_constant__ WfBuf wf)
{
    __shared__ unsigned int warp_sums[32];
    unsigned int *h = wf.hist + (size_t)blockIdx.x * kSortScanBlock + threadIdx.x * 4;
    uint4 v = *reinterpret_cast<uint4 *>(h);
    unsigned int t = v.x + v.y + v.z + v.w;
    unsigned int incl = t;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned int w = warp_sums[lane], wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned int o = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += o;
        }
        warp_sums[lane] = wi - w;
        if (lane == 31) wf.sums[blockIdx.x] = wi;
    }
    __syncthreads();
    unsigned int base = warp_sums[warp] + incl - t;
    uint4 o;
    o.x = base; o.y = base + v.x; o.z = o.y + v.y; o.w = o.z + v.z;
    *reinterpret_cast<uint4 *>(h) = o;
}
// phase B: exclusive scan of the kSortBlocks block totals (one block)
__global__ void __launch_bounds__(kSortScanBThreads) wf_bin_scan_b(const __grid_constant__ WfBuf wf)
{
    __shared__ unsigned int warp_sums[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int v[kSortScanBItems];
    unsigned int t = 0;
#pragma unroll
    for (int k = 0; k < kSortScanBItems; k++) { v[k] = wf.sums[threadIdx.x * kSortScanBItems + k]; t += v[k]; }
    unsigned int incl = t;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned int w = lane < kSortScanBThreads / 32 ? warp_sums[lane] : 0u, wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned int o = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += o;
        }
        warp_sums[lane] = wi - w;
    }
    __syncthreads();
    unsigned int run = warp_sums[warp] + incl - t;
#pragma unroll
    for (int k = 0; k < kSortScanBItems; k++) { wf.sums[threadIdx.x * kSortScanBItems + k] = run; run += v[k]; }
}
// scatter: every raw hit record moves to its cell's range of the sorted hit queue
__global__ void __launch_bounds__(kWfThreads) wf_bin_scatter(const __grid_constant__ WfBuf wf, int bounce)
{
    const unsigned int n_hits = wf.ctr[bounce * kWfCtr + WF_NHITS];
    for (size_t h = (size_t)blockIdx.x * kWfThreads + threadIdx.x; h < n_hits; h += (size_t)gridDim.x * kWfThreads) {
        unsigned int key = wf.r_key[h];
        size_t s = (size_t)atomicAdd(wf.hist + key, 1u) + wf.sums[key / kSortScanBlock];
        const uint4 *sh = reinterpret_cast<const uint4 *>(wf.raw_head + h);
        const uint4 *st = reinterpret_cast<const uint4 *>(wf.raw_tail + h);
        uint4 r0 = sh[0], r1 = sh[1], r2 = st[0], r3 = st[1], r4 = st[2], r5 = st[3];
        uint4 *dh = reinterpret_cast<uint4 *>(wf.hit_head + s);
        uint4 *dt = reinterpret_cast<uint4 *>(wf.hit_tail + s);
        dh[0] = r0; dh[1] = r1; dt[0] = r2; dt[1] = r3; dt[2] = r4; dt[3] = r5;
    }
}

// ------------------------------------------------------------------ shadow queries by direction
// Cell of a direction in a light's cube map, in FP32 from the filter ray's direction: the operations of
// light_grid_cell_f32() in light_grid.cpp (whose slack covers their rounding; tests/test_light_grid.py checks the
// listing with this very computation).  Two FP64 divisions per shadow ray became one FP32 reciprocal.
__device__ __forceinline__ unsigned int light_grid_cell_dev(const SRay &f, int res)
{
    const float ax = fabsf(f.dx), ay = fabsf(f.dy), az = fabsf(f.dz);
    int m = 0;
    float am = ax, dm = f.dx, du = f.dy, dv = f.dz;
    if (ay > am) { m = 1; am = ay; dm = f.dy; du = f.dz; dv = f.dx; }
    if (az > am) { m = 2; am = az; dm = f.dz; du = f.dx; dv = f.dy; }
    const int face = 2 * m + (dm < 0.0f ? 1 : 0);
    const float inv = __frcp_rn(am);
    const float u = du * inv, v = dv * inv;
    const float half = 0.5f * (float)res;
    int iu = (int)floorf((u + 1.0f) * half), iv = (int)floorf((v + 1.0f) * half);
    iu = min(max(iu, 0), res - 1);
    iv = min(max(iv, 0), res - 1);
    return (unsigned int)((face * res + iv) * res + iu);
}

// Is any sphere in the way of the shadow ray (O = the light, D) before its target?  `best` holds
// the target as incumbent.  Candidates come from the light's direction grid, nearest first; each
// goes through the FP32 filter and then the literal FP64 test, exactly like a BVH leaf sphere.
template <bool COUNT>
__device__ __forceinline__ bool light_grid_occluded(const DevScene &sc, const LightGridDev &lg, const SRay &f, d3 O,
                                                    d3 D, double a, double inv_sqrt_a, const Hit &best, int target,
                                                    Tally<COUNT> &tl)
{
    const float cull0 = cullk_from(f, inv_sqrt_a, best);
    const unsigned int cell = light_grid_cell_dev(f, lg.res);
    // the head of the cell carries its nearest candidate and the range of the others: one dependent
    // fetch for the rays that the first candidate settles (most of them)
    float c[8];
    ldg256(lg.head + cell, c);
    unsigned int e = __float_as_uint(c[6]);
    const unsigned int e1 = __float_as_uint(c[7]);
    for (;;) {
        if (c[5] > cull0) break;                         // this and all later candidates lie beyond the target
        const float4 fs = make_float4(c[0], c[1], c[2], c[3]);
        const int sph = __float_as_int(c[4]);
        const bool more = e < e1;
        if (more) ldg256(lg.cand + e, c);                // in flight while this candidate is tested
        e++;
        float fb, fv;
        TALLY(filter);
        // the target itself is the usual first candidate of a lit ray: it is recognised before the stage-2 cull
        if (filter_stage1(f, fs, fb, fv) && obj_code(OBJ_SPHERE, sph) != target && filter_stage2(f, fs, fb, fv, cull0)) {
            double th;
            TALLY(exact_sph);
            if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + sph), th) && better(th, sc.sph_order[sph], best)) return true;
        }
        if (!more) break;
    }
    for (int k = 0; k < lg.n_always; k++) {
        const int sph = lg.always[k];
        if (obj_code(OBJ_SPHERE, sph) == target) continue;
        double th;
        TALLY(exact_sph);
        if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + sph), th) && better(th, sc.sph_order[sph], best)) return true;
    }
    return false;
}

// ------------------------------------------------------------------ kernels
// lanes below `lane` in mask m
__device__ __forceinline__ int rank_in(unsigned int m, int lane) { return __popc(m & ((1u << lane) - 1u)); }

__device__ __forceinline__ void write_hit(HitHead *heads, HitTail *tails, size_t s, d3 P, d3 N, d3 D, int obj, int order,
                                          int pid, double W)
{
    // three 256-bit stores: {P, obj | order}, {N, pid}, {D, W}
    const double oo = __longlong_as_double(((long long)order << 32) | (long long)(unsigned int)obj);
    const double pp = __longlong_as_double((long long)(unsigned int)pid);
    st_rec32(heads + s, P.x, P.y, P.z, oo);
    st_rec32(tails + s, N.x, N.y, N.z, pp);
    st_rec32(reinterpret_cast<char *>(tails + s) + 32, D.x, D.y, D.z, W);
}

// The reflection ray of a hit (erl:216-224): leaves the hit location along the bounced direction and carries the
// path's weight times (number of lights * reflectivity) — what the reference's fold adds L times over (erl:239-247).
// A path ends at the depth limit, at a surface that reflects nothing, and when its weight is zero.  Every lane of the
// warp calls this; `hit` says whether the lane has one.
__device__ __forceinline__ void emit_next_rays(const DevScene &sc, const FrameParams &fp, const WfBuf &wf, int bounce,
                                               unsigned int *ctr, int lane, bool hit, d3 P, d3 N, d3 D, int obj, int pid, double W)
{
    bool cont = false;
    double refl = 0.0;
    if (hit && bounce + 1 < fp.depth) {
        refl = reflectivity_of(sc, obj);
        cont = !(refl == 0.0 || W == 0.0);
    }
    const unsigned int m = __ballot_sync(0xffffffffu, cont);
    if (!m) return;
    unsigned int slot0 = 0;
    if (lane == 0) slot0 = atomicAdd(ctr + WF_NNEXT, (unsigned int)__popc(m));
    slot0 = __shfl_sync(0xffffffffu, slot0, 0);
    if (cont) {
        const size_t s = slot0 + rank_in(m, lane);
        const d3 nd = vbounce(D, N);                                  // erl:219-221
        st_rec32(wf.nq + s, P.x, P.y, P.z, W * ((double)sc.n_lights * refl));
        st_rec32(reinterpret_cast<char *>(wf.nq + s) + 32, nd.x, nd.y, nd.z, __longlong_as_double((long long)(unsigned int)pid));
    }
}

// The path kernels' own emission: hit records and reflection rays of up to 32 hits with ONE atomic (the counters of
// the hit queue and of the next path queue are neighbours: a 64-bit add reserves both ranges).  Every lane calls.
static_assert(WF_NHITS == 0 && WF_NNEXT == 1, "one 64-bit add reserves hits (low word) and next rays (high word)");
__device__ __forceinline__ void emit_hits_and_rays(const DevScene &sc, const FrameParams &fp, const WfBuf &wf, int bounce,
                                                   unsigned int *ctr, int lane, bool hit, d3 P, d3 N, d3 D, int obj,
                                                   int order, int pid, double W)
{
    const unsigned int mh = __ballot_sync(0xffffffffu, hit);
    if (!mh) return;
    bool cont = false;
    double refl = 0.0;
    if (hit && bounce + 1 < fp.depth) {
        refl = reflectivity_of(sc, obj);
        cont = !(refl == 0.0 || W == 0.0);
    }
    const unsigned int mc = __ballot_sync(0xffffffffu, cont);
    unsigned long long old = 0;
    if (lane == 0)
        old = atomicAdd(reinterpret_cast<unsigned long long *>(ctr + WF_NHITS),
                        (unsigned long long)__popc(mh) | ((unsigned long long)__popc(mc) << 32));
    old = __shfl_sync(0xffffffffu, old, 0);
    if (hit) write_hit(wf.hit_head, wf.hit_tail, (size_t)(unsigned int)old + rank_in(mh, lane), P, N, D, obj, order, pid, W);
    if (cont) {
        const size_t s = (size_t)(old >> 32) + rank_in(mc, lane);
        const d3 nd = vbounce(D, N);                                  // erl:219-221
        st_rec32(wf.nq + s, P.x, P.y, P.z, W * ((double)sc.n_lights * refl));
        st_rec32(reinterpret_cast<char *>(wf.nq + s) + 32, nd.x, nd.y, nd.z, __longlong_as_double((long long)(unsigned int)pid));
    }
}

// Work distribution of the traversal kernels.  A warp owns a chunk of kWfChunk consecutive
// queue entries at a time (one atomic per chunk) and works through it in batches of 32, so the
// rays a lane sees one after another are 32 entries apart in the (binned) queue: neighbours in
// space.  That is what makes the previous ray's sphere a good first guess for the next one.
#ifndef ERT_WF_CHUNK
#define ERT_WF_CHUNK 128
#endif
constexpr unsigned int kWfChunk = ERT_WF_CHUNK;
#ifndef ERT_WF_OCC_CACHE
#define ERT_WF_OCC_CACHE 8
#endif
constexpr int kOccCache = ERT_WF_OCC_CACHE;      // recent occluders a warp remembers (wf_trace_shadow)
static_assert(kWfChunk % 32 == 0, "chunks are whole batches");

// Chunk length for a queue of `total` entries: kWfChunk, but short queues (a band of a frame
// split over several GPUs, late bounces) are cut finer so that every warp of the grid gets
// several chunks and the tail of the launch stays short.
__device__ __forceinline__ unsigned int chunk_len(unsigned long long total)
{
    const unsigned long long warps = (unsigned long long)gridDim.x * (kWfThreads / 32);
    unsigned long long c = total / (warps * 8);
    c &= ~31ull;
    return c < 32 ? 32u : (c > kWfChunk ? kWfChunk : (unsigned int)c);
}
__device__ __forceinline__ bool next_chunk(unsigned long long *cursor, unsigned long long total, int lane,
                                           unsigned long long &begin, unsigned long long &end)
{
    const unsigned int len = chunk_len(total);
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(cursor, (unsigned long long)len);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= total) return false;
    begin = base;
    end = base + len < total ? base + len : total;
    return true;
}

// A warp that has taken the chunk [begin, end) of the path queue asks L2 for its lines: the rays of a chunk are
// handed out a few at a time as lanes finish, and each hand-out would otherwise wait for HBM with the whole
// warp standing still.  Eight arrays (origin, direction, weight, pixel), sixteen entries per line.
__device__ __forceinline__ void prefetch_path_chunk(const WfBuf &wf, unsigned long long begin, unsigned long long end, int lane)
{
    // two 64-byte rays per 128-byte line
    for (unsigned long long e = begin + (unsigned long long)(2 * lane); e < end; e += 64) prefetch_l2(wf.q + e);
}

// Path rays of one bounce: nearest_object_intersecting_ray/2 (erl:300-346) for every ray of
// the path queue (FIRST: for every pixel, rays generated on the fly).  EMIT: the batch also turns
// its hits into hit records (what wf_emit_hits does from the result arrays) — the warp is back
// together after every batch, so the FP64 of the hit location and normal runs on full warps and
// the results never travel through HBM.
template <bool FIRST, bool COUNT, bool EMIT, bool GRID, bool TRI = false>
__global__ void __launch_bounds__(kWfThreads, GRID ? ERT_GRID_MINBLOCKS : ERT_WF_MINBLOCKS)
wf_trace_path(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
              const __grid_constant__ WfBuf wf, int bounce)
{
    __shared__ double slots[kRaySlotDoubles][kWfThreads];
    RaySlot ray;
    ray.p = &slots[0][threadIdx.x];
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned long long n = FIRST ? (unsigned long long)wf.n_pad
                                       : (unsigned long long)wf.ctr[(bounce - 1) * kWfCtr + WF_NNEXT];
    unsigned long long *cursor = reinterpret_cast<unsigned long long *>(ctr + WF_FETCH_PATH);
    const int lane = threadIdx.x & 31;
    Tally<COUNT> tl;
    unsigned int rays = 0;
    int hint = -1;                                   // sphere hit by this lane's previous ray
    unsigned long long begin, end;
    while (next_chunk(cursor, n, lane, begin, end)) {
        for (unsigned long long b0 = begin; b0 < end; b0 += 32) {
            const unsigned long long i64 = b0 + lane;
            const bool in_range = i64 < end;
            const unsigned int i = (unsigned int)i64;
            bool valid = false;
            int pid = 0;
            Hit best;
            best.obj = -1; best.t = 0.0; best.order = 0x7fffffff;
            SRay f;
            GridWalk gw;
            GridRay gr;
            bool walking = false, searched = false;
            int skip = -1;
            if (in_range) {
                if constexpr (FIRST) {
                    // the pixel's colour starts at +0.0 (the frame's first launch visits every pixel exactly once:
                    // no separate 200 MB memset in front of the frame)
                    const size_t np = (size_t)wf.n_pad;
                    wf.C[i] = 0.0; wf.C[np + i] = 0.0; wf.C[2 * np + i] = 0.0;
                }
                d3 O = mk(0, 0, 0), D = mk(0, 0, 1);
                path_ray_of_index(fp, wf, FIRST, i, O, D, pid, valid);
                if (valid) {
                    rays++;
                    scan_others<COUNT, TRI>(sc, O, D, best, -1, tl);
                    double a, inv;
                    const bool filtered = make_sray(sc, O, D, f, a, inv);
                    ray.put(O, D, a, inv);
                    if (sc.n_spheres > 0) {
                        if (FIRST && hint >= 0) {                     // first reflections have too little in common (measured: 7.505 vs 7.487 ms)
                            // seed the search with the previous ray's sphere: a real candidate of the
                            // scan, so the minimum over (t, order) is unchanged
                            double t;
                            TALLY(exact_sph);
                            PROBE(7, 1);
                            if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + hint), t)) {
                                int ord = sc.sph_order[hint];
                                if (better(t, ord, best)) {
                                    best.t = t; best.order = ord; best.obj = obj_code(OBJ_SPHERE, hint);
                                    skip = best.obj;
                                }
                            }
                        }
                        if constexpr (GRID) {
                            walking = grid_begin<COUNT>(gw, gr, sc, ray, f, inv, skip, best, tl);
                        } else if (!filtered) {
                            best = scan_spheres_instead(&sc, O, D, best, skip, false, -1);
                        } else {
                            Trav<false> tr;
                            int stack[kBvhStack];
                            trav_start(tr, stack, f, inv, best);
                            while (!trav_step<false, COUNT>(tr, stack, sc, ray, f, best, skip, -1, tl)) { }
                        }
                        searched = true;
                    }
                }
            }
            if constexpr (GRID) {
                // the lanes of the batch walk to their next cell with spheres and filter them on their own,
                // then meet for the FP64 tests of the survivors
                while (__any_sync(0xffffffffu, walking)) {
                    unsigned int surv = 0u, obase = 0u;
                    int cell = 0;
                    float te = 0.f;
                    bool found = false;
                    if (walking) found = grid_find<COUNT>(gw, gr, sc, ray, f, best, skip, tl, surv, cell, obase, te);
                    __syncwarp();
                    if (surv) grid_exact<COUNT>(sc, f, ray, cell, obase, surv, skip, best, gw.cullk, tl);
                    if (walking) walking = found ? !grid_leave(gw, te) : false;
                }
            }
            if (searched && best.obj >= 0 && obj_type(best.obj) == OBJ_SPHERE) hint = obj_index(best.obj);
            if constexpr (!EMIT) {
                if (in_range) {
                    __stcs(wf.res_hit + i, make_int2(valid ? best.obj : -1, hit_order(sc, best)));
                    __stcs(wf.res_t + i, best.t);
                }
            } else {
                const bool hit = valid && best.obj >= 0;
                d3 P = mk(0, 0, 0), N = P, D = P;
                double W = 0.0;
                if (hit) {
                    const d3 O = ray.O();
                    D = ray.D();
                    P = vadd(O, vscale(D, best.t));                   // erl:384-387 / 443-447 / 471-475
                    N = hit_normal(sc, best.obj, P);
                    W = path_weight_of_index(wf, FIRST, i);
                }
                emit_hits_and_rays(sc, fp, wf, bounce, ctr, lane, hit, P, N, D, best.obj, hit ? hit_order(sc, best) : 0, pid, W);
            }
        }
    }
    flush_counters<COUNT>(fp, (int)rays, tl);
}

// Path rays of bounces >= 1 have nothing to do with their queue neighbours (they leave curved
// surfaces in all directions), walks differ in length several-fold, and a batch of 32 waits for
// its longest one.  This form keeps the warp resident and hands new rays to lanes that have
// finished once fewer than kRefillBelow lanes are still walking.  (Set-up of a path ray is a
// queue read and a plane test, cheap enough to run on a few lanes at a time; for shadow rays,
// whose set-up is heavy FP64, the same scheme lost.)
#ifndef ERT_WF_REFILL
#define ERT_WF_REFILL 20
#endif
constexpr int kRefillBelow = ERT_WF_REFILL;
#ifndef ERT_WF_REFILL_MINBLOCKS
#define ERT_WF_REFILL_MINBLOCKS 4
#endif
// EMIT: rays whose walk is over do not leave their result in HBM for wf_emit_hits; the hits wait in a small
// per-warp queue and, 32 at a time, one per lane, become hit records (location and normal in FP64 on a full warp,
// one atomic per 32 hits, coalesced record stores).
struct alignas(16) FinishedHit {
    double t;
    unsigned int idx;           // entry of the path queue
    int obj;
};
constexpr int kFinQueue = 64;   // up to 31 waiting + 32 lanes finishing in one step
template <bool COUNT, bool GRID, bool EMIT, bool TRI = false>
__global__ void __launch_bounds__(kWfThreads, GRID ? ERT_GRID_MINBLOCKS : ERT_WF_REFILL_MINBLOCKS)
wf_trace_path_refill(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
                     const __grid_constant__ WfBuf wf, int bounce)
{
    __shared__ double slots[kRaySlotDoubles][kWfThreads];
    __shared__ FinishedHit fin_all[EMIT ? kWfThreads / 32 : 1][EMIT ? kFinQueue : 1];
    FinishedHit *fin = fin_all[EMIT ? (threadIdx.x >> 5) : 0];
    int n_fin = 0;                                   // the same in every lane
    RaySlot ray;
    ray.p = &slots[0][threadIdx.x];
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned long long n = (unsigned long long)wf.ctr[(bounce - 1) * kWfCtr + WF_NNEXT];
    unsigned long long *cursor = reinterpret_cast<unsigned long long *>(ctr + WF_FETCH_PATH);
    const int lane = threadIdx.x & 31;
    Tally<COUNT> tl;
    unsigned int rays = 0;
    bool have = false;
    unsigned long long pos = 0, end = 0;             // the warp's current chunk
    bool drained = false;                            // no chunk left in the queue
    unsigned int idx = 0;
    SRay f;
    Hit best;
    best.obj = -1; best.t = 0.0; best.order = 0x7fffffff;
    Trav<false> tr;
    int stack[GRID ? 1 : kBvhStack];
    tr.node = kTravDone; tr.sp = 0; tr.cullk = 0.f;
    GridWalk gw;
    GridRay gr;
    gw.id = -1;
    // turns the first `take` queued hits into hit records, one per lane (erl:384-390, 443-451, 471-476)
    auto emit_finished = [&](int take) {
        __syncwarp();
        {
            const bool hit = lane < take;
            d3 P = mk(0, 0, 0), N = P, D = P;
            double W = 0.0;
            int pid = 0, obj = -1, order = 0;
            if (hit) {
                const FinishedHit fh = fin[lane];
                d3 O;
                bool valid;
                path_ray_of_index(fp, wf, false, fh.idx, O, D, pid, valid, &W);
                obj = fh.obj;
                order = object_order(sc, obj);
                P = vadd(O, vscale(D, fh.t));
                N = hit_normal(sc, obj, P);
            }
            emit_hits_and_rays(sc, fp, wf, bounce, ctr, lane, hit, P, N, D, obj, order, pid, W);
        }
        __syncwarp();
        FinishedHit keep;
        keep.t = 0.0; keep.idx = 0u; keep.obj = -1;
        if (take + lane < n_fin) keep = fin[take + lane];
        __syncwarp();
        if (take + lane < n_fin) fin[lane] = keep;
        n_fin -= take;
        __syncwarp();
    };
    for (;;) {
        const unsigned int idle = __ballot_sync(0xffffffffu, !have);
        if (32 - __popc(idle) < kRefillBelow && !drained) {
            if (pos >= end) {
                if (!next_chunk(cursor, n, lane, pos, end)) { drained = true; pos = end = 0; }
                else prefetch_path_chunk(wf, pos, end, lane);
            }
            if (pos < end) {
                const unsigned long long i64 = pos + (unsigned long long)rank_in(idle, lane);
                const unsigned long long adv = pos + (unsigned long long)__popc(idle);
                pos = adv < end ? adv : end;
                if (!have && i64 < end) {
                    const unsigned int i = (unsigned int)i64;
                    bool valid;
                    int pid;
                    d3 O = mk(0, 0, 0), D = mk(0, 0, 1);
                    path_ray_of_index(fp, wf, false, i, O, D, pid, valid);
                    idx = i;
                    rays++;
                    best.obj = -1; best.t = 0.0; best.order = 0x7fffffff;
                    scan_others<COUNT, TRI>(sc, O, D, best, -1, tl);
                    if (sc.n_spheres > 0) {
                        double a, inv;
                        const bool filtered = make_sray(sc, O, D, f, a, inv);
                        ray.put(O, D, a, inv);
                        if constexpr (GRID) {
                            if (f.m4 <= sc.cg.eps) {
                                float cullk = cullk_from(f, inv, best);
                                grid_big_spheres<COUNT>(sc, f, ray, -1, best, cullk, tl);
                                grid_start(gw, gr, sc, f, cullk);
                            } else {
                                Hit tmp = best;
                                walk_bvh_instead(&sc, ray.p, -1, &tmp);
                                best = tmp;
                                gw.id = -1;                  // the first step reports the ray as done
                            }
                        } else if (!filtered) {
                            best = scan_spheres_instead(&sc, O, D, best, -1, false, -1);
                            tr.node = kTravDone;             // the first step reports the ray as done
                        } else {
                            trav_start(tr, stack, f, inv, best);
                        }
                    } else {
                        // no spheres: the first step below reports the ray as done (planes and triangles are in `best`)
                        gw.id = -1;
                        tr.node = kTravDone;
                    }
                    have = true;
                }
            }
        }
        if (!__any_sync(0xffffffffu, have)) {
            if (drained) break;
            continue;
        }
        for (;;) {
            bool over = false;
            if constexpr (GRID) {
                // the lanes walk to their next cell with spheres and filter them on their own, then meet
                // for the FP64 tests of the survivors
                unsigned int surv = 0u, obase = 0u;
                int cell = 0;
                float te = 0.f;
                bool found = false;
                if (have) found = grid_find<COUNT>(gw, gr, sc, ray, f, best, -1, tl, surv, cell, obase, te);
                __syncwarp();
                if (surv) grid_exact<COUNT>(sc, f, ray, cell, obase, surv, -1, best, gw.cullk, tl);
                if (have) over = found ? grid_leave(gw, te) : true;
            } else {
                if (have) over = trav_step<false, COUNT>(tr, stack, sc, ray, f, best, -1, -1, tl);
            }
            if constexpr (EMIT) {
                const bool fin_hit = over && best.obj >= 0;
                const unsigned int fm = __ballot_sync(0xffffffffu, fin_hit);
                if (fm) {
                    if (fin_hit) {
                        FinishedHit fh;
                        fh.t = best.t; fh.idx = idx; fh.obj = best.obj;
                        fin[n_fin + rank_in(fm, lane)] = fh;
                    }
                    n_fin += __popc(fm);
                    if (n_fin >= 32) emit_finished(32);
                }
                if (over) have = false;
            } else if (over) {
                __stcs(wf.res_hit + idx, make_int2(best.obj, hit_order(sc, best)));
                __stcs(wf.res_t + idx, best.t);
                have = false;
            }
            const int act = __popc(__ballot_sync(0xffffffffu, have));
            if (act == 0 || (!drained && act < kRefillBelow)) break;
        }
    }
    if constexpr (EMIT) {
        if (n_fin > 0) emit_finished(n_fin);
    }
    flush_counters<COUNT>(fp, (int)rays, tl);
}

// Turns the nearest-hit results of one bounce into the hit queue: hit location and normal
// (erl:384-390, 443-451, 471-476), compaction, and (SORT) the cell histogram for the binning.
template <bool FIRST, bool SORT>
__global__ void __launch_bounds__(kWfThreads)
wf_emit_hits(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
             const __grid_constant__ WfBuf wf, int bounce)
{
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned int n = FIRST ? (unsigned int)wf.n_pad : wf.ctr[(bounce - 1) * kWfCtr + WF_NNEXT];
    const int lane = threadIdx.x & 31;
    const unsigned int warp = (blockIdx.x * kWfThreads + threadIdx.x) >> 5;
    const unsigned int n_warps = (gridDim.x * kWfThreads) >> 5;
    HitHead *out_head = SORT ? wf.raw_head : wf.hit_head;
    HitTail *out_tail = SORT ? wf.raw_tail : wf.hit_tail;
    // A warp takes kEmitBatches batches of 32 entries per round and reserves their hit slots with ONE
    // atomic: every warp of the grid adds to the same counter, and at one atomic per 32 entries the
    // launch waited on that address more than on memory.
    constexpr int kEmitBatches = 4;
    for (unsigned long long base = (unsigned long long)warp * (32 * kEmitBatches); base < n;
         base += (unsigned long long)n_warps * (32 * kEmitBatches)) {
        int2 r[kEmitBatches];
        unsigned int m[kEmitBatches];
        unsigned int total = 0;
#pragma unroll
        for (int k = 0; k < kEmitBatches; k++) {
            const unsigned long long i64 = base + (unsigned long long)(32 * k + lane);
            r[k] = make_int2(-1, 0);
            if (i64 < n) r[k] = wf.res_hit[(unsigned int)i64];
            m[k] = __ballot_sync(0xffffffffu, r[k].x >= 0);
            total += __popc(m[k]);
        }
        if (!total) continue;
        unsigned int slot0 = 0;
        if (lane == 0) slot0 = atomicAdd(ctr + WF_NHITS, total);
        slot0 = __shfl_sync(0xffffffffu, slot0, 0);
#pragma unroll
        for (int k = 0; k < kEmitBatches; k++) {
            const bool hit = r[k].x >= 0;
            d3 P = mk(0, 0, 0), N = P, D = P;
            double W = 0.0;
            int pid = 0;
            if (hit) {
                const unsigned int i = (unsigned int)base + (unsigned int)(32 * k + lane);
                d3 O;
                bool valid;
                path_ray_of_index(fp, wf, FIRST, i, O, D, pid, valid);
                double t = wf.res_t[i];
                P = vadd(O, vscale(D, t));                            // erl:384-387 / 443-447 / 471-475
                N = hit_normal(sc, r[k].x, P);
                W = path_weight_of_index(wf, FIRST, i);
                size_t s = slot0 + rank_in(m[k], lane);
                write_hit(out_head, out_tail, s, P, N, D, r[k].x, r[k].y, pid, W);
                if constexpr (SORT) {
                    unsigned int key = sort_cell(sc, P);
                    wf.r_key[s] = key;
                    atomicAdd(wf.hist + key, 1u);
                }
            }
            if (m[k]) emit_next_rays(sc, fp, wf, bounce, ctr, lane, hit, P, N, D, r[k].x, pid, W);
            slot0 += __popc(m[k]);
        }
    }
}

// shadow_factor/4 (erl:256-267) of every (light, hit) pair of one bounce, light-major so that a
// warp holds rays that leave one light towards neighbouring hit locations.  A ray is first tried
// against the sphere that shadowed this lane's previous ray: any object that beats the target's
// (t, order) settles the question (erl:263), so a neighbour's occluder usually ends the query
// without a walk.
template <bool COUNT, bool USE_GRID, bool TRI = false>
__global__ void __launch_bounds__(kWfThreads, ERT_SHADOW_MINBLOCKS)
wf_trace_shadow(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
                const __grid_constant__ WfBuf wf, int bounce)
{
    __shared__ double slots[kRaySlotDoubles][kWfThreads];
    RaySlot ray;
    ray.p = &slots[0][threadIdx.x];
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned int n_hits = ctr[WF_NHITS];
    const unsigned long long total = (unsigned long long)n_hits * (unsigned long long)sc.n_lights;
    unsigned long long *cursor = reinterpret_cast<unsigned long long *>(ctr + WF_FETCH_SHADOW);
    const int lane = threadIdx.x & 31;
    const size_t np = (size_t)wf.n_pad;
    Tally<COUNT> tl;
    unsigned int rays = 0;
    int hint = -1;                                   // sphere that shadowed this lane's previous ray
    // the warp's recent occluders: filter sphere + index, a ring the whole warp reads by broadcast
    __shared__ float4 occ_f_all[kWfThreads / 32][kOccCache];
    __shared__ int occ_i_all[kWfThreads / 32][kOccCache];
    float4 *occ_f = occ_f_all[threadIdx.x >> 5];
    int *occ_i = occ_i_all[threadIdx.x >> 5];
    for (int k = lane; k < kOccCache; k += 32) {
        occ_f[k] = make_float4(0.f, 0.f, 0.f, -3.0e38f);       // never passes the filter
        occ_i[k] = -1;
    }
    int occ_head = 0;
    __syncwarp();
    unsigned long long begin, end;
    while (next_chunk(cursor, total, lane, begin, end)) {
        for (unsigned long long b0 = begin; b0 < end; b0 += 32) {
            const unsigned long long j = b0 + lane;
            int found = -1;                          // sphere a walk of this batch found in the way
            if (j < end) {
            unsigned int l, h;
            if (total <= 0xffffffffull) {
                l = (unsigned int)j / n_hits;
                h = (unsigned int)j - l * n_hits;
            } else {
                l = (unsigned int)(j / n_hits);
                h = (unsigned int)(j - (unsigned long long)l * n_hits);
            }
            rays++;
            bool lit = false;
            {
                const double4 r0 = ld_rec32(wf.hit_head + h);
                // the next batch's record (same light, 32 hits on) and this target's FP64 sphere: on their
                // way to L1 while the direction is normalised
                if (h + 32u < n_hits) prefetch_l1(wf.hit_head + h + 32u);
                d3 P = mk(r0.x, r0.y, r0.z);
                const int target = (int)(__double_as_longlong(r0.w) & 0xffffffffll);
                const int order = (int)(__double_as_longlong(r0.w) >> 32);
                if (obj_type(target) == OBJ_SPHERE) prefetch_l1(sc.sph_exact + obj_index(target));
                const double *lt = sc.lights + 9 * (size_t)l;
                d3 O = mk(lt[3], lt[4], lt[5]);
                d3 D = vnormalize(vsub(P, O));                     // erl:257-260
                double a = D.x * D.x + D.y * D.y + D.z * D.z;
                double t;
                // "nearest == Object" (erl:263) <=> Object is hit and nothing beats its (t, order)
                if (object_exact(sc, target, O, D, a, t)) {
                    Hit best;
                    best.t = t; best.order = order; best.obj = target;
                    scan_others_shadow<COUNT, TRI>(sc, O, D, best, target, tl);
                    lit = best.obj == target;
                    if (lit && hint >= 0 && obj_code(OBJ_SPHERE, hint) != target) {
                        double th;
                        TALLY(exact_sph);
                        if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + hint), th) && better(th, sc.sph_order[hint], best))
                            lit = false;
                    }
                    if (lit && sc.n_spheres > 0 && USE_GRID && l < (unsigned int)sc.lg_count) {
                        // this light has a direction grid: a few candidates, no walk
                        SRay f;
                        double a2, inv;
                        if (make_sray(sc, O, D, f, a2, inv))
                            lit = !light_grid_occluded<COUNT>(sc, sc.lgrids[l], f, O, D, a, inv, best, target, tl);
                        else
                            lit = scan_spheres_instead(&sc, O, D, best, target, true, target).obj == target;
                    } else if (lit && sc.n_spheres > 0) {
                        SRay f;
                        double a2, inv;
                        const bool filtered = make_sray(sc, O, D, f, a2, inv);
                        // the warp's recent occluders, FP32 filter first (out of range it may drop one: the literal
                        // scan below finds it)
                        const float cull0 = cullk_from(f, inv, best);
                        for (int k = 0; k < kOccCache && lit; k++) {
                            const float4 fs = occ_f[k];
                            float fb, fv;
                            TALLY(filter);
                            if (filter_stage1(f, fs, fb, fv) && filter_stage2(f, fs, fb, fv, cull0)) {
                                const int sph = occ_i[k];
                                if (obj_code(OBJ_SPHERE, sph) != target) {
                                    double th;
                                    TALLY(exact_sph);
                                    if (sphere_exact(O, D, a, ld_sphere(sc.sph_exact + sph), th) && better(th, sc.sph_order[sph], best)) {
                                        lit = false;
                                        hint = sph;
                                    }
                                }
                            }
                        }
                        if (lit && !filtered) {
                            best = scan_spheres_instead(&sc, O, D, best, target, true, target);
                            lit = best.obj == target;
                        } else if (lit) {
                            ray.put(O, D, a2, inv);
                            Trav<true> tr;
                            int stack[kBvhStack];
                            trav_start(tr, stack, f, inv, best);
                            while (!trav_step<true, COUNT>(tr, stack, sc, ray, f, best, target, target, tl)) { }
                            lit = best.obj == target;
                            if (!lit && obj_type(best.obj) == OBJ_SPHERE) { hint = obj_index(best.obj); found = hint; }
                        }
                    }
                }
            }
            wf.lit[(size_t)l * np + h] = lit;
            }
            // new occluders enter the warp's ring (one lane per distinct sphere)
            const unsigned int fm = __ballot_sync(0xffffffffu, found >= 0);
            if (fm) {
                bool ins = false;
                if (found >= 0) {
                    const unsigned int same = __match_any_sync(fm, found);
                    ins = (__ffs(same) - 1) == lane;
                }
                const unsigned int im = __ballot_sync(0xffffffffu, ins);
                __syncwarp();
                if (ins) {
                    const int slot = (occ_head + rank_in(im, lane)) % kOccCache;
                    occ_f[slot] = __ldg(sc.sph_filter + found);
                    occ_i[slot] = found;
                }
                occ_head = (occ_head + __popc(im)) % kOccCache;
                __syncwarp();
            }
        }
    }
    flush_counters<COUNT>(fp, (int)rays, tl);
}

// Folds the lights of every hit of one bounce into the pixel's colour (erl:209-252 in forward form, see
// pix_consume).  The reflection rays of the next bounce were emitted with the hits (emit_next_rays).
__global__ void __launch_bounds__(kWfThreads, ERT_SHADE_MINBLOCKS)
wf_shade(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
         const __grid_constant__ WfBuf wf, int bounce)
{
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned int n_hits = ctr[WF_NHITS];
    const int lane = threadIdx.x & 31;
    const unsigned int warp = (blockIdx.x * kWfThreads + threadIdx.x) >> 5;
    const unsigned int n_warps = (gridDim.x * kWfThreads) >> 5;
    const size_t np = (size_t)wf.n_pad;
    const int L = sc.n_lights;
    for (unsigned long long base = (unsigned long long)warp * 32; base < n_hits; base += (unsigned long long)n_warps * 32) {
        size_t h = (size_t)base + lane;
        bool valid = h < n_hits;
        int pid = 0;
        d3 P = mk(0, 0, 0), N = P, D = P;
        if (valid) {
            HitHead hh;
            HitTail ht;
            {
                const uint4 *sh = reinterpret_cast<const uint4 *>(wf.hit_head + h);
                const uint4 *st = reinterpret_cast<const uint4 *>(wf.hit_tail + h);
                uint4 *dh = reinterpret_cast<uint4 *>(&hh);
                uint4 *dt = reinterpret_cast<uint4 *>(&ht);
                dh[0] = sh[0]; dh[1] = sh[1];
                dt[0] = st[0]; dt[1] = st[1]; dt[2] = st[2]; dt[3] = st[3];
            }
            pid = ht.pid;
            P = mk(hh.P[0], hh.P[1], hh.P[2]);
            N = mk(ht.N[0], ht.N[1], ht.N[2]);
            D = mk(ht.D[0], ht.D[1], ht.D[2]);
            const double *mat = material_ptr(sc, hh.obj);
            d3 S = mk(0.0, 0.0, 0.0);
            for (int l = 0; l < L; l++) {
                if (wf.lit[(size_t)l * np + h]) S = vadd(S, light_term(sc.lights + 9 * (size_t)l, mat, P, N, D));
            }
            d3 Cold = mk(0.0, 0.0, 0.0);
            if (bounce > 0) Cold = mk(wf.C[pid], wf.C[np + pid], wf.C[2 * np + pid]);
            const d3 Cnew = vadd(Cold, vscale(S, ht.W));
            wf.C[pid] = Cnew.x; wf.C[np + pid] = Cnew.y; wf.C[2 * np + pid] = Cnew.z;
        }
    }
}

// ------------------------------------------------------------------ shadow rays: FP32 triage
// Most shadow rays of a crowded scene are blocked, and nearly always by the nearest sphere of their direction
// cell.  shadow_blocked() proves that in FP32 where it can: the light's ray towards the hit certainly meets the
// cell's first candidate S (impact parameter by cross product, so the error grows with the distance from the
// light, not with its square), S's reference Distance certainly lies below the target's, and therefore
// "nearest == Object" (erl:263) is false whatever else the scan finds — no FP64 normalise, no literal tests.
// It answers true only with every rounding of its own arithmetic AND of the reference's FP64 evaluation inside
// the margins below; everything else (lit rays, near ties, grazing rays, awkward geometry) is left to the
// literal path.
//
// Frame: the light O is the origin.  With u = 2^-24, rho = |C - O|, L = |P - O|:
//   direction  df = fl(P - O) normalised in FP32 (products, sums, rsqrtf <= 2 ulp): |df - D^| <= 7.4u  (12u used)
//   centre     cf - fl(O): |error| <= eta_c + sqrt(3) u |O|_inf + u rho =: ec
//   impact     q = (C - O) x D^;  |qf - q| <= ec + 17u rho                      (24u rho used)
//   along      b = (C - O) . D^;  |bf - b| <= ec + 12.6u rho                    (24u rho used)
//   radius     R = fl_up(r^2 (1 + 2^-18) + pad_c), so r^2 >= (R - pad_c_max)(1 - 2^-17) - 8uR
// Reference (erl:364-397, A = D.D = 1 +- 1e-15): Discriminant = 4A(r^2 - q^2) >= 0.001, T = b - sqrt(r^2 - q^2),
// both roots >= 0 iff the origin is outside and b > 0; its FP64 evaluation moves Discriminant by <= 5e-15 rho^2 and
// T by <= 6e-14 rho^2 once Discriminant >= 0.0016: the 1e-12 rho^2 terms cover both.
__device__ __forceinline__ unsigned int light_cell_of(float dx, float dy, float dz, int res)
{
    const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
    int m = 0;
    float am = ax, dm = dx, du = dy, dv = dz;
    if (ay > am) { m = 1; am = ay; dm = dy; du = dz; dv = dx; }
    if (az > am) { m = 2; am = az; dm = dz; du = dx; dv = dy; }
    const int face = 2 * m + (dm < 0.0f ? 1 : 0);
    const float inv = __frcp_rn(am);
    const float u = du * inv, v = dv * inv;
    const float half = 0.5f * (float)res;
    int iu = (int)floorf((u + 1.0f) * half), iv = (int)floorf((v + 1.0f) * half);
    iu = min(max(iu, 0), res - 1);
    iv = min(max(iv, 0), res - 1);
    return (unsigned int)((face * res + iv) * res + iu);
}
#ifndef ERT_TRIAGE_CANDS
#define ERT_TRIAGE_CANDS 4
#endif
constexpr int kTriageCands = ERT_TRIAGE_CANDS;   // candidates of a direction cell the triage looks at
#ifdef ERT_PROBE
__device__ unsigned long long g_sb_reason[8];
#define SB_REASON(k) atomicAdd(&g_sb_reason[k], 1ull)
#else
#define SB_REASON(k) do { } while (0)
#endif
__device__ __forceinline__ bool shadow_blocked(const DevScene &sc, const LightGridDev &lg, const double *lt, d3 P,
                                               int target, float4 tf)
{
    const float u = ERT_U;
    const float fx = (float)(P.x - lt[3]), fy = (float)(P.y - lt[4]), fz = (float)(P.z - lt[5]);
    const float l2 = fx * fx + fy * fy + fz * fz;
    if (!(l2 > 1e-20f && l2 < 1e20f)) return false;
    const float inv = rsqrtf(l2);
    const float dx = fx * inv, dy = fy * inv, dz = fz * inv;
    float c[8];
    ldg256(lg.head + light_cell_of(dx, dy, dz, lg.res), c);
    if (__float_as_int(c[4]) < 0) { SB_REASON(0); return false; }   // nothing listed in this direction
    const float ox = (float)lt[3], oy = (float)lt[4], oz = (float)lt[5];
    const float ec0 = 1.01f * (sc.eta_c_max + 1.75f * u * fmaxf(fmaxf(fabsf(ox), fabsf(oy)), fabsf(oz)));
    // lower bound of the target's Distance, should the ray meet the target at all
    float s_lo;
    if (obj_type(target) == OBJ_SPHERE) {
        const float tx = tf.x - ox, ty = tf.y - oy, tz = tf.z - oz;
        const float trho2 = tx * tx + ty * ty + tz * tz;
        const float tb = dx * tx + dy * ty + dz * tz;
        s_lo = tb - (ec0 + 26.f * u * sqrtf(trho2)) - sqrtf(tf.w) * (1.f + 4.f * u) - 4.f * u * fabsf(tb) - 1e-12f * trho2 - 1e-7f;
    } else if (obj_type(target) == OBJ_PLANE) {
        // the ray meets the plane where the hit lies (to the rounding of the hit location) unless it grazes it
        const double *pl = sc.planes + 4 * obj_index(target);
        const float nx = (float)pl[0], ny = (float)pl[1], nz = (float)pl[2];
        const float nd = nx * dx + ny * dy + nz * dz;
        if (!(fabsf(nd) > 1e-3f * sqrtf(nx * nx + ny * ny + nz * nz))) return false;
        s_lo = l2 * inv * (1.f - 1e-5f) - 1e-7f;
    } else {
        return false;
    }
    // the candidates of the cell, nearest first, until one certainly blocks the ray or the rest lie beyond the target
    unsigned int e = __float_as_uint(c[6]);
    const unsigned int e1 = __float_as_uint(c[7]);
#pragma unroll 1
    for (int tries = 0; tries < kTriageCands; tries++) {
        if (c[5] > s_lo) { SB_REASON(1); return false; }             // dmin: this and all later ones are too far
        const float cx = c[0] - ox, cy = c[1] - oy, cz = c[2] - oz, R = c[3];
        const int sph = __float_as_int(c[4]);
        const bool more = e < e1;
        if (more) ldg256(lg.cand + e, c);                            // in flight while this candidate is tested
        e++;
        if (obj_code(OBJ_SPHERE, sph) != target) {
            const float rho2 = cx * cx + cy * cy + cz * cz;
            const float rho = sqrtf(rho2);
            const float b = dx * cx + dy * cy + dz * cz;
            const float qx = cy * dz - cz * dy, qy = cz * dx - cx * dz, qz = cx * dy - cy * dx;
            const float err = ec0 + 26.f * u * rho;                  // bounds both |qf - q| and |bf - b|
            const float qmax = sqrtf(qx * qx + qy * qy + qz * qz) * (1.f + 8.f * u) + err;
            const float fp64_noise = 1e-12f * rho2;
            // lower bound of r^2 - q^2, its own roundings taken off
            const float T = ((R - sc.pad_c_max) * (1.f - 7.62939453125e-6f) - 8.f * u * R) - qmax * qmax * (1.f + 4.f * u) - 8.f * u * R;
            // Discriminant >= 0.001 with room to spare; the light is outside S and S lies ahead
            if (T > 0.0004f + fp64_noise && b - err > sqrtf(R) * (1.f + 4.f * u)) {
                float s_up = b + err - sqrtf(T) * (1.f - 4.f * u);               // >= the reference's Distance of S ...
                s_up += 4.f * u * b + 4e-6f * fabsf(s_up) + fp64_noise + 1e-7f;  // ... and its evaluation
                if (s_up < s_lo) return true;
            }
        }
        if (!more) { SB_REASON(2); return false; }
    }
    SB_REASON(3);
    return false;
}

// shadow_factor/4 and the light fold in ONE pass over the hits, for scenes whose lights all have a direction grid
// (no walk, no per-warp occluder ring).  A warp takes a chunk of up to 128 hits and goes through it in three
// phases, each of which packs its work over the lanes first:
//   1. triage: every (hit, light) pair goes through shadow_blocked(); the pairs it cannot settle are listed in
//      shared memory;
//   2. the listed pairs, 32 at a time and one per lane whatever hit they belong to, take the literal path
//      (FP64 direction, the target's literal test — "nearest == Object" needs the target hit —, planes and
//      triangles, the candidates of the direction cell) and mark the lights that reach their hit;
//   3. the hits some light reaches, again 32 at a time, fold those lights into their pixel in list order
//      (erl:209-252 in forward form, wf_shade's arithmetic).
// The shadow factors never travel through HBM, and the FP64 work runs on nearly full warps although only a
// third of the rays and a third of the hits need it.
#ifndef ERT_SS_MINBLOCKS
#define ERT_SS_MINBLOCKS 4
#endif
constexpr int kSsMaxLights = 8;                  // three bits of a pair's entry; ert_api.cu uses the kernel for <= 8 lights
static_assert(kWfChunk <= 128, "a chunk's hits are numbered with seven bits");
template <bool COUNT, bool TRI = false>
__global__ void __launch_bounds__(kWfThreads, ERT_SS_MINBLOCKS)
wf_shadow_shade(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp,
                const __grid_constant__ WfBuf wf, int bounce)
{
    __shared__ unsigned int sh_lit_all[kWfThreads / 32][kWfChunk];                      // lights that reach each hit
    __shared__ unsigned short sh_list_all[kWfThreads / 32][kWfChunk * kSsMaxLights];   // open pairs: slot << 3 | light; then lit slots
    unsigned int *sh_lit = sh_lit_all[threadIdx.x >> 5];
    unsigned short *sh_list = sh_list_all[threadIdx.x >> 5];
    unsigned int *ctr = wf.ctr + bounce * kWfCtr;
    const unsigned int n_hits = ctr[WF_NHITS];
    unsigned long long *cursor = reinterpret_cast<unsigned long long *>(ctr + WF_FETCH_SHADOW);
    const int lane = threadIdx.x & 31;
    const size_t np = (size_t)wf.n_pad;
    const int L = sc.n_lights;
    Tally<COUNT> tl;
    unsigned int rays = 0;
    unsigned long long begin, end;
    // appends `mine` entries of this lane to the list (every lane calls); returns where this lane's entries start
    auto reserve = [&](int mine, int &n_list) -> int {
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        const int at = n_list + incl - mine;
        n_list += __shfl_sync(0xffffffffu, incl, 31);
        return at;
    };
    while (next_chunk(cursor, (unsigned long long)n_hits, lane, begin, end)) {
        const int nb = (int)(end - begin);
        // ---- 1. triage
        int n_list = 0;
        for (int s0 = 0; s0 < nb; s0 += 32) {
            const int slot = s0 + lane;
            unsigned int open = 0u;                                  // lights whose ray the triage could not settle
            if (slot < nb) {
                const double4 r0 = ld_rec32(wf.hit_head + begin + slot);
                rays += (unsigned int)L;
                sh_lit[slot] = 0u;
                const d3 P = mk(r0.x, r0.y, r0.z);
                const int target = (int)(__double_as_longlong(r0.w) & 0xffffffffll);
                float4 tf = make_float4(0.f, 0.f, 0.f, 0.f);
                if (obj_type(target) == OBJ_SPHERE) tf = __ldg(sc.sph_filter + obj_index(target));
                for (int l = 0; l < L; l++) {
                    if (!shadow_blocked(sc, sc.lgrids[l], sc.lights + 9 * (size_t)l, P, target, tf)) open |= 1u << l;
                }
            }
            int at = reserve(__popc(open), n_list);
            WF_ASSERT(n_list <= (int)(kWfChunk * kSsMaxLights) && nb <= (int)kWfChunk, "list %d chunk %d", n_list, nb);
            while (open) {
                const int l = __ffs((int)open) - 1;
                open &= open - 1u;
                sh_list[at++] = (unsigned short)((slot << 3) | l);
            }
        }
        PROBE(0, lane == 0 ? (unsigned int)n_list : 0u);
        __syncwarp();
        // ---- 2. the literal path for the open pairs
        for (int k0 = 0; k0 < n_list; k0 += 32) {
            const int k = k0 + lane;
            if (k < n_list) {
                const unsigned int pr = sh_list[k];
                const int slot = (int)(pr >> 3), l = (int)(pr & 7u);
                WF_ASSERT(slot < nb && l < L, "pair %u of chunk %d, %d lights", pr, nb, L);
                const double4 q0 = ld_rec32(wf.hit_head + begin + slot);
                const d3 Ph = mk(q0.x, q0.y, q0.z);
                const int tgt = (int)(__double_as_longlong(q0.w) & 0xffffffffll);
                const int order = (int)(__double_as_longlong(q0.w) >> 32);
                const double *lt = sc.lights + 9 * (size_t)l;
                const d3 O = mk(lt[3], lt[4], lt[5]);
                const d3 D = vnormalize(vsub(Ph, O));                  // erl:257-260
                const double a = D.x * D.x + D.y * D.y + D.z * D.z;
                double t;
                // "nearest == Object" (erl:263) <=> Object is hit and nothing beats its (t, order)
                if (object_exact(sc, tgt, O, D, a, t)) {
                    Hit best;
                    best.t = t; best.order = order; best.obj = tgt;
                    scan_others_shadow<COUNT, TRI>(sc, O, D, best, tgt, tl);
                    bool lit = best.obj == tgt;
                    if (lit && sc.n_spheres > 0) {
                        SRay f;
                        double a2, inv;
                        if (make_sray(sc, O, D, f, a2, inv))
                            lit = !light_grid_occluded<COUNT>(sc, sc.lgrids[l], f, O, D, a, inv, best, tgt, tl);
                        else
                            lit = scan_spheres_instead(&sc, O, D, best, tgt, true, tgt).obj == tgt;
                    }
                    if (lit) atomicOr(sh_lit + slot, 1u << l);
                    PROBE(2, lit ? 1u : 0u);
                }
            }
        }
        __syncwarp();
        // ---- 3. the fold.  A hit no light reaches adds S * W = (0,0,0) * W to its pixel: the colour buffer starts at
        // +0.0 and a sum that starts there is never -0.0, so for any finite W the addition changes no bit and the
        // record's tail stays unread.  (A non-finite W needs a reflectivity beyond 1e60: BEAM floats cannot hold the
        // products the reference would form with it, erl:239-247 raises badarith long before.)
        n_list = 0;
        for (int s0 = 0; s0 < nb; s0 += 32) {
            const int slot = s0 + lane;
            const bool any = slot < nb && sh_lit[slot] != 0u;
            const int at = reserve(any ? 1 : 0, n_list);
            if (any) sh_list[at] = (unsigned short)slot;
        }
        __syncwarp();
        for (int k0 = 0; k0 < n_list; k0 += 32) {
            const int k = k0 + lane;
            if (k < n_list) {
                const int slot = (int)sh_list[k];
                WF_ASSERT(slot < nb, "slot %d of chunk %d", slot, nb);
                const unsigned int litmask = sh_lit[slot];
                const size_t h = (size_t)begin + slot;
                const double4 q0 = ld_rec32(wf.hit_head + h);
                const d3 P = mk(q0.x, q0.y, q0.z);
                const int target = (int)(__double_as_longlong(q0.w) & 0xffffffffll);
                HitTail ht;
                {
                    const double4 t0 = ld_rec32(wf.hit_tail + h), t1 = ld_rec32(reinterpret_cast<const char *>(wf.hit_tail + h) + 32);
                    double4 *dt = reinterpret_cast<double4 *>(&ht);
                    dt[0] = t0; dt[1] = t1;
                }
                const int pid = ht.pid;
                d3 S = mk(0.0, 0.0, 0.0);
                const d3 N = mk(ht.N[0], ht.N[1], ht.N[2]);
                const d3 Dp = mk(ht.D[0], ht.D[1], ht.D[2]);
                const double *mat = material_ptr(sc, target);
                for (int l = 0; l < L; l++) {
                    if (litmask & (1u << l)) S = vadd(S, light_term(sc.lights + 9 * (size_t)l, mat, P, N, Dp));
                }
                d3 Cold = mk(0.0, 0.0, 0.0);
                if (bounce > 0) Cold = mk(wf.C[pid], wf.C[np + pid], wf.C[2 * np + pid]);
                const d3 Cnew = vadd(Cold, vscale(S, ht.W));
                wf.C[pid] = Cnew.x; wf.C[np + pid] = Cnew.y; wf.C[2 * np + pid] = Cnew.z;
            }
        }
        __syncwarp();
    }
    flush_counters<COUNT>(fp, (int)rays, tl);
}

__global__ void __launch_bounds__(kWfThreads)
wf_finalize(const __grid_constant__ FrameParams fp, const __grid_constant__ WfBuf wf)
{
    const size_t np = (size_t)wf.n_pad;
    for (size_t i = (size_t)blockIdx.x * kWfThreads + threadIdx.x; i < np; i += (size_t)gridDim.x * kWfThreads) {
        int X, ly, Y;
        bool inside;
        pixel_of_index(fp, wf, (int)i, X, ly, Y, inside);
        if (!inside) continue;
        Pix p;
        p.C = mk(wf.C[i], wf.C[np + i], wf.C[2 * np + i]);
        pix_store(p, fp, X, ly);
    }
}

}  // namespace ert
