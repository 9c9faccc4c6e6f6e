// Brute-force scan (ERT_ACCEL_LINEAR past one resident tile): the GPU's own statement of the
// reference's linear scan (erl:300-346), and the kernel the FP32-issue roofline is about.
//
// Every ray tests EVERY sphere with the conservative FP32 filter (DESIGN.md "Filter bounds"):
// 10 FP32-pipe lane-instructions per (ray, sphere).  What bounds the kernel is the dispatch port of
// the SM sub-partition (one warp instruction per clock; a packed FP32 instruction takes two), so
// everything that is not one of those ten is kept off the inner loop:
//
//   * packed FP32 (fma.rn.f32x2 / sub / mul -> FFMA2, FADD2, FMUL2): one instruction tests TWO spheres
//     for one ray.  The sphere list is stored pair-interleaved ({cx0,cx1,cy0,cy1},{cz0,cz1,R0,R1}), so
//     two broadcast LDS.128 feed kScanRays x 2 tests, the sphere operands are bank-aligned register
//     pairs and the ray operands use the scalar-broadcast form (`R.F32`): 6 registers per ray.  (The
//     scalar form of the same loop loses 10 % to register-bank conflicts, tools/scan_probe.cu.)
//   * kScanRays rays per thread share every LDS.128;
//   * a group of 16 spheres keeps only the largest stage-1 value per ray (one FMNMX3 per pair) and
//     ONE compare per ray decides whether any sphere of the group can pass (v >= -theta).  Only then —
//     a few groups per thousand — the warp looks closer, together: the ray's constants are
//     broadcast, 16 lanes run stage 1 on one sphere each, and the spheres that pass go into the
//     warp's candidate queue as (ray, sphere) pairs;
//   * the literal FP64 test (erl:364-397) runs on candidates, 32 at a time, one per lane — full warps
//     instead of one lane inside the loop — and folds into the ray's result with a 128-bit
//     compare-and-swap on {Distance, list position, object}: the (t, order) minimum of erl:319 does
//     not depend on the order in which candidates arrive.  Shadow rays (erl:256-267) set a flag;
//   * tiles of 512 spheres stream global -> shared through a ring of 1-D bulk async copies
//     (cp.async.bulk + mbarrier).  There is no block-wide barrier: the warp that is last to finish a
//     tile (a shared-memory counter tells it) refills that stage, so warps drift apart by up to
//     kScanStages - 1 tiles.
//
// Work split: the (ray batch) x (tile) space of a launch is linearised and cut into gridDim.x equal
// contiguous ranges, one short block each (several per resident slot, so an SM stays full until the
// grid drains) — a launch of 15 k rays over 1 M spheres fills the machine as well as one of 8 M rays
// over 10 k.  Planes, triangles (always FP64, erl:353-356) and the shadow targets are done once per
// ray by wf_scan_init before the scan; wf_scan_finish hands the results to the next stage.
#pragma once

#include "ert_wavefront.cuh"

namespace ert {

#ifndef ERT_SCAN_RAYS
#define ERT_SCAN_RAYS 4
#endif
#ifndef ERT_SCAN_MINBLOCKS
#define ERT_SCAN_MINBLOCKS 4
#endif
#ifndef ERT_SCAN_STAGES
#define ERT_SCAN_STAGES 4
#endif
constexpr int kScanThreads = 128;
constexpr int kScanWarps = kScanThreads / 32;
constexpr int kScanRays = ERT_SCAN_RAYS;                     // rays per thread
constexpr int kScanBatch = kScanThreads * kScanRays;         // rays per batch
constexpr int kScanTile = 512;                               // spheres per tile (8 KB)
constexpr int kScanStages = ERT_SCAN_STAGES;
constexpr int kScanGroup = 16;                               // spheres per pass decision (<= 32: one lane each)
constexpr int kScanQueue = 64;                               // candidate slots per warp
constexpr int kScanSmem = kScanStages * kScanTile * 16;
static_assert(kScanTile % kScanGroup == 0 && kScanGroup % 2 == 0 && kScanGroup <= 32, "tiles are whole groups of whole pairs");
static_assert(kScanQueue >= 32 + kScanGroup, "the queue takes one more group after a batch is due");

typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(u64 v, float &lo, float &hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 neg2(u64 a) { float lo, hi; upk2(a, lo, hi); return pk2(-lo, -hi); }
// {x, x} built where it is used (volatile: not hoisted out of the loop as a register pair), so that ptxas folds it
// into the scalar-broadcast operand form (`R.F32`) of FADD2/FMUL2/FFMA2: a ray costs 6 registers, not 12
__device__ __forceinline__ u64 bc2(float x) { u64 r; asm volatile("mov.b64 %0, {%1,%1};" : "=l"(r) : "f"(x)); return r; }
__device__ __forceinline__ void cas128(void *addr, u64 cl, u64 ch, u64 nl, u64 nh, u64 &ol, u64 &oh)
{
    asm volatile("{\n\t.reg .b128 c, n, o;\n\tmov.b128 c, {%3, %4};\n\tmov.b128 n, {%5, %6};\n\t"
                 "atom.global.cas.b128 o, [%2], c, n;\n\tmov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(ol), "=l"(oh) : "l"(addr), "l"(cl), "l"(ch), "l"(nl), "l"(nh) : "memory");
}

// rays of a launch: path queue of the bounce (FIRST: every pixel of the part) or (light, hit) pairs
template <bool SHADOW, bool FIRST>
__device__ __forceinline__ unsigned long long scan_ray_count(const DevScene &sc, const WfBuf &wf, int bounce, unsigned int &n_hits)
{
    n_hits = 0;
    if constexpr (SHADOW) {
        n_hits = wf.ctr[bounce * kWfCtr + WF_NHITS];
        return (unsigned long long)n_hits * (unsigned long long)sc.n_lights;
    } else {
        return FIRST ? (unsigned long long)wf.n_pad : (unsigned long long)wf.ctr[(bounce - 1) * kWfCtr + WF_NNEXT];
    }
}

// the ray of queue entry i, in FP64
template <bool SHADOW, bool FIRST>
__device__ __forceinline__ void scan_ray_of_index(const DevScene &sc, const FrameParams &fp, const WfBuf &wf,
                                                  unsigned long long i, unsigned int n_hits, d3 &O, d3 &D, bool &valid,
                                                  int &target, int &target_order, unsigned int &l, unsigned int &h)
{
    target = -1; target_order = 0; l = 0; h = 0;
    if constexpr (SHADOW) {
        l = (unsigned int)(i / n_hits);
        h = (unsigned int)(i - (unsigned long long)l * n_hits);
        const double4 r0 = ld_rec32(wf.hit_head + h);
        const d3 P = mk(r0.x, r0.y, r0.z);
        target = (int)(__double_as_longlong(r0.w) & 0xffffffffll);
        target_order = (int)(__double_as_longlong(r0.w) >> 32);
        const double *lt = sc.lights + 9 * (size_t)l;
        O = mk(lt[3], lt[4], lt[5]);
        D = vnormalize(vsub(P, O));                                 // erl:257-260
        valid = true;
    } else {
        int pid;
        path_ray_of_index(fp, wf, FIRST, (unsigned int)i, O, D, pid, valid);
    }
}

// Before the scan, once per ray: planes and triangles (FP64, erl:353-356) seed the path ray's result; a shadow
// ray's target is tested ("nearest == Object", erl:263, needs the target hit), its Distance kept for the
// candidates to beat, and planes/triangles in front of it settle the ray at once.
template <bool SHADOW, bool FIRST, bool COUNT, bool TRI = false>
__global__ void __launch_bounds__(256)
wf_scan_init(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp, const __grid_constant__ WfBuf wf,
             int bounce)
{
    unsigned int n_hits;
    const unsigned long long n = scan_ray_count<SHADOW, FIRST>(sc, wf, bounce, n_hits);
    Tally<COUNT> tl;
    unsigned int rays = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        d3 O = mk(0, 0, 0), D = mk(0, 0, 1);
        bool valid;
        int target, target_order;
        unsigned int l, h;
        scan_ray_of_index<SHADOW, FIRST>(sc, fp, wf, i, n_hits, O, D, valid, target, target_order, l, h);
        Hit best;
        best.obj = -1; best.t = 0.0; best.order = 0x7fffffff;
        if (valid) rays++;
        if constexpr (SHADOW) {
            const double a = D.x * D.x + D.y * D.y + D.z * D.z;
            double t = 0.0;
            bool occluded = true;
            if (object_exact(sc, target, O, D, a, t)) {
                best.t = t; best.order = target_order; best.obj = target;
                scan_others_shadow<COUNT, TRI>(sc, O, D, best, target, tl);
                occluded = best.obj != target;
            }
            wf.sp_occ[i] = occluded ? 1 : 0;
            wf.sp_t[i] = t;
        } else {
            if (valid) scan_others<COUNT, TRI>(sc, O, D, best, -1, tl);
            ScanBest b;
            b.t = best.t; b.order = best.order; b.obj = valid ? best.obj : -2;       // -2: no ray here (padding pixel)
            wf.sp_best[i] = b;
        }
    }
    flush_counters<COUNT>(fp, (int)rays, tl);
}

// The literal test of one candidate, one per lane (erl:364-397), folded into the ray's result.
template <bool SHADOW, bool FIRST>
__device__ __noinline__ void scan_resolve(const DevScene *scp, const FrameParams *fpp, const WfBuf *wfp, unsigned int n_hits,
                                          unsigned long long i, int sph)
{
    const DevScene &sc = *scp;
    d3 O = mk(0, 0, 0), D = mk(0, 0, 1);
    bool valid;
    int target, target_order;
    unsigned int l, h;
    if constexpr (SHADOW) {
        if (wfp->sp_occ[i]) return;                                  // settled already
    }
    scan_ray_of_index<SHADOW, FIRST>(sc, *fpp, *wfp, i, n_hits, O, D, valid, target, target_order, l, h);
    const int code = obj_code(OBJ_SPHERE, sph);
    if (SHADOW && code == target) return;
    const double a = D.x * D.x + D.y * D.y + D.z * D.z;
    double t;
    if (!sphere_exact(O, D, a, ld_sphere(sc.sph_exact + sph), t)) return;
    const int ord = sc.sph_order[sph];
    if constexpr (SHADOW) {
        Hit tg;
        tg.t = wfp->sp_t[i]; tg.order = target_order; tg.obj = target;
        if (better(t, ord, tg)) wfp->sp_occ[i] = 1;                 // something is nearer than the target: shadow factor 0
    } else {
        ScanBest *slot = wfp->sp_best + i;
        // The first look at the slot must be one atomic 128-bit read: two 64-bit loads can straddle another lane's
        // swap and pair the Distance 0.0 of "no hit yet" with the new object — a hit at distance 0 that nothing
        // beats, and the candidate would walk away.  A compare-and-swap whose new value equals its compare value
        // changes nothing and returns the whole record.
        u64 cx, cy;
        cas128(slot, 0ull, 0ull, 0ull, 0ull, cx, cy);
        for (;;) {
            Hit cb;
            cb.t = __longlong_as_double((long long)cx);
            cb.order = (int)(cy & 0xffffffffull);
            cb.obj = (int)(cy >> 32);
            if (!better(t, ord, cb)) return;
            u64 ol, oh;
            cas128(slot, cx, cy, (u64)__double_as_longlong(t), ((u64)(unsigned int)code << 32) | (u64)(unsigned int)ord, ol, oh);
            if (ol == cx && oh == cy) return;
            cx = ol; cy = oh;
        }
    }
}

// How a launch over n rays is cut (block b owns the linear range [begin(b), begin(b+1)) of (batch, tile) pairs)
struct ScanCut {
    unsigned long long W, G;
    unsigned int n_tiles;
    __device__ __forceinline__ ScanCut(unsigned long long n_rays, int n_spheres, unsigned int grid)
    {
        n_tiles = (unsigned int)((n_spheres + kScanTile - 1) / kScanTile);
        W = ((n_rays + kScanBatch - 1) / kScanBatch) * n_tiles;
        G = grid < W ? grid : W;                             // every block below G owns at least one tile
    }
    __device__ __forceinline__ unsigned long long begin(unsigned long long b) const { return b * W / G; }
};

template <bool SHADOW, bool FIRST, bool COUNT>
__global__ void __launch_bounds__(kScanThreads, ERT_SCAN_MINBLOCKS)
wf_scan(const __grid_constant__ DevScene sc, const __grid_constant__ FrameParams fp, const __grid_constant__ WfBuf wf,
        int bounce)
{
    extern __shared__ __align__(128) unsigned char scan_smem[];
    __shared__ __align__(8) uint64_t full[kScanStages];
    __shared__ unsigned int done[kScanStages];
    __shared__ uint2 cand_all[kScanWarps][kScanQueue];              // (ray, sphere)
    unsigned int n_hits;
    const unsigned long long n = scan_ray_count<SHADOW, FIRST>(sc, wf, bounce, n_hits);
    if (n == 0) return;
    const ScanCut cut(n, sc.n_spheres, gridDim.x);
    if (blockIdx.x >= cut.G) return;
    const unsigned long long lo = cut.begin(blockIdx.x), hi = cut.begin(blockIdx.x + 1ull);
    const unsigned int total = (unsigned int)(hi - lo);             // tiles this block streams
    const unsigned int n_tiles = cut.n_tiles;
    const float4 *pairs = sc.sph_pairs;
    float4 *ring = reinterpret_cast<float4 *>(scan_smem);
    const unsigned int tile0 = (unsigned int)(lo % n_tiles);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kScanStages; s++) { mbar_init(&full[s], 1); done[s] = 0u; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (unsigned int q = 0; q < (unsigned int)kScanStages && q < total; q++) {
            const unsigned int t = (tile0 + q) % n_tiles;
            mbar_expect_tx(&full[q], kScanTile * 16u);
            bulk_g2s(ring + (size_t)q * kScanTile, pairs + (size_t)t * kScanTile, kScanTile * 16u, &full[q]);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float kInf = __int_as_float(0x7f800000);
    uint2 *cand = cand_all[warp];
    int n_cand = 0;                                                  // the same in every lane of the warp
    Tally<COUNT> tl;
    // runs the literal tests of the first `take` candidates of the queue, one per lane
    auto drain = [&](int take) {
        __syncwarp();
        if (lane < take) {
            const uint2 c = cand[lane];
            if constexpr (COUNT) tl.exact_sph++;
            scan_resolve<SHADOW, FIRST>(&sc, &fp, &wf, n_hits, (unsigned long long)c.x, (int)c.y);
        }
        __syncwarp();
        uint2 keep = make_uint2(0u, 0u);
        if (take + lane < n_cand) keep = cand[take + lane];
        __syncwarp();
        if (take + lane < n_cand) cand[lane] = keep;                 // at most kScanGroup - 1 < 32 entries stay
        n_cand -= take;
        __syncwarp();
    };
    // per-ray state of the inner loop: FP32 origin and direction, and the pass threshold (-theta; +Inf = this ray
    // is not searching: out of range or settled; -Inf = every group is looked at closely)
    float ox[kScanRays], oy[kScanRays], oz[kScanRays], dx[kScanRays], dy[kScanRays], dz[kScanRays], nth[kScanRays];
    unsigned long long beta = lo / n_tiles;                          // current ray batch
    unsigned int tile = tile0;
#pragma unroll 1
    for (unsigned int q = 0; q < total; q++) {
        if (q == 0 || tile == 0) {
            // this warp's rays of batch beta
#pragma unroll
            for (int r = 0; r < kScanRays; r++) {
                const unsigned long long i = beta * kScanBatch + (unsigned long long)(warp * kScanRays + r) * 32 + lane;
                bool search = false;
                SRay f;
                f.ox = f.oy = f.oz = 0.f; f.dx = f.dy = 0.f; f.dz = 1.f; f.theta = 0.f;
                if (i < n) {
                    d3 O = mk(0, 0, 0), D = mk(0, 0, 1);
                    bool valid;
                    int target, target_order;
                    unsigned int l, h;
                    scan_ray_of_index<SHADOW, FIRST>(sc, fp, wf, i, n_hits, O, D, valid, target, target_order, l, h);
                    search = valid;
                    if constexpr (SHADOW) search = !wf.sp_occ[i];     // target missed, or a plane/triangle in front of it
                    if (search) {
                        double a2, inv;
                        make_sray(sc, O, D, f, a2, inv);
                    }
                }
                ox[r] = f.ox; oy[r] = f.oy; oz[r] = f.oz; dx[r] = f.dx; dy[r] = f.dy; dz[r] = f.dz;
                const float oabs = fmaxf(fmaxf(fabsf(f.ox), fabsf(f.oy)), fabsf(f.oz));
                // fmaxf drops NaNs and the filter must pass them: a ray whose v could be Inf - Inf has every group
                // looked at closely (coordinates beyond 1e17, never in practice)
                nth[r] = !search ? kInf : ((oabs + sc.abs_max < 1e17f) ? -f.theta : -kInf);
            }
        }
        const unsigned int stage = q % kScanStages, use = q / kScanStages;
        mbar_wait(&full[stage], use & 1u);
        const float4 *tp = ring + (size_t)stage * kScanTile;
        const int cnt_tile = min(kScanTile, sc.n_spheres - (int)tile * kScanTile);
        if constexpr (COUNT) {
#pragma unroll
            for (int r = 0; r < kScanRays; r++) if (nth[r] != kInf) tl.filter += cnt_tile;
        }
#pragma unroll 1
        for (int k0 = 0; k0 < kScanTile; k0 += kScanGroup) {
            float mg[kScanRays];
#pragma unroll
            for (int r = 0; r < kScanRays; r++) mg[r] = -kInf;
#pragma unroll
            for (int u = 0; u < kScanGroup; u += 2) {
                const float4 s0 = tp[k0 + u], s1 = tp[k0 + u + 1];
                const u64 CX = pk2(s0.x, s0.y), CY = pk2(s0.z, s0.w), CZ = pk2(s1.x, s1.y), RR = pk2(s1.z, s1.w);
#pragma unroll
                for (int r = 0; r < kScanRays; r++) {
                    // per sphere the operations of filter_stage1(): v = b*b - (|c-o|^2 - R), with -(...) folded
                    // into the operand signs (exact: rounding is symmetric)
                    const u64 cx = sub2(CX, bc2(ox[r])), cy = sub2(CY, bc2(oy[r])), cz = sub2(CZ, bc2(oz[r]));
                    const u64 b = fma2(bc2(dz[r]), cz, fma2(bc2(dy[r]), cy, mul2(bc2(dx[r]), cx)));
                    const u64 nw = fma2(neg2(cx), cx, fma2(neg2(cy), cy, fma2(neg2(cz), cz, RR)));
                    const u64 v = fma2(b, b, nw);
                    float v0, v1;
                    upk2(v, v0, v1);
                    mg[r] = fmaxf(fmaxf(mg[r], v0), v1);
                }
            }
            bool any = false;
#pragma unroll
            for (int r = 0; r < kScanRays; r++) any |= !(mg[r] < nth[r]);
            if (__any_sync(0xffffffffu, any)) {
                // the warp looks at the group together: for every (lane, ray) that flagged it, lane k runs stage 1 on
                // sphere k with that ray's constants; the spheres that pass are candidates
                const int cnt = min(kScanGroup, cnt_tile - k0);      // real spheres of the group (the padding never passes)
                const float *grp = reinterpret_cast<const float *>(tp + k0);
                float4 fs = make_float4(0.f, 0.f, 0.f, -3.0e38f);
                if (lane < cnt) {
                    const float *p = grp + (lane >> 1) * 8 + (lane & 1);
                    fs = make_float4(p[0], p[2], p[4], p[6]);
                }
#pragma unroll
                for (int r = 0; r < kScanRays; r++) {
                    unsigned int m = __ballot_sync(0xffffffffu, !(mg[r] < nth[r]));
                    while (m) {
                        const int src = __ffs((int)m) - 1;
                        m &= m - 1u;
                        SRay f;
                        f.ox = __shfl_sync(0xffffffffu, ox[r], src); f.oy = __shfl_sync(0xffffffffu, oy[r], src);
                        f.oz = __shfl_sync(0xffffffffu, oz[r], src); f.dx = __shfl_sync(0xffffffffu, dx[r], src);
                        f.dy = __shfl_sync(0xffffffffu, dy[r], src); f.dz = __shfl_sync(0xffffffffu, dz[r], src);
                        const float th = __shfl_sync(0xffffffffu, nth[r], src);
                        f.theta = -th;                                // -Inf threshold -> theta = +Inf: everything passes
                        float b, v;
                        const bool pass = lane < cnt && filter_stage1(f, fs, b, v);
                        const unsigned int pm = __ballot_sync(0xffffffffu, pass);
                        if (pm) {
                            const unsigned long long i = beta * kScanBatch + (unsigned long long)(warp * kScanRays + r) * 32 + src;
                            if (pass) cand[n_cand + rank_in(pm, lane)] = make_uint2((unsigned int)i, (unsigned int)((int)tile * kScanTile + k0 + lane));
                            n_cand += __popc(pm);
                            if (n_cand >= 32) drain(32);
                        }
                    }
                }
            }
        }
        // this warp is done with the stage; the last warp of the block to say so refills it
        __syncwarp();
        if (lane == 0) {
            const unsigned int old = atomicAdd(&done[stage], 1u);
            if (old + 1u == (unsigned int)kScanWarps * (use + 1u) && q + kScanStages < total) {
                const unsigned int t = (tile0 + q + kScanStages) % n_tiles;
                mbar_expect_tx(&full[stage], kScanTile * 16u);
                bulk_g2s(ring + (size_t)stage * kScanTile, pairs + (size_t)t * kScanTile, kScanTile * 16u, &full[stage]);
            }
        }
        if (++tile == n_tiles) { tile = 0; beta++; }
    }
    if (n_cand > 0) drain(n_cand);
    flush_counters<COUNT>(fp, 0, tl);
}

// After the scan: results to where the next stage reads them.
template <bool SHADOW, bool FIRST>
__global__ void __launch_bounds__(256)
wf_scan_finish(const __grid_constant__ DevScene sc, const __grid_constant__ WfBuf wf, int bounce)
{
    unsigned int n_hits;
    const unsigned long long n = scan_ray_count<SHADOW, FIRST>(sc, wf, bounce, n_hits);
    const size_t np = (size_t)wf.n_pad;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        if constexpr (SHADOW) {
            // shadow_factor (erl:256-267): 1 iff nothing is nearer than the target
            const unsigned int l = (unsigned int)(i / n_hits), h = (unsigned int)(i - (unsigned long long)l * n_hits);
            wf.lit[(size_t)l * np + h] = wf.sp_occ[i] ? 0 : 1;
        } else {
            const ScanBest b = wf.sp_best[i];
            __stcs(wf.res_hit + i, make_int2(b.obj < 0 ? -1 : b.obj, b.order));
            __stcs(wf.res_t + i, b.t);
        }
    }
}


}  // namespace ert
