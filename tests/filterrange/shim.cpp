// Test-only restatement in host C++ of the FP32 sphere filter of the device code, operation for operation: the filter
// sphere (make_filter_sphere, scene_math.h, used as it is), the ray constants of make_fray (ert_device.cuh) and
// make_sray (ert_wavefront.cuh) with their range rule, filter_stage1 / filter_stage2, both slab tests (the
// megakernel's slab_hit and the wavefront's slab_test), cull_from / cullk_from, and the shadow triage
// shadow_blocked for one direction-cell candidate.  Built with -ffp-contract=off, like the device code's
// -fmad=false; every __fmaf_rn is std::fmaf.  __frcp_rn and __double2float_ru are correctly rounded, as 1.0f / x and
// f_round_up are.  rsqrtf (2 ulp on the device) is 1 / sqrtf here: the triage's verdicts past its range do not
// depend on that last bit.
#include <cmath>
#include <cstdint>
#include <cstring>

#include "../../eraytracer_b200/csrc/scene_math.h"

using namespace ert;

namespace {
constexpr float kU = 5.9604644775390625e-8f;         // ERT_U
constexpr double kKD = 1.0000019073486328125;        // ERT_KD
constexpr float kRel16 = 1.52587890625e-5f;          // ERT_REL16
constexpr float kRel17 = 7.62939453125e-6f;          // ERT_REL17
constexpr float kKappa = 1.00006103515625f;          // ERT_KAPPA
constexpr float kFilterRange = 1e17f;                // kFilterRange
const float kInf = INFINITY;

struct Scene {                                       // the DevScene constants the filter reads
    float r_max, pad_c_max, eta_c_max, abs_max;
};

// FRay and SRay in one: the megakernel's slab constants (n*, f*) and the wavefront's (kl*, kh*)
struct Ray {
    float ox, oy, oz, dx, dy, dz;
    float theta, bcull, pad2, m4;
    float ix, iy, iz, nx, ny, nz, fx, fy, fz;         // make_fray
    float jx, jy, jz, klx, kly, klz, khx, khy, khz;   // make_sray
    double inv_sqrt_a, a;
    bool in_range;
};

float clamp_dir(float d)
{
    if (std::fabs(d) < 1e-20f) return d < 0.f ? -1e-20f : 1e-20f;
    return d;
}

// make_fray (want_slabs) and make_sray on the same ray; `rule` 0 leaves the range rule out
void make_ray(const Scene &sc, const double *O, const double *D, bool sray, bool rule, Ray &f)
{
    const double a = D[0] * D[0] + D[1] * D[1] + D[2] * D[2];
    const double inv = sray ? ((std::fabs(a - 1.0) <= 1e-9) ? (1.5 - 0.5 * a) : 1.0 / std::sqrt(a)) : 1.0 / std::sqrt(a);
    f.a = a;
    f.inv_sqrt_a = inv;
    f.ox = (float)O[0]; f.oy = (float)O[1]; f.oz = (float)O[2];
    const double k = inv * kKD;
    f.dx = (float)(D[0] * k); f.dy = (float)(D[1] * k); f.dz = (float)(D[2] * k);
    float eo = 2.0f * std::fmax(std::fmax(std::fabs((float)(O[0] - (double)f.ox)), std::fabs((float)(O[1] - (double)f.oy))),
                                std::fabs((float)(O[2] - (double)f.oz)));
    eo *= 1.0001f;
    f.theta = 16.0f * sc.r_max * eo + 8.0f * eo * (eo / kU);
    f.bcull = 2.0f * (5.0f * kU * sc.r_max + 2.0f * eo + 2.0f * sc.eta_c_max);
    f.pad2 = 2.0f * (f.theta + sc.pad_c_max) + 1e-30f;
    const float oabs = std::fmax(std::fmax(std::fabs(f.ox), std::fabs(f.oy)), std::fabs(f.oz));
    const float m = eo + 32.0f * kU * (oabs + sc.abs_max);
    f.m4 = 4.0f * m;
    {   // make_fray's slabs
        const float dx = clamp_dir(f.dx), dy = clamp_dir(f.dy), dz = clamp_dir(f.dz);
        f.ix = 1.0f / dx; f.iy = 1.0f / dy; f.iz = 1.0f / dz;
        const float sx = dx < 0.f ? -m : m, sy = dy < 0.f ? -m : m, sz = dz < 0.f ? -m : m;
        f.nx = -(f.ox + sx) * f.ix; f.ny = -(f.oy + sy) * f.iy; f.nz = -(f.oz + sz) * f.iz;
        f.fx = -(f.ox - sx) * f.ix; f.fy = -(f.oy - sy) * f.iy; f.fz = -(f.oz - sz) * f.iz;
    }
    {   // make_sray's slabs
        f.jx = 1.0f / clamp_dir(f.dx); f.jy = 1.0f / clamp_dir(f.dy); f.jz = 1.0f / clamp_dir(f.dz);
        f.klx = -(f.ox + m) * f.jx; f.kly = -(f.oy + m) * f.jy; f.klz = -(f.oz + m) * f.jz;
        f.khx = -(f.ox - m) * f.jx; f.khy = -(f.oy - m) * f.jy; f.khz = -(f.oz - m) * f.jz;
    }
    f.in_range = !rule || oabs + sc.abs_max < kFilterRange;
    if (!f.in_range && !sray) f.theta = f.bcull = f.m4 = kInf;       // make_fray only: its scans without a tree
}

float cull_from(const Ray &f, bool have, double t)
{
    if (!have) return kInf;
    const float sf = f_round_up(t * f.inv_sqrt_a);
    return sf + std::fabs(sf) * kRel16 + f.m4;
}
float cullk_from(const Ray &f, bool have, double t)
{
    if (!have) return kInf;
    const float sf = f_round_up(t * f.inv_sqrt_a);
    return (sf + std::fabs(sf) * kRel16 + f.m4) * kKappa;
}

bool filter_stage1(const Ray &f, const float s[4], float &b, float &v)
{
    const float cx = s[0] - f.ox, cy = s[1] - f.oy, cz = s[2] - f.oz;
    b = std::fmaf(f.dz, cz, std::fmaf(f.dy, cy, f.dx * cx));
    const float w = std::fmaf(cx, cx, std::fmaf(cy, cy, std::fmaf(cz, cz, -s[3])));
    v = std::fmaf(b, b, -w);
    return !(v < -f.theta);
}
bool filter_stage2(const Ray &f, const float s[4], float b, float v, float cull)
{
    if (b < -f.bcull) return false;
    if (cull == kInf) return true;
    const float arg = std::fmax(v, 0.f) + kRel17 * (b * b + s[3]) + f.pad2;
    const float s_lo = b - std::fabs(b) * kRel16 - std::sqrt(arg) * 1.000001f - f.bcull;
    return !(s_lo > cull);
}

// slab_hit of the megakernel (ert_device.cuh)
bool slab_hit(const Ray &f, const float lo[3], const float hi[3], float cull)
{
    const float nx = f.dx < 0.f ? hi[0] : lo[0], fx = f.dx < 0.f ? lo[0] : hi[0];
    const float ny = f.dy < 0.f ? hi[1] : lo[1], fy = f.dy < 0.f ? lo[1] : hi[1];
    const float nz = f.dz < 0.f ? hi[2] : lo[2], fz = f.dz < 0.f ? lo[2] : hi[2];
    const float t0x = std::fmaf(nx, f.ix, f.nx), t1x = std::fmaf(fx, f.ix, f.fx);
    const float t0y = std::fmaf(ny, f.iy, f.ny), t1y = std::fmaf(fy, f.iy, f.fy);
    const float t0z = std::fmaf(nz, f.iz, f.nz), t1z = std::fmaf(fz, f.iz, f.fz);
    const float tnear = std::fmax(std::fmax(t0x, t0y), std::fmax(t0z, 0.f));
    const float tfar = std::fmin(std::fmin(t1x, t1y), std::fmin(t1z, cull));
    return tnear - std::fabs(tnear) * kRel16 <= tfar + std::fabs(tfar) * kRel16;
}
// slab_test of the wavefront (ert_wavefront.cuh)
bool slab_test(const Ray &f, const float lo[3], const float hi[3], float cullk)
{
    const float ax = std::fmaf(lo[0], f.jx, f.klx), bx = std::fmaf(hi[0], f.jx, f.khx);
    const float ay = std::fmaf(lo[1], f.jy, f.kly), by = std::fmaf(hi[1], f.jy, f.khy);
    const float az = std::fmaf(lo[2], f.jz, f.klz), bz = std::fmaf(hi[2], f.jz, f.khz);
    const float tn = std::fmax(std::fmax(std::fmin(ax, bx), std::fmin(ay, by)), std::fmin(az, bz));
    const float tf = std::fmin(std::fmin(std::fmax(ax, bx), std::fmax(ay, by)), std::fmax(az, bz));
    const float tnear = std::fmax(tn, 0.f);
    return tnear <= std::fmin(tf * kKappa, cullk);
}
}  // namespace

extern "C" {

// For config k: the ray rays6[6k..6k+5] against the sphere sph4[4k..4k+3], alone in its scene (the scene constants are
// the sphere's own, which makes abs_max as small as it can be).  box6[6k..] is an enclosing box {lo[3], hi[3]} (a BVH
// node above the sphere's leaf); the sphere's own outward-rounded box is tested as well.  t_inc[k]: Distance of an
// incumbent that the sphere ties (NaN: none).  Per config, flags[k] of both ray set-ups (bits 0-7 make_fray, 8-15
// make_sray):
//   bit 0 in range, 1 stage 1 passes, 2 stage 2 passes without an incumbent, 3 stage 2 passes with the incumbent,
//   4 the slab test passes the sphere's box and 5 the enclosing box without an incumbent, 6 both with the incumbent.
// v_out[2k], v_out[2k+1]: stage 1's w and v of make_fray's ray.
void fr_check(const double *rays6, const double *sph4, const double *box6, const double *t_inc, long long n, int rule,
              int *flags, float *v_out)
{
    for (long long k = 0; k < n; k++) {
        const double *O = rays6 + 6 * k, *D = O + 3, *s = sph4 + 4 * k;
        float fs[4], pad_c, eta_c;
        make_filter_sphere(s, s[3], fs, pad_c, eta_c);
        Scene sc;
        sc.r_max = f_round_up(std::fabs(s[3]));
        sc.pad_c_max = pad_c;
        sc.eta_c_max = eta_c;
        sc.abs_max = 0.f;
        for (int a = 0; a < 3; a++) sc.abs_max = std::max(sc.abs_max, f_round_up(std::fabs(s[a]) + std::fabs(s[3])));
        float lo[3], hi[3], elo[3], ehi[3];
        sphere_box(s, lo, hi);
        for (int a = 0; a < 3; a++) {
            elo[a] = f_round_down(box6[6 * k + a]);
            ehi[a] = f_round_up(box6[6 * k + 3 + a]);
        }
        const bool have = !std::isnan(t_inc[k]);
        int out = 0;
        for (int w = 0; w < 2; w++) {
            Ray f;
            make_ray(sc, O, D, w == 1, rule != 0, f);
            float b, v;
            const bool s1 = filter_stage1(f, fs, b, v);
            const float c0 = w ? cullk_from(f, false, 0.0) : cull_from(f, false, 0.0);
            const float c1 = w ? cullk_from(f, have, t_inc[k]) : cull_from(f, have, t_inc[k]);
            auto slab = [&](const float *l, const float *h, float c) { return w ? slab_test(f, l, h, c) : slab_hit(f, l, h, c); };
            int fl = (f.in_range ? 1 : 0) | (s1 ? 2 : 0) | (filter_stage2(f, fs, b, v, c0) ? 4 : 0) |
                     (filter_stage2(f, fs, b, v, c1) ? 8 : 0) | (slab(lo, hi, c0) ? 16 : 0) | (slab(elo, ehi, c0) ? 32 : 0) |
                     ((slab(lo, hi, c1) && slab(elo, ehi, c1)) ? 64 : 0);
            out |= fl << (8 * w);
            if (w == 0) {
                const float cx = fs[0] - f.ox, cy = fs[1] - f.oy, cz = fs[2] - f.oz;
                v_out[2 * k] = std::fmaf(cx, cx, std::fmaf(cy, cy, std::fmaf(cz, cz, -fs[3])));
                v_out[2 * k + 1] = v;
            }
        }
        flags[k] = out;
    }
}

// shadow_blocked (ert_wavefront.cuh) for a sphere target {tc, tr}, a light at lt[3..5] (lt[0..2] unused, as on the
// device), the hit location P, and ONE candidate of the direction cell: the sphere {cc, cr} with the cell's nearest
// distance dmin (the head's c[5]).  The scene constants are those of the two spheres.  Returns 1 for "blocked".
int fr_shadow_blocked(const double *lt, const double *P, const double *tc, double tr, const double *cc, double cr,
                      float dmin)
{
    float tf[4], cf[4], pad_t, eta_t, pad_s, eta_s;
    make_filter_sphere(tc, tr, tf, pad_t, eta_t);
    make_filter_sphere(cc, cr, cf, pad_s, eta_s);
    const float pad_c_max = std::max(pad_t, pad_s), eta_c_max = std::max(eta_t, eta_s);
    const float u = kU;
    const float fx = (float)(P[0] - lt[3]), fy = (float)(P[1] - lt[4]), fz = (float)(P[2] - lt[5]);
    const float l2 = fx * fx + fy * fy + fz * fz;
    if (!(l2 > 1e-20f && l2 < 1e20f)) return 0;
    const float inv = 1.0f / std::sqrt(l2);
    const float dx = fx * inv, dy = fy * inv, dz = fz * inv;
    const float ox = (float)lt[3], oy = (float)lt[4], oz = (float)lt[5];
    const float ec0 = 1.01f * (eta_c_max + 1.75f * u * std::fmax(std::fmax(std::fabs(ox), std::fabs(oy)), std::fabs(oz)));
    const float tx = tf[0] - ox, ty = tf[1] - oy, tz = tf[2] - oz;
    const float trho2 = tx * tx + ty * ty + tz * tz;
    const float tb = dx * tx + dy * ty + dz * tz;
    const float s_lo = tb - (ec0 + 26.f * u * std::sqrt(trho2)) - std::sqrt(tf[3]) * (1.f + 4.f * u) - 4.f * u * std::fabs(tb) -
                       1e-12f * trho2 - 1e-7f;
    if (dmin > s_lo) return 0;
    const float cx = cf[0] - ox, cy = cf[1] - oy, cz = cf[2] - oz, R = cf[3];
    const float rho2 = cx * cx + cy * cy + cz * cz;
    const float rho = std::sqrt(rho2);
    const float b = dx * cx + dy * cy + dz * cz;
    const float qx = cy * dz - cz * dy, qy = cz * dx - cx * dz, qz = cx * dy - cy * dx;
    const float err = ec0 + 26.f * u * rho;
    const float qmax = std::sqrt(qx * qx + qy * qy + qz * qz) * (1.f + 8.f * u) + err;
    const float fp64_noise = 1e-12f * rho2;
    const float T = ((R - pad_c_max) * (1.f - 7.62939453125e-6f) - 8.f * u * R) - qmax * qmax * (1.f + 4.f * u) - 8.f * u * R;
    if (T > 0.0004f + fp64_noise && b - err > std::sqrt(R) * (1.f + 4.f * u)) {
        float s_up = b + err - std::sqrt(T) * (1.f - 4.f * u);
        s_up += 4.f * u * b + 4e-6f * std::fabs(s_up) + fp64_noise + 1e-7f;
        if (s_up < s_lo) return 1;
    }
    return 0;
}
}
