"""CPU check of the FP32 sphere filter at every magnitude (ert_device.cuh make_fray, ert_wavefront.cuh make_sray).

The filter's bounds (DESIGN.md "Filter bounds") hold while |o|_inf + abs_max stays below kFilterRange (1e17).
Beyond it the squares of stage 1 overflow float: |c - o|^2 - R becomes +Inf, v = b*b - Inf = -Inf, and stage 1 would
reject a sphere the ray hits.  The range rule sends such rays to the literal FP64 test of every sphere instead, and
the scans that have no tree to leave pass every sphere through the filter.

tests/filterrange/shim.cpp restates the filter sphere, both ray set-ups, both filter stages, both slab tests and the
cull distances operation for operation in float32 (g++ -ffp-contract=off, std::fmaf for __fmaf_rn), and this file
holds them to the literal FP64 test of raytracer.erl:364-397 (sphere_exact of test_shadow_triage_bounds.py):

    the FP64 test hits  ==>  the ray is routed to the FP64 fallback (out of range), or stage 1, stage 2 (with and
                             without an incumbent it ties) and the slab tests of the sphere's box and of an
                             enclosing box all pass it.

With the range rule switched off, the same sweep loses hits, among them the far planets of TABLE below.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from test_shadow_triage_bounds import sphere_exact

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "filterrange", "_build")
SO = os.path.join(BUILD, "libfilterrange_test.so")
vp, ll = ctypes.c_void_p, ctypes.c_longlong

IN_RANGE, STAGE1, STAGE2, STAGE2_CULL, BOX, ENCLOSING, BOXES_CULL = 1, 2, 4, 8, 16, 32, 64
ALL_PASS = STAGE1 | STAGE2 | STAGE2_CULL | BOX | ENCLOSING | BOXES_CULL


@pytest.fixture(scope="module")
def fr():
    os.makedirs(BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO,
                           os.path.join(HERE, "filterrange", "shim.cpp")])
    L = ctypes.CDLL(SO)
    L.fr_check.argtypes = [vp, vp, vp, vp, ll, ctypes.c_int, vp, vp]
    L.fr_shadow_blocked.argtypes = [vp, vp, vp, ctypes.c_double, vp, ctypes.c_double, ctypes.c_float]
    L.fr_shadow_blocked.restype = ctypes.c_int
    return L


def check(L, O, D, C, r, rule=True, enclose=None):
    """Runs fr_check over configs; returns (FP64 hit, t, flags of make_fray, flags of make_sray, w, v)."""
    n = len(r)
    O = np.ascontiguousarray(O, np.float64).reshape(n, 3)
    D = np.ascontiguousarray(D, np.float64).reshape(n, 3)
    C = np.ascontiguousarray(C, np.float64).reshape(n, 3)
    r = np.ascontiguousarray(r, np.float64)
    hit, t = sphere_exact(O, D, C, r)
    rays = np.ascontiguousarray(np.hstack([O, D]))
    sph = np.ascontiguousarray(np.hstack([C, r[:, None]]))
    if enclose is None:
        # a BVH node above the leaf: the sphere's box grown to take in the origin's neighbourhood and the scene's middle
        enclose = np.hstack([np.minimum(C - r[:, None], np.minimum(O, 0.0) - 1.0),
                             np.maximum(C + r[:, None], np.maximum(O, 0.0) + 1.0)])
    box = np.ascontiguousarray(enclose, np.float64)
    # the tightest incumbent the sphere still wins against: a tie at its own Distance
    t_inc = np.ascontiguousarray(np.where(hit, t, np.nan))
    flags = np.zeros(n, np.int32)
    wv = np.zeros(2 * n, np.float32)
    L.fr_check(rays.ctypes.data, sph.ctypes.data, box.ctypes.data, t_inc.ctypes.data, n, 1 if rule else 0,
               flags.ctypes.data, wv.ctypes.data)
    return hit, t, flags & 0xff, flags >> 8, wv[0::2], wv[1::2]


def lost(hit, ff, fs):
    """Configs the FP64 test hits that a filter path would drop: in range and some stage or box test rejects."""
    bad = np.zeros(len(hit), bool)
    for f in (ff, fs):
        bad |= hit & ((f & IN_RANGE) != 0) & ((f & ALL_PASS) != ALL_PASS)
    return bad


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


# ---- the cases of the table: a far planet, and a light far from a near sphere -----------------------------------
TABLE = [
    # O, D, C, r, does the reference hit?
    ((0, 0, 0), (0, 0, 1), (0, 0, 1e18), 1e17, True),
    ((0, 0, 0), (0, 0, 1), (0, 0, 2e19), 1e18, True),
    ((0, 0, 0), (0, 0, 1), (0, 0, 1e20), 1e19, True),
    # From 1e19 on (long before), the reference's Discriminant of a unit sphere cancels to exactly 0: b*b and 4*a*c
    # both round to 4*fl(|O - C|^2), the "- r*r" is lost.  The reference itself does not see the sphere.
    ((0, 1e19, 0), (0, -1, 0), (0, 0, 0), 1.0, False),
    ((0, 1.9e19, 0), (0, -1, 0), (0, 0, 0), 1.0, False),
    ((0, 1e20, 0), (0, -1, 0), (0, 0, 0), 1.0, False),
    # occluders the reference does see from there: large enough that r*r survives the rounding of |O - C|^2
    ((0, 1.9e19, 0), (0, -1, 0), (0, 0, 0), 1e13, True),
    ((0, 1e20, 0), (0, -1, 0), (0, 0, 0), 1e15, True),
]


def _table():
    O = np.array([c[0] for c in TABLE], float)
    D = np.array([c[1] for c in TABLE], float)
    C = np.array([c[2] for c in TABLE], float)
    r = np.array([c[3] for c in TABLE], float)
    return O, D, C, r, np.array([c[4] for c in TABLE])


def test_table_cases_are_lost_without_the_range_rule(fr):
    O, D, C, r, want = _table()
    hit, t, ff, fs, w, v = check(fr, O, D, C, r, rule=False)
    assert (hit == want).all(), hit
    # stage 1 overflows once |O - C| passes about 1.85e19: w = +Inf, v = -Inf, and the hit is rejected
    overflow = np.isinf(w) & (w > 0)
    assert (np.isneginf(v) == overflow).all()
    assert overflow.tolist() == [False, True, True, False, True, True, True, True]
    assert not (ff[overflow] & STAGE1).any() and not (fs[overflow] & STAGE1).any()
    dropped = lost(hit, ff, fs)
    assert dropped.tolist() == [False, True, True, False, False, False, True, True]
    # with the rule, every one of them is routed to the FP64 fallback, and nothing is lost
    hit, t, ff, fs, w, v = check(fr, O, D, C, r, rule=True)
    assert not lost(hit, ff, fs).any()
    assert not (ff[overflow] & IN_RANGE).any() and not (fs[overflow] & IN_RANGE).any()
    # the first planet still passes the filter, but 1.1e18 is past the range too
    assert not (ff & IN_RANGE).any() and not (fs & IN_RANGE).any()


# ---- the sweep --------------------------------------------------------------------------------------------------
def _distances():
    d = [1.0, 10.0, 1e3, 1e6, 1e10, 1e14, 1e16]
    d += list(2.0 ** np.arange(56, 67))               # 7e16 ... 7.4e19, by powers of 2 across 1e17 ... 1e20
    d += [1e17, 1e18, 1.84e19, 1.85e19, 1.9e19, 2e19, 1e20, 1e22, 1e25, 1e30, 1e34, 1e38]
    return np.array(d)


RADII = np.array([1e-3, 1e-2, 0.1, 0.5, 0.9, 0.999])
ORIGINS = [np.zeros(3), np.array([1e16, 0, 0]), np.array([0, -3e18, 0]), np.array([2e19, 1e19, -1e19]),
           np.array([0, 0, 1e30]), np.array([1e39, 0, 0]), np.array([0, -1e100, 0])]
DIRECTIONS = [np.array([0, 0, 1.0]), np.array([-1.0, 0, 0]), np.array([0, 1e-40, 1.0]), np.array([1e-39, -1.0, 1e-42]),
              unit([0.3, -0.5, 0.8]), unit([1.0, 1.0, 1.0])]


def _perp(D):
    a = np.zeros(3)
    a[np.argmin(np.abs(D))] = 1.0
    p = np.cross(D, a)
    return p / np.linalg.norm(p)


def _f32(x):
    """x rounded to float where float holds it (coordinates past FLT_MAX stay as they are)"""
    return np.where(np.abs(x) < 3e38, x.astype(np.float32, casting="unsafe") if np.all(np.abs(x) < 3e38) else x, x)


def _sweep(exact_f32):
    """Rays aimed at sphere centres, at half the radius and grazing (impact parameter within 1e-6 of r)."""
    O, D, C, r = [], [], [], []
    rng = np.random.default_rng(7)
    for o in ORIGINS:
        for d in DIRECTIONS:
            u = d / np.linalg.norm(d)
            p = _perp(u)
            for dist in _distances():
                for rf in RADII:
                    rad = rf * dist
                    for q in (0.0, 0.5, 1.0 - 1e-6):
                        c = o + dist * u + q * rad * p
                        if exact_f32:
                            c, oo = _f32(c), _f32(o)
                        else:
                            c = c * (1.0 + rng.uniform(-1e-12, 1e-12, 3)) + rng.uniform(-0.3, 0.3, 3)
                            oo = o * (1.0 + 1e-13) + 0.1
                        O.append(oo)
                        D.append(d)
                        C.append(c)
                        r.append(rad)
    return np.array(O), np.array(D), np.array(C), np.array(r)


@pytest.mark.parametrize("exact_f32", [True, False], ids=["float-exact", "not-float-exact"])
def test_every_fp64_hit_passes_the_filter_or_takes_the_fallback(fr, exact_f32):
    O, D, C, r = _sweep(exact_f32)
    # the reference must be finite here: |O - C| stays far below 1e154
    assert np.abs(C - O).max() < 1e140
    hit, t, ff, fs, w, v = check(fr, O, D, C, r)
    assert hit.sum() > len(hit) // 2
    bad = lost(hit, ff, fs)
    assert not bad.any(), (O[bad][:4], D[bad][:4], C[bad][:4], r[bad][:4], ff[bad][:4], fs[bad][:4])
    # the two set-ups agree on the range
    assert ((ff & IN_RANGE) == (fs & IN_RANGE)).all()
    # out of range, make_fray's constants pass every sphere through both stages, hit or not: the megakernel's tiled
    # scan and the linear and warp ray batches rely on it (wf_scan, the other scan without a tree, sets its own
    # stage-1 threshold; make_sray leaves its constants as they are)
    out = (ff & IN_RANGE) == 0
    assert out.any() and (~out).any()
    assert ((ff[out] & (STAGE1 | STAGE2 | STAGE2_CULL)) == (STAGE1 | STAGE2 | STAGE2_CULL)).all()
    # the rule is |o|_inf + abs_max < 1e17 in float
    amax = np.max(np.abs(C) + r[:, None], axis=1)
    oabs = np.max(np.abs(O), axis=1)
    assert (out[oabs + amax >= 1.01e17]).all() and (~out[oabs + amax < 0.99e17]).all()


@pytest.mark.parametrize("exact_f32", [True, False], ids=["float-exact", "not-float-exact"])
def test_the_sweep_loses_hits_without_the_range_rule(fr, exact_f32):
    O, D, C, r = _sweep(exact_f32)
    hit, t, ff, fs, w, v = check(fr, O, D, C, r, rule=False)
    bad = lost(hit, ff, fs)
    in_range = (check(fr, O, D, C, r, rule=True)[2] & IN_RANGE) != 0
    # hits are lost, and only where the rule now sends the ray to the FP64 fallback
    assert bad.sum() > 1000
    assert not bad[in_range].any()
    # every hit whose stage 1 overflowed (w = +Inf, v = -Inf) is among them
    overflow = hit & np.isposinf(w) & np.isneginf(v)
    assert overflow.sum() > 1000 and bad[overflow].all()


# ---- shadow triage past its range -------------------------------------------------------------------------------
def _triage(L, light, P, tc, tr, cc, cr, dmin=-np.inf):
    lt = np.zeros(9)
    lt[3:6] = light
    P, tc, cc = (np.ascontiguousarray(x, np.float64) for x in (P, tc, cc))
    return L.fr_shadow_blocked(lt.ctypes.data, P.ctypes.data, tc.ctypes.data, tr, cc.ctypes.data, cr, dmin)


def test_shadow_triage_never_claims_blocked_past_its_range(fr):
    # in range it does prove a plain occluder (the check has teeth)
    tc, tr = np.array([0.0, 0, 0]), 1.0
    P = np.array([0.0, 1.0, 0])
    assert _triage(fr, [0, 10.0, 0], P, tc, tr, [0, 5.0, 0], 1.0) == 1
    n_blocked = 0
    for dist in (1e10, 1e16, 1.9e19, 1e20, 1e30, 1e39, 1e100):
        for occ in (0.5, 0.9):
            light = np.array([0.0, dist, 0.0])
            # the light far away: |P - L|^2 >= 1e20, or Inf, or NaN
            r_occ = max(1.0, 1e-3 * dist)
            assert _triage(fr, light, P, tc, tr, [0, occ * dist, 0], r_occ) == 0
            assert _triage(fr, light, P, tc, tr, [0, 5.0, 0], 1.0) == 0
    # a near light and candidates (or targets) past the range: the squares are Inf or NaN
    for far in (1e19, 1e20, 1e30, 1e39, 1e100):
        light = np.array([0.0, 10.0, 0.0])
        assert _triage(fr, light, P, tc, tr, [0, far, 0], 0.5 * far) == 0
        assert _triage(fr, light, P, tc, tr, [0, -far, 0], 0.999 * far) == 0
        assert _triage(fr, light, [0, -far + 1.0, 0], [0, -far, 0], 1.0, [0, 5.0, 0], 1.0) == 0
        n_blocked += _triage(fr, light, P, tc, tr, [far, far, far], far)
    assert n_blocked == 0
