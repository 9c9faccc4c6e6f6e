"""CPU tests of ert_scene_update's refit (eraytracer_b200/csrc/scene_math.h, the per-node code the device kernels of
ert_update.cuh run) over trees made by bvh_build.cpp, of the shared filter sphere, of the ert_update_info layout and
of the animation generator.

A refit keeps the tree's topology and recomputes its boxes; the walks stay the linear scan's as long as every stored
child box contains the outward-rounded box of every primitive below it.  That is checked here after arbitrary
motion, and a refit of unmoved primitives must give the builder's node array back byte for byte."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import clustered_scene

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "refit", "_build")
SO = os.path.join(BUILD, "librefit_test.so")
# FP32 filter spheres of C3 as flatten() made them before make_filter_sphere moved to scene_math.h
C3_FILTER_SHA256 = "d9694733ea6d5abe33ddd66918bd0c4de412479c255b2660a5aaad0f38fd0baa"
vp, ll = ctypes.c_void_p, ctypes.c_longlong


@pytest.fixture(scope="module")
def rf():
    os.makedirs(BUILD, exist_ok=True)
    src = [os.path.join(HERE, "refit", "shim.cpp"), os.path.join(ROOT, "eraytracer_b200", "csrc", "bvh_build.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO] + src
                          + ["-lpthread"])
    L = ctypes.CDLL(SO)
    L.rf_sphere_build.restype = vp
    L.rf_sphere_build.argtypes = [vp, vp, ll]
    L.rf_tri_build.restype = vp
    L.rf_tri_build.argtypes = [vp, ll]
    for name in ("rf_sphere_free", "rf_tri_free"):
        getattr(L, name).argtypes = [vp]
    L.rf_sphere_refit.argtypes = [vp, vp, vp]
    L.rf_tri_refit.argtypes = [vp, vp]
    L.rf_tri_refit.restype = ctypes.c_double
    for name in ("rf_sphere_nodes", "rf_tri_nodes"):
        getattr(L, name).restype = ll
        getattr(L, name).argtypes = [vp, vp, ll]
    for name in ("rf_sphere_violations", "rf_tri_violations"):
        getattr(L, name).restype = ll
        getattr(L, name).argtypes = [vp]
    L.rf_tri_constants.argtypes = [vp, vp]
    L.rf_filters.argtypes = [vp, vp, ll, vp]
    return L


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _nodes(fn, h):
    n = fn(h, None, 0)
    buf = np.zeros(n, dtype=np.uint8)
    fn(h, buf.ctypes.data, n)
    return buf.tobytes()


def _tris(table):
    return _c(np.concatenate([table['v1'], table['v2'], table['v3']], axis=1))


def _sphere_scenes():
    c3 = sc.synthetic_scene("c3").spheres
    m3 = sc.mesh_scene("m3").spheres
    cl = clustered_scene()[0].spheres
    return {"c3": c3, "m3": m3, "clustered": cl}


@pytest.mark.parametrize("name", ["c3", "m3", "clustered"])
def test_refit_of_unmoved_spheres_is_the_build(rf, name):
    sp = _sphere_scenes()[name]
    c, r = _c(sp['center']), _c(sp['radius'])
    h = rf.rf_sphere_build(c.ctypes.data, r.ctypes.data, len(r))
    built = _nodes(rf.rf_sphere_nodes, h)
    rf.rf_sphere_refit(h, c.ctypes.data, r.ctypes.data)
    assert _nodes(rf.rf_sphere_nodes, h) == built
    assert rf.rf_sphere_violations(h) == 0
    rf.rf_sphere_free(h)


def test_refit_of_unmoved_triangles_is_the_build(rf):
    t = _tris(sc.mesh_scene("m3").triangles)
    h = rf.rf_tri_build(t.ctypes.data, len(t))
    built = _nodes(rf.rf_tri_nodes, h)
    k0 = np.zeros(2)
    rf.rf_tri_constants(h, k0.ctypes.data)
    rf.rf_tri_refit(h, t.ctypes.data)
    k1 = np.zeros(2)
    rf.rf_tri_constants(h, k1.ctypes.data)
    assert _nodes(rf.rf_tri_nodes, h) == built
    assert k0.tobytes() == k1.tobytes()
    rf.rf_tri_free(h)


MOTIONS = ["jitter", "far_swaps", "radii_x10", "negative_radii", "coords_1e6"]


def _move_spheres(c, r, how, rng):
    c, r = c.copy(), r.copy()
    n = len(r)
    if how == "jitter":
        c += rng.normal(0, 0.3, c.shape)
    elif how == "far_swaps":
        k = rng.permutation(n)[: n // 4]
        c[k] = c[np.roll(k, 1)]                       # spheres trade places across the scene
    elif how == "radii_x10":
        r *= 10.0
    elif how == "negative_radii":
        r = np.where(rng.uniform(0, 1, n) < 0.5, -r, r)
    elif how == "coords_1e6":
        c = rng.uniform(-1e6, 1e6, c.shape)
        r = rng.uniform(0, 1e3, n)
    if how != "coords_1e6":
        c = c.astype(np.float32).astype(np.float64)
    return _c(c), _c(r)


@pytest.mark.parametrize("how", MOTIONS)
@pytest.mark.parametrize("name", ["c3", "clustered"])
def test_refitted_sphere_boxes_contain_their_spheres(rf, name, how):
    sp = _sphere_scenes()[name]
    c, r = _c(sp['center']), _c(sp['radius'])
    rng = np.random.default_rng(10 * MOTIONS.index(how) + len(name))
    h = rf.rf_sphere_build(c.ctypes.data, r.ctypes.data, len(r))
    for _ in range(3):                                # repeated refits of the same topology
        c2, r2 = _move_spheres(c, r, how, rng)
        rf.rf_sphere_refit(h, c2.ctypes.data, r2.ctypes.data)
        assert rf.rf_sphere_violations(h) == 0
    # a refit back to the build's values restores the build
    h2 = rf.rf_sphere_build(c.ctypes.data, r.ctypes.data, len(r))
    rf.rf_sphere_refit(h, c.ctypes.data, r.ctypes.data)
    assert _nodes(rf.rf_sphere_nodes, h) == _nodes(rf.rf_sphere_nodes, h2)
    rf.rf_sphere_free(h)
    rf.rf_sphere_free(h2)


@pytest.mark.parametrize("how", ["jitter", "far_swaps", "scale_x10", "coords_1e6"])
def test_refitted_triangle_boxes_contain_their_triangles(rf, how):
    t = _tris(sc.mesh_scene("m3").triangles)
    rng = np.random.default_rng(len(how))
    h = rf.rf_tri_build(t.ctypes.data, len(t))
    t2 = t.copy()
    if how == "jitter":
        t2 += rng.normal(0, 0.2, t2.shape)
    elif how == "far_swaps":
        k = rng.permutation(len(t))[: len(t) // 4]
        t2[k] = t2[np.roll(k, 1)]
    elif how == "scale_x10":
        t2 *= 10.0
    else:
        t2 = rng.uniform(-1e6, 1e6, t2.shape)
    a_max = rf.rf_tri_refit(h, t2.ctypes.data)
    assert a_max <= 1e30
    assert rf.rf_tri_violations(h) == 0
    rf.rf_tri_free(h)


def test_triangle_beyond_the_float_range_is_reported(rf):
    """A tree triangle moved past kTriAlwaysAbs: the refit reports it (ert_scene_update then rebuilds on the host)."""
    t = _tris(sc.mesh_scene("m3").triangles)
    h = rf.rf_tri_build(t.ctypes.data, len(t))
    t2 = t.copy()
    t2[5, 0:3] = 2e30
    assert rf.rf_tri_refit(h, t2.ctypes.data) > 1e30
    rf.rf_tri_free(h)


def test_shared_filter_sphere_keeps_the_c3_table(rf):
    sp = sc.synthetic_scene("c3").spheres
    c, r = _c(sp['center']), _c(sp['radius'])
    out = np.zeros((len(r), 4), dtype=np.float32)
    rf.rf_filters(c.ctypes.data, r.ctypes.data, len(r), out.ctypes.data)
    assert hashlib.sha256(out.tobytes()).hexdigest() == C3_FILTER_SHA256


def test_update_info_layout_matches_the_header(tmp_path):
    src = tmp_path / "info.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "ert_b200.h"
#define F(m) printf("%s %zu\n", #m, offsetof(ert_update_info, m));
int main(void) {
    printf("size %zu\n", sizeof(ert_update_info));
    F(changed) F(done) F(has_cell_grid) F(light_grids) F(light_grids_rebuilt) F(reserved) F(h2d_bytes) F(host_ms)
    F(device_ms) F(sphere_area_ratio) F(triangle_area_ratio)
    printf("flags %u %u\n", ERT_UPDATE_REBUILD_GRIDS, ERT_UPDATE_REBUILD);
    return 0;
}
''')
    exe = tmp_path / "info"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict(line.split(" ", 1) for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got.pop("size")) == ctypes.sizeof(_lib.UpdateInfo)
    assert got.pop("flags") == "%d %d" % (_lib.UPDATE_REBUILD_GRIDS, _lib.UPDATE_REBUILD)
    for name, off in got.items():
        assert getattr(_lib.UpdateInfo, name).offset == int(off), name
    assert [n for n, _ in _lib.UpdateInfo._fields_] == list(got)


def _flat_bytes(f):
    return [np.ascontiguousarray(t).tobytes() for t in (f.lights, f.spheres, f.triangles, f.planes)]


@pytest.mark.parametrize("name", ["c3", "m3"])
def test_animated_scene(name):
    still = sc.synthetic_scene(name) if name == "c3" else sc.mesh_scene(name)
    assert _flat_bytes(sc.animated_scene(name, 0)) == _flat_bytes(still)
    for k in (1, 16, 40):
        f = sc.animated_scene(name, k)
        for a, b in zip((f.lights, f.spheres, f.triangles, f.planes), (still.lights, still.spheres, still.triangles,
                                                                        still.planes)):
            assert len(a) == len(b) and np.array_equal(a['order'], b['order'])
        d = np.linalg.norm(f.spheres['center'] - still.spheres['center'], axis=1)
        assert 0 < d.max() <= sc.ANIM_AMPLITUDE * 1.001
        assert np.array_equal(f.spheres['radius'], still.spheres['radius'])
        assert np.array_equal(f.spheres['center'], f.spheres['center'].astype(np.float32).astype(np.float64))
        if name == "m3":
            for v in ("v1", "v2", "v3"):
                assert np.array_equal(f.triangles[v], f.triangles[v].astype(np.float32).astype(np.float64))
            assert not np.array_equal(f.triangles['v1'], still.triangles['v1'])
        assert _flat_bytes(sc.animated_scene(name, k)) == _flat_bytes(f)        # deterministic
