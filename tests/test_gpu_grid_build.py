"""The device grid builders (grid_build.cuh) on the GPU.

Through tests/gridbuild/shim.cu they must give the host builders' bytes (cell grid: blocks, overflow lists, big list,
geometry; direction grids: cell_off, cand, head, always) and the same "no grid" decisions, and a device-built
direction grid must list every sphere a shadow ray can touch.  Through the C ABI, ert_scene_update with
ERT_UPDATE_REBUILD_GRIDS must leave a scene that renders, counts and reports its grids exactly like a fresh
ert_scene_create of the same tables, while uploading only the changed tables."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import clustered_scene
from test_grid_build_host import CAND_DT, HERE, declare, host_cell, host_light, raw, scene_lights, sphere_table

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "eraytracer_b200", "csrc")
BUILD = os.path.join(HERE, "gridbuild", "_build")
SO = os.path.join(BUILD, "libgridbuild_test.so")
vp, ll = ctypes.c_void_p, ctypes.c_longlong
MAX_ENTRIES = 1 << 27                      # kLightGridMaxEntries

RENDER_ACCELS = ("exact", "linear", "bvh", "bvh_mega", "grid", "auto")
FAST_ACCELS = ("bvh", "bvh_mega", "grid", "auto")
COUNTERS = ("rays", "sphere_filter_tests", "box_tests", "exact_sphere_tests", "exact_other_tests", "cell_steps",
            "path_box_tests", "path_filter_tests", "shadow_box_tests", "shadow_filter_tests")


@pytest.fixture(scope="module")
def gd(gpu):
    os.makedirs(BUILD, exist_ok=True)
    src = [os.path.join(HERE, "gridbuild", "shim.cu"), os.path.join(CSRC, "cell_grid.cpp"),
           os.path.join(CSRC, "light_grid.cpp")]
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
                           "-Xcompiler", "-fPIC", "-shared", "-o", SO] + src + ["-lpthread"])
    L = declare(ctypes.CDLL(SO))
    for f in ("gd_cell", "gd_light", "gd_cell_blocks", "gd_cell_over_filter", "gd_cell_over_sph", "gd_cell_big",
              "gd_light_cell_off", "gd_light_cand", "gd_light_head", "gd_light_always"):
        getattr(L, f).restype = vp
    L.gd_cell.argtypes = [vp, ll, ctypes.c_double]
    L.gd_light.argtypes = [vp, ll, vp, ctypes.c_int, ctypes.c_ulonglong]
    for f in ("gd_cell_n_blocks", "gd_cell_n_over", "gd_cell_n_big", "gd_light_n_entries", "gd_light_n_always"):
        getattr(L, f).restype = ll
        getattr(L, f).argtypes = [vp]
    for f in ("gd_cell_blocks", "gd_cell_over_filter", "gd_cell_over_sph", "gd_cell_big", "gd_light_cell_off",
              "gd_light_cand", "gd_light_head", "gd_light_always", "gd_cell_enabled", "gd_light_ok", "gd_cell_free",
              "gd_light_free"):
        getattr(L, f).argtypes = [vp]
    L.gd_cell_geometry.argtypes = [vp, vp, vp, vp, vp]
    return L


def device_cell(L, sph, density):
    g = L.gd_cell(sph.ctypes.data, len(sph), density)
    assert g, "CUDA error in the device cell-grid builder"
    res, lo, hi, cs = np.zeros(3, np.int32), np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(3, np.float32)
    L.gd_cell_geometry(g, res.ctypes.data, lo.ctypes.data, hi.ctypes.data, cs.ctypes.data)
    n_over = L.gd_cell_n_over(g)
    out = (bool(L.gd_cell_enabled(g)), res.tobytes() + lo.tobytes() + hi.tobytes() + cs.tobytes(),
           raw(L.gd_cell_blocks(g), 128 * L.gd_cell_n_blocks(g)), raw(L.gd_cell_over_filter(g), 16 * n_over),
           raw(L.gd_cell_over_sph(g), 4 * n_over), raw(L.gd_cell_big(g), 4 * L.gd_cell_n_big(g)))
    L.gd_cell_free(g)
    return out


def device_light(L, sph, light, res, budget=MAX_ENTRIES):
    """(cell_off, cand, head, always) of the device builder, or None when it refuses the light."""
    light = np.ascontiguousarray(light, dtype=np.float64)
    g = L.gd_light(sph.ctypes.data, len(sph), light.ctypes.data, res, budget)
    assert g, "CUDA error in the device direction-grid builder"
    if not L.gd_light_ok(g):
        L.gd_light_free(g)
        return None
    nc, ne, na = 6 * res * res, L.gd_light_n_entries(g), L.gd_light_n_always(g)
    out = (raw(L.gd_light_cell_off(g), 4 * (nc + 1)), raw(L.gd_light_cand(g), 32 * ne),
           raw(L.gd_light_head(g), 32 * nc), raw(L.gd_light_always(g), 4 * na))
    L.gd_light_free(g)
    return out


def _shifted(flat, by):
    flat.spheres['center'] = flat.spheres['center'] + by
    flat.lights['location'] = flat.lights['location'] + by
    return flat


SCENES = {
    "c3": lambda: sc.synthetic_scene("c3"),
    "c4": lambda: sc.synthetic_scene("c4"),
    "clustered": lambda: clustered_scene()[0],
    "m3": lambda: sc.mesh_scene("m3"),
    "c3_shift_300": lambda: _shifted(sc.synthetic_scene("c3"), 300.3),      # centres no longer float32
    "c3_shift_1e4": lambda: _shifted(sc.synthetic_scene("c3"), 1e4),        # too far out for a cell grid
}


@pytest.mark.parametrize("name", list(SCENES))
def test_cell_grid_is_the_host_grid(gd, name):
    sph = sphere_table(SCENES[name]())
    for density in (0.35, 1.0):
        host = host_cell(gd, sph, density)
        dev = device_cell(gd, sph, density)
        assert host[0] == (name != "c3_shift_1e4"), (name, density)
        assert dev[0] == host[0], (name, density)
        if host[0]:
            for k, part in enumerate(("geometry", "blocks", "over_filter", "over_sph", "big")):
                assert dev[1 + k] == host[1 + k], (name, density, part)


def test_no_grid_cases_agree(gd):
    base = sphere_table(sc.synthetic_scene("c3"))
    cases = {}
    s = base.copy()
    s[:130, :3] = s[200, :3] + np.linspace(0, 1e-3, 130)[:, None]     # a knot: one cell with > 127 entries
    s[:130, 3] = 0.01
    cases["knot"] = s
    s = base.copy()
    s[:40, 3] = 30.0                                                  # 40 spheres over more than 512 cells each
    cases["big40"] = s
    s = base.copy()
    s[0, :3] = (2e6, 0.0, 0.0)                                        # abs_max beyond 1e6
    cases["far"] = s
    cases["255"] = base[:255].copy()                                  # fewer than kCellGridMinSpheres
    for name, s in cases.items():
        s = np.ascontiguousarray(s)
        for density in (0.35, 1.0):
            assert not host_cell(gd, s, density)[0], name
            assert not device_cell(gd, s, density)[0], name
    # 32 big spheres still make a grid, listed in sphere order
    s = base.copy()
    s[[3, 9, 700, 1200] + list(range(2000, 2028)), 3] = 30.0
    host, dev = host_cell(gd, s, 0.35), device_cell(gd, s, 0.35)
    assert host[0] and dev[0] and np.frombuffer(host[5], np.int32).size == 32
    assert dev[1:] == host[1:]


def special_lights(sph):
    k = len(sph) // 3
    c, r = sph[k, :3], abs(sph[k, 3])
    return [c + np.array([0.1, -0.2, 0.05]) * r,                      # inside a sphere
            c + np.array([1.0005 * r, 0.0, 0.0]),                     # just outside one
            np.array([1e4, -3e3, 2e3])]                               # far away: every sphere in a few cells


@pytest.mark.parametrize("name", list(SCENES))
def test_direction_grids_are_the_host_grids(gd, name):
    flat = SCENES[name]()
    sph = sphere_table(flat)
    lights = scene_lights(flat)[:8]
    plan = [(l, 128) for l in lights] + [(l, 32) for l in special_lights(sph)]
    if name != "c4":
        plan += [(l, 32) for l in lights] + [(l, 128) for l in special_lights(sph)]
    for i, (light, res) in enumerate(plan):
        host = host_light(gd, sph, light, res, packed=True)
        dev = device_light(gd, sph, light, res)
        assert (host is None) == (dev is None), (name, i, res)
        if host is None:
            continue
        cell_off, _, _, always, cand, head = host
        for part, a, b in (("cell_off", dev[0], cell_off), ("cand", dev[1], cand), ("head", dev[2], head),
                           ("always", dev[3], always)):
            assert a == b, (name, i, res, part)


def test_entry_budget_decides_like_the_host(gd):
    flat = sc.synthetic_scene("c3")
    sph = sphere_table(flat)
    light = scene_lights(flat)[0]
    host = host_light(gd, sph, light, 32)
    n = len(host[1]) // 8
    assert n > 0
    assert device_light(gd, sph, light, 32, budget=n - 1) is None
    dev = device_light(gd, sph, light, 32, budget=n)
    assert dev is not None and len(dev[1]) == 32 * n


def touched(light, d, centers, radii):
    oc = centers - light
    b = oc @ d
    disc = b * b - (np.einsum("ij,ij->i", oc, oc) - radii ** 2)
    return np.nonzero((disc >= 0) & (b + np.sqrt(np.maximum(disc, 0)) >= 0))[0]


@pytest.mark.parametrize("res", [16, 128])
def test_device_direction_grid_lists_every_touched_sphere(gd, res):
    """Completeness on the device's own arrays: the head and the cand range of the cell a shadow ray looks in
    (FP64 and FP32 cell rules), plus the always-list, hold every sphere the ray touches."""
    rng = np.random.default_rng(5)
    n = 4000
    centers = rng.uniform(-40, 40, (n, 3))
    radii = rng.uniform(0.2, 1.5, n)
    light = np.array([3.0, -7.0, 1.5])
    centers[0], radii[0] = light + [0.1, 0.2, -0.1], 1.0
    centers[1], radii[1] = light + [2.0, 0.0, 0.0], 1.999
    centers[2], radii[2] = light + [5.0, 5.0, 0.0], 2.0
    sph = np.ascontiguousarray(np.concatenate([centers, radii[:, None]], 1))
    off, cand, head, always = device_light(gd, sph, light, res)
    cand, head = np.frombuffer(cand, CAND_DT), np.frombuffer(head, CAND_DT)
    always = set(np.frombuffer(always, np.int32).tolist())
    assert 0 in always and 1 not in always
    d = rng.normal(size=(2000, 3))
    to_c = centers[rng.integers(0, n, 2000)] - light
    perp = np.cross(to_c, rng.normal(size=(2000, 3)))
    perp /= np.linalg.norm(perp, axis=1, keepdims=True)
    rim = to_c + perp * radii[rng.integers(0, n, 2000), None] * rng.uniform(0.9, 1.0, (2000, 1))
    special = np.array([[1, 1, 0], [1, -1, 0], [0, 1, 1], [1, 1, 1], [-1, 1, 1], [1, 0, 0], [0, 0, -1], [-1, -1, -1],
                        [1, 1, 1e-17], [1, 1 - 1e-16, 0]], dtype=np.float64)
    dirs = np.concatenate([d, rim, special])
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    n_touch = 0
    for k in range(len(dirs)):
        hit = touched(light, dirs[k], centers, radii)
        n_touch += len(hit)
        dk = np.ascontiguousarray(dirs[k])
        d32 = np.ascontiguousarray(dirs[k] * 1.0000019073486328, dtype=np.float32)
        for c in (gd.gh_light_cell(dk.ctypes.data, res), gd.gh_light_cell_f32(d32.ctypes.data, res)):
            h = head[c]
            listed = set(always)
            if h["sphere"] >= 0:
                listed.add(int(h["sphere"]))
                listed |= set(cand["sphere"][h["pad"][0]:h["pad"][1]].tolist())
            assert set(hit.tolist()) <= listed, (k, dirs[k])
    assert n_touch > 2000


# ---- through the C ABI ------------------------------------------------------------------------------------------

def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _grids(dev, flat):
    """(has_cell_grid, light_grids) of a scene, read with an update that changes nothing."""
    info = flat.update(dev)
    assert info["changed"] == [] and info["done"] == [], info
    return info["has_cell_grid"], info["light_grids"]


def _frames(dev, accels, w=64, h=36, depth=3):
    return {a: dev.render(w, h, depth, fmt="f64", accel=a) for a in accels}


def _counters(dev, accels, w=64, h=36, depth=3):
    out = {}
    for a in accels:
        _, st = dev.render(w, h, depth, fmt="f64", accel=a, flags=_lib.FLAG_COUNT_TESTS)
        out[a] = {k: st[k] for k in COUNTERS}
    return out


def _assert_like_fresh(dev, flat, accels=RENDER_ACCELS, counters=False):
    """Same grids and bit-equal frames as a fresh create of `flat`; with counters, also every test counter of every
    accel.  Counters need the scene back at the tables its BVHs were built from: a refitted tree prunes less tightly
    than a built one, so away from them the BVH walks count more box and filter tests whatever the grids hold."""
    fresh = flat.upload(0)
    try:
        assert _grids(dev, flat) == _grids(fresh, flat)
        got, want = _frames(dev, accels), _frames(fresh, accels)
        for a in accels:
            assert np.array_equal(_bits(got[a][0]), _bits(want[a][0])), a
            assert got[a][1]["rays"] == want[a][1]["rays"], a
        if counters:
            assert _counters(dev, accels) == _counters(fresh, accels)
    finally:
        fresh.close()


TABLE_BYTES = {"spheres": lambda f: 32 * len(f.spheres), "light_pos": lambda f: 72 * len(f.lights),
               "lights": lambda f: 72 * len(f.lights), "triangles": lambda f: 72 * len(f.triangles),
               "camera": lambda f: 0}


def _changed_bytes(info, flat):
    return sum(TABLE_BYTES[c](flat) for c in set(info["changed"]))


def _hand_moved(flat, k):
    """every tenth sphere shifted and resized, the first light moved"""
    s = flat.spheres
    s['center'][::10] += np.array([0.37, -0.21, 0.55]) * k
    s['radius'][::10] *= 1.0 + 0.05 * k
    flat.lights['location'][0] += (0.5 * k, 0.25, -0.5)
    return flat


ABI_SCENES = {
    "c3": (lambda: sc.synthetic_scene("c3"), lambda k: sc.animated_scene("c3", k)),
    "clustered": (lambda: clustered_scene()[0], lambda k: _hand_moved(clustered_scene()[0], k)),
    "m3": (lambda: sc.mesh_scene("m3"), lambda k: sc.animated_scene("m3", k)),
    "c4": (lambda: sc.synthetic_scene("c4"), lambda k: sc.animated_scene("c4", k)),
}


@pytest.mark.parametrize("name", list(ABI_SCENES))
def test_rebuilt_grids_equal_a_fresh_create(gpu, name):
    still, moved = ABI_SCENES[name]
    accels = FAST_ACCELS if name == "c4" else RENDER_ACCELS
    dev = still().upload(0)
    for k in (5, 16):
        flat = moved(k)
        info = flat.update(dev, rebuild_grids=True)
        assert "spheres" in info["changed"], info
        assert "rebuild_cell_grid" in info["done"] and "rebuild_light_grids" in info["done"], info
        assert info["h2d_bytes"] <= _changed_bytes(info, flat) + 4096, info
        assert info["device_ms"] > 0, info
        _assert_like_fresh(dev, flat, accels)
    if name == "c3":
        # hand-made moves of another kind on top
        flat = _hand_moved(sc.animated_scene("c3", 16), 3)
        info = flat.update(dev, rebuild_grids=True)
        assert info["h2d_bytes"] <= _changed_bytes(info, flat) + 4096, info
        _assert_like_fresh(dev, flat, accels)
    # back at the built tables the lists and their order show in the counters: the host's
    flat = still()
    info = flat.update(dev, rebuild_grids=True)
    assert "rebuild_cell_grid" in info["done"] and info["light_grids_rebuilt"] == info["light_grids"], info
    _assert_like_fresh(dev, flat, accels, counters=True)
    dev.close()


def test_grids_grow_and_shrink_back(gpu):
    still = sc.synthetic_scene("c3")
    dev = still.upload(0)
    spread = sc.synthetic_scene("c3")
    spread.spheres['center'] = spread.spheres['center'] * 2.0
    info = spread.update(dev, rebuild_grids=True)
    assert info["has_cell_grid"] == 1, info
    _assert_like_fresh(dev, spread)
    info = still.update(dev, rebuild_grids=True)
    _assert_like_fresh(dev, still, counters=True)
    spread.update(dev, rebuild_grids=True)
    _assert_like_fresh(dev, spread, FAST_ACCELS)
    dev.close()


def test_light_only_move_rebuilds_that_light(gpu):
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    flat.lights['location'][1] = (-25.0, -12.0, 25.0)
    info = flat.update(dev, rebuild_grids=True)
    assert "light_pos" in info["changed"], info
    assert info["done"] == ["rebuild_light_grids"] and info["light_grids_rebuilt"] == 1, info
    assert info["has_cell_grid"] == 1 and info["light_grids"] == 3, info
    assert info["h2d_bytes"] <= _changed_bytes(info, flat) + 4096, info
    _assert_like_fresh(dev, flat, counters=True)
    dev.close()


def test_dropped_grids_come_back_with_a_later_update(gpu):
    still = sc.synthetic_scene("c3")
    dev = still.upload(0)
    flat = sc.animated_scene("c3", 8)
    info = flat.update(dev)
    assert info["has_cell_grid"] == 0 and info["light_grids"] == 0, info
    info = flat.update(dev, rebuild_grids=True)
    assert info["changed"] == [], info
    assert "rebuild_cell_grid" in info["done"] and info["light_grids_rebuilt"] == 3, info
    assert info["h2d_bytes"] <= 4096, info
    _assert_like_fresh(dev, flat)
    # the same after the spheres went back (default update: dropped again), then an update that changes nothing
    info = still.update(dev)
    assert info["has_cell_grid"] == 0 and info["light_grids"] == 0, info
    info = still.update(dev, rebuild_grids=True)
    assert info["changed"] == [] and info["h2d_bytes"] <= 4096, info
    _assert_like_fresh(dev, still, counters=True)
    dev.close()


def test_drift_over_64_steps(gpu):
    dev = sc.synthetic_scene("c3").upload(0)
    for k in range(1, 65):
        flat = sc.animated_scene("c3", k)
        info = flat.update(dev, rebuild_grids=True)
        assert info["has_cell_grid"] == 1 and info["light_grids"] == 3, (k, info)
    _assert_like_fresh(dev, flat)
    still = sc.synthetic_scene("c3")
    still.update(dev, rebuild_grids=True)
    _assert_like_fresh(dev, still, counters=True)
    dev.close()


def test_a_knot_drops_the_cell_grid_until_it_disperses(gpu):
    still = sc.synthetic_scene("c3")
    dev = still.upload(0)
    knot = sc.synthetic_scene("c3")
    order = np.argsort(knot.spheres['order'])
    idx = order[:130]
    knot.spheres['center'][idx] = knot.spheres['center'][order[200]] + np.linspace(0, 1e-3, 130)[:, None]
    knot.spheres['radius'][idx] = 0.01
    info = knot.update(dev, rebuild_grids=True)
    assert info["has_cell_grid"] == 0 and "rebuild_cell_grid" in info["done"], info
    _assert_like_fresh(dev, knot)
    info = still.update(dev, rebuild_grids=True)
    assert info["has_cell_grid"] == 1, info
    _assert_like_fresh(dev, still, counters=True)
    dev.close()


def test_clone_of_a_device_rebuilt_scene(gpu):
    dev = sc.synthetic_scene("c3").upload(0)
    flat = sc.animated_scene("c3", 16)
    flat.update(dev, rebuild_grids=True)
    want, cnt = _frames(dev, RENDER_ACCELS), _counters(dev, RENDER_ACCELS)
    clone = dev.clone(0)
    got = _frames(clone, RENDER_ACCELS)
    for a in RENDER_ACCELS:
        assert np.array_equal(_bits(got[a][0]), _bits(want[a][0])), a
    assert _counters(clone, RENDER_ACCELS) == cnt
    assert _grids(clone, flat) == _grids(dev, flat)
    # updating the clone leaves its source alone
    sc.animated_scene("c3", 40).update(clone, rebuild_grids=True)
    again = _frames(dev, RENDER_ACCELS)
    for a in RENDER_ACCELS:
        assert np.array_equal(_bits(again[a][0]), _bits(want[a][0])), a
    assert _counters(dev, RENDER_ACCELS) == cnt
    clone.close()
    dev.close()
