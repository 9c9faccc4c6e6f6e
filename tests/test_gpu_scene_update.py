"""ert_scene_update on the GPU: a scene updated in place renders exactly what a fresh ert_scene_create of the same
tables renders, for every accel, and keeps its other promises (unchanged scenes on errors, queued frames, clones)."""
import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import assert_double_parity, clustered_scene, oracle_frame, quantise

pytestmark = pytest.mark.gpu

RENDER_ACCELS = ("exact", "linear", "bvh", "bvh_mega", "grid", "auto")
TRACE_ACCELS = ("exact", "linear", "bvh", "bvh_mega", "grid", "warp", "auto")
COUNTERS = ("rays", "sphere_filter_tests", "box_tests", "exact_sphere_tests", "exact_other_tests", "cell_steps")


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _frames(dev, w, h, depth, accels=RENDER_ACCELS, **kw):
    return {a: dev.render(w, h, depth, fmt="f64", accel=a, **kw) for a in accels}


def _assert_same_frames(got, want):
    """Bit-equal frames and equal ray counts, accel for accel (a dropped grid changes the accel a request runs, not
    the frame)."""
    for a in want:
        f, st = got[a]
        g, st2 = want[a]
        assert np.array_equal(_bits(f), _bits(g)), a
        assert st["rays"] == st2["rays"], a


def _assert_all_equal(got, ref):
    g, st2 = ref
    for a, (f, st) in got.items():
        assert np.array_equal(_bits(f), _bits(g)), a
        assert st["rays"] == st2["rays"], a


def _counters(dev, w, h, depth, accels=RENDER_ACCELS):
    out = {}
    for a in accels:
        _, st = dev.render(w, h, depth, fmt="f64", accel=a, flags=_lib.FLAG_COUNT_TESTS)
        out[a] = {k: st[k] for k in COUNTERS}
    return out


def _demo_moved(k):
    flat = sc.flatten(sc.demo_scene())
    flat.spheres['center'] += np.array([[0.3, -0.2, 0.5]]) * k
    flat.spheres['radius'] *= 1.0 + 0.1 * k
    flat.triangles['v2'] += np.array([0.5, 0.25, -1.0]) * k
    flat.lights['location'][0] += (1.0 * k, 0.5, 0.0)
    return flat


def _clustered_moved(k):
    flat, _ = clustered_scene()
    moved = sc._moved_spheres(flat.spheres, 0x5EED, k)
    return sc.FlatScene(flat.camera, flat.lights, moved, flat.triangles, flat.planes)


SCENES = {
    "demo": (lambda: sc.flatten(sc.demo_scene()), _demo_moved),
    "c3": (lambda: sc.synthetic_scene("c3"), lambda k: sc.animated_scene("c3", k)),
    "clustered": (lambda: clustered_scene()[0], _clustered_moved),
    "m3": (lambda: sc.mesh_scene("m3"), lambda k: sc.animated_scene("m3", k)),
}


def test_identity_update_changes_nothing(gpu):
    for name in ("c3", "m3"):
        flat = SCENES[name][0]()
        dev = flat.upload(0)
        before = _frames(dev, 64, 36, 3)
        cnt = _counters(dev, 64, 36, 3)
        info = flat.update(dev)
        assert info["changed"] == [] and info["done"] == [], info
        assert info["has_cell_grid"] == before["grid"][1]["has_cell_grid"], info
        assert info["light_grids"] == 3 and info["h2d_bytes"] == 0, info
        _assert_same_frames(_frames(dev, 64, 36, 3), before)
        assert _counters(dev, 64, 36, 3) == cnt
        dev.close()


def test_round_trip_reproduces_the_build(gpu):
    """update(k) then update(0): the device's refit, filters and constants give the host's bits back (every counter
    of every accel equal to the fresh scene's; the grids are rebuilt from the same inputs)."""
    for name in ("c3", "clustered", "m3"):
        still, moved = SCENES[name]
        dev = still().upload(0)
        cnt = _counters(dev, 64, 36, 3)
        before = _frames(dev, 64, 36, 3)
        grids = still().update(dev)
        info = moved(16).update(dev)
        assert "refit_spheres" in info["done"] and info["sphere_area_ratio"] != 1.0, info
        info = still().update(dev, rebuild_grids=True)
        assert abs(info["sphere_area_ratio"] - 1.0) < 1e-12, info
        if name == "m3":
            assert "refit_triangles" in info["done"] and abs(info["triangle_area_ratio"] - 1.0) < 1e-12, info
        assert (info["has_cell_grid"], info["light_grids"]) == (grids["has_cell_grid"], grids["light_grids"]), info
        assert _counters(dev, 64, 36, 3) == cnt, name
        _assert_same_frames(_frames(dev, 64, 36, 3), before)
        dev.close()


@pytest.mark.parametrize("name", list(SCENES))
def test_moved_scene_equals_a_fresh_create(gpu, name):
    still, moved = SCENES[name]
    dev = still().upload(0)
    for k in (5, 16):
        flat = moved(k)
        info = flat.update(dev)
        assert "spheres" in info["changed"], info
        fresh = flat.upload(0)
        for depth in (1, 4):
            _assert_same_frames(_frames(dev, 80, 45, depth), _frames(fresh, 80, 45, depth))
        fresh.close()
    # the reference itself on a lattice of pixels
    w, h, depth = 48, 27, 3
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    for a in ("bvh", "grid", "auto"):
        f, st = dev.render(w, h, depth, fmt="f64", accel=a)
        q, _ = dev.render(w, h, depth, fmt="rgb8", accel=a)
        assert st["rays"] == ref_rays, a
        assert np.array_equal(q.astype(np.int64), quantise(ref)), a
        assert_double_parity(f, ref)
    dev.close()


def test_c4_band_after_animation_steps(gpu):
    dev = sc.synthetic_scene("c4").upload(0)
    for k in (1, 2, 13):
        flat = sc.animated_scene("c4", k)
        info = flat.update(dev)
    assert info["h2d_bytes"] == 32 * len(flat.spheres), info
    assert "drop_cell_grid" in info["done"] or info["has_cell_grid"] == 0, info
    fresh = flat.upload(0)
    W, H, n_parts = 3840, 2160, 270
    for part in (0, 130):
        for a in ("bvh", "bvh_mega", "grid", "auto"):
            f, st = dev.render(W, H, 5, fmt="f64", accel=a, band_rows=8, n_parts=n_parts, part=part)
            g, st2 = fresh.render(W, H, 5, fmt="f64", accel=a if a in ("bvh", "bvh_mega") else "bvh",
                                  band_rows=8, n_parts=n_parts, part=part)
            rows = slice(8 * part, 8 * part + 8)
            assert np.array_equal(_bits(f[rows]), _bits(g[rows])), (part, a)
            assert st["rays"] == st2["rays"], (part, a)
    dev.close()
    fresh.close()


def test_trace_rays_equal_a_fresh_create(gpu):
    still = sc.synthetic_scene("c3")
    dev = still.upload(0)
    flat = sc.animated_scene("c3", 16)
    flat.update(dev)
    fresh = flat.upload(0)
    rng = np.random.default_rng(9)
    n = 100_000
    O = rng.uniform(-10, 10, (n, 3)) + np.array([0, -10, -2])
    D = rng.normal(0, 1, (n, 3)) + np.array([0, 0, 1.5])
    old_c, new_c = still.spheres['center'], flat.spheres['center']
    k = rng.integers(0, len(old_c), 20_000)
    Oa = np.repeat(np.array([[0.0, 0.0, -2.0]]), 2 * len(k), axis=0)
    Da = np.concatenate([old_c[k], new_c[k]]) - Oa
    rays = np.ascontiguousarray(np.concatenate([np.concatenate([O, D], 1), np.concatenate([Oa, Da], 1)]))
    for a in TRACE_ACCELS:
        o, t = dev.trace_rays(rays, accel=a)
        o2, t2 = fresh.trace_rays(rays, accel=a)
        assert np.array_equal(o, o2) and np.array_equal(_bits(t), _bits(t2)), a
    # the rays aimed at the new centres reach many of the moved spheres (C3 is dense: the others are occluded)
    o, _ = dev.trace_rays(rays[n + len(k):], accel="bvh")
    assert (o == flat.spheres['order'][k]).mean() > 0.1
    dev.close()
    fresh.close()


def test_repeated_updates_drift(gpu):
    dev = sc.synthetic_scene("c3").upload(0)
    for k in range(1, 65):
        flat = sc.animated_scene("c3", k)
        flat.update(dev)
        if k % 8 == 0:
            fresh = flat.upload(0)
            _assert_all_equal(_frames(dev, 64, 36, 3, ("bvh", "grid", "auto")), fresh.render(64, 36, 3, fmt="f64",
                                                                                             accel="bvh"))
            fresh.close()
    dev.close()


def test_partial_changes(gpu):
    still = sc.synthetic_scene("c3")
    dev = still.upload(0)
    # materials only: both kinds of grid stay
    flat = sc.synthetic_scene("c3")
    flat.spheres['material']['colour'] = flat.spheres['material']['colour'][:, ::-1]
    flat.planes['material']['reflectivity'] = 0.5
    info = flat.update(dev)
    assert set(info["changed"]) == {"sphere_mat", "planes"} and info["done"] == [], info
    assert info["has_cell_grid"] == 1 and info["light_grids"] == 3, info
    fresh = flat.upload(0)
    _assert_same_frames(_frames(dev, 64, 36, 3), _frames(fresh, 64, 36, 3))
    fresh.close()
    # light 1 moved: the cell grid stays, its direction grid (and the ones after it) are cut
    flat.lights['location'][1] = (-25.0, -12.0, 25.0)
    info = flat.update(dev)
    assert "light_pos" in info["changed"] and "drop_light_grids" in info["done"], info
    assert info["has_cell_grid"] == 1 and info["light_grids"] == 1, info
    fresh = flat.upload(0)
    _assert_same_frames(_frames(dev, 64, 36, 3), _frames(fresh, 64, 36, 3))
    fresh.close()
    # spheres moved: the cell grid is dropped, REBUILD_GRIDS brings every grid back
    flat = sc.animated_scene("c3", 8)
    flat.lights['location'][1] = (-25.0, -12.0, 25.0)
    info = flat.update(dev)
    assert info["has_cell_grid"] == 0 and info["light_grids"] == 0, info
    assert dev.render(16, 9, 1, accel="grid")[1]["accel_used"] == "bvh"
    info = flat.update(dev, rebuild_grids=True)
    assert info["has_cell_grid"] == 1 and info["light_grids"] == 3, info
    assert "rebuild_cell_grid" in info["done"] and info["light_grids_rebuilt"] == 3, info
    fresh = flat.upload(0)
    _assert_same_frames(_frames(dev, 64, 36, 3), _frames(fresh, 64, 36, 3))
    # REBUILD: the create path, counters equal to the fresh scene's
    sc.animated_scene("c3", 20).update(dev)
    info = flat.update(dev, rebuild=True)
    assert "rebuild" in info["done"] and info["sphere_area_ratio"] == 1.0, info
    assert _counters(dev, 64, 36, 3) == _counters(fresh, 64, 36, 3)
    fresh.close()
    dev.close()


def test_triangle_past_the_float_range_rebuilds_the_triangle_tree(gpu):
    flat = sc.mesh_scene("m3")
    dev = flat.upload(0)
    far = sc.mesh_scene("m3")
    far.triangles['v1'][100] = (2e30, 0.0, 50.0)
    info = far.update(dev)
    assert "rebuild_tri_bvh" in info["done"], info
    fresh = far.upload(0)
    _assert_same_frames(_frames(dev, 64, 36, 3), _frames(fresh, 64, 36, 3))
    fresh.close()
    # and back: the triangle returns to the tree of a rebuilt scene
    info = flat.update(dev)
    assert "refit_triangles" in info["done"], info
    fresh = flat.upload(0)
    _assert_same_frames(_frames(dev, 64, 36, 3), _frames(fresh, 64, 36, 3))
    fresh.close()
    dev.close()


def test_bad_updates_leave_the_scene_untouched(gpu):
    flat = sc.synthetic_scene("c3", n_spheres=500)
    dev = flat.upload(0)
    before = _frames(dev, 48, 27, 3, ("bvh", "auto"))
    bad = []
    f = sc.synthetic_scene("c3", n_spheres=500)
    bad.append((f.camera, f.lights, f.spheres[:-1], f.triangles, f.planes))             # wrong count
    f = sc.synthetic_scene("c3", n_spheres=500)
    f.spheres['order'][7] = 10_000                                                       # missing + extra order
    bad.append((f.camera, f.lights, f.spheres, f.triangles, f.planes))
    f = sc.synthetic_scene("c3", n_spheres=500)
    f.spheres['order'][7] = f.spheres['order'][8]                                        # duplicate order
    bad.append((f.camera, f.lights, f.spheres, f.triangles, f.planes))
    f = sc.synthetic_scene("c3", n_spheres=500)
    f.spheres['order'][7] = f.planes['order'][0]                                         # order of another kind
    bad.append((f.camera, f.lights, f.spheres, f.triangles, f.planes))
    f = sc.synthetic_scene("c3", n_spheres=500)
    f.spheres['center'][:, 0] += 1.0
    f.spheres['center'][499, 1] = np.nan                                                 # NaN after moved values
    bad.append((f.camera, f.lights, f.spheres, f.triangles, f.planes))
    for args in bad:
        with pytest.raises(_lib.BadArg):
            dev.update(*args)
        _assert_same_frames(_frames(dev, 48, 27, 3, ("bvh", "auto")), before)
    # the tables in another order are the same scene
    f = sc.synthetic_scene("c3", n_spheres=500)
    info = dev.update(f.camera, f.lights[::-1], f.spheres[::-1], f.triangles, f.planes)
    assert info["changed"] == [], info
    dev.close()


def test_frames_in_flight_render_the_old_scene(gpu):
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    w, h = 128, 72
    old = dev.render(w, h, 3, fmt="f64", accel="auto")[0]
    dev.render_async(w, h, 3, slot=0, fmt="f64", accel="auto")
    dev.render_async(w, h, 3, slot=1, fmt="f64", accel="bvh")
    moved = sc.animated_scene("c3", 16)
    moved.update(dev)
    for slot in (0, 1):
        out = np.zeros((h, w, 3))
        _lib.check(_lib.load().ert_download(dev.handle, slot, out.ctypes.data, out.nbytes))
        assert np.array_equal(_bits(out), _bits(old)), slot
    fresh = moved.upload(0)
    assert np.array_equal(_bits(dev.render(w, h, 3, fmt="f64", accel="auto")[0]),
                          _bits(fresh.render(w, h, 3, fmt="f64", accel="auto")[0]))
    fresh.close()
    dev.close()


def test_clones_of_updated_scenes(gpu):
    still = sc.mesh_scene("m3")
    dev = still.upload(0)
    moved = sc.animated_scene("m3", 16)
    moved.update(dev)
    want = _frames(dev, 64, 36, 3)
    clone = dev.clone(0)
    _assert_same_frames(_frames(clone, 64, 36, 3), want)
    # updating the clone leaves its source alone
    sc.animated_scene("m3", 40).update(clone)
    _assert_same_frames(_frames(dev, 64, 36, 3), want)
    clone.close()
    # every GPU: its own clone, updated, renders its part of the frame
    w, h, depth = 96, 54, 3
    full, _ = dev.render(w, h, depth, fmt="f64")
    base = still.upload(0)
    clones = [base.clone(g) for g in range(gpu)]
    out = np.zeros_like(full)
    for g, c in enumerate(clones):
        moved.update(c)
        f, _ = c.render(w, h, depth, fmt="f64", band_rows=8, n_parts=gpu, part=g)
        for b in range(g, (h + 7) // 8, gpu):
            out[8 * b:8 * b + 8] = f[8 * b:8 * b + 8]
    assert np.array_equal(_bits(out), _bits(full))
    for c in clones:
        c.close()
    base.close()
    dev.close()
