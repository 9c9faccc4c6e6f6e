"""Every sphere kernel at large magnitudes, held to the FP64 reference.

The FP32 sphere filter and the sphere slab tests are sound while |o|_inf + abs_max stays below kFilterRange (1e17,
ert_device.cuh).  A ray beyond it decides every sphere with the literal FP64 test (scan_spheres_instead), and the
scans without a tree pass every sphere through the filter (tests/test_filter_range.py checks both on the CPU).  The
scenes here put a sphere, a light, the camera or a ray origin beyond that range, and past FLT_MAX:

1. Far planet: C3 cut to 40, 300 and 3000 spheres (either side of the 16/17, 192/193 and 256 switches) and one big
   sphere at distance / radius 5e16 / 5e15 up to 1e100 / 1e99, in the view, behind and beside near spheres; depth 1
   and 4, so reflection rays leave the planet from origins around its distance and come back.
2. Distant light: one of the three lights at 1e16 ... 1e39 in two directions, near spheres shadowing each other,
   under every shadow sequence of launch_wavefront (fused, binned, unsorted, the scan), told apart by launch counts.
3. Far origins: a camera 1e20 from the scene with its screen scaled so that the primary rays spread, the whole scene
   translated by 1e18 and 1e20, and ray batches from far origins along axis-parallel, denormal and grazing
   directions, for every trace accel.
4. Updates that move a sphere out to a planet's place and a light out to a distant one and back: equal to a fresh
   create of the same tables, and to the oracle.
Every frame is rendered a second time with FLAG_COUNT_TESTS, which must change no bit, ray count or launch.

The references: oracle_frame (the C restatement, FP64) with assert_double_parity, equal quantise and equal ray
counts; trace_rays(accel="exact") for ray batches, itself held to orc.nearest_batch.  Sphere colours are random per
sphere, the planet has its own and every light its own, so that a lost sphere or a dropped occluder changes a colour.

The TRI=0 instantiations that run the FP32 sphere filter or a sphere slab test (`cuobjdump --dump-resource-usage`
of libert_b200.so; C: COUNT = 0, 1 through _render; G: GRID = 0, 1), and the tests that reach them with a ray
beyond the range.  Every frame of a far-planet scene is out of range for every ray (abs_max holds the planet).

  render_free_kernel<3, C, 0>         test_far_planet (bvh_mega; auto at 40 spheres is linear)
  render_tiled_kernel<C, 0>           test_far_planet, test_distant_light (linear at 40 spheres)
  wf_scan<*, *, C> (and wf_scan_init / wf_scan_finish)
                                      test_far_planet, test_distant_light (linear at 300 and 3000 spheres)
  wf_trace_path<1, C, 1, G, 0>, <0, C, 1, G, 0>, <0, C, 0, G, 0>
                                      test_far_planet (bvh, grid, auto at 300 / 3000), test_distant_light (every
                                      shadow sequence), test_far_camera, test_translated_scene; G = 1 where a cell
                                      grid exists: the distant-light and far-camera scenes at 3000 spheres
  wf_trace_path_refill<C, G, *, 0>    bounces 2-3 of the depth-4 frames above
  wf_trace_shadow<C, 1, 0>, <C, 0, 0> test_distant_light (binned and unsorted, with and without FLAG_NO_LIGHT_GRID),
                                      test_far_planet at 40 spheres (no direction grids below 64 spheres)
  wf_shadow_shade<C, 0>               test_distant_light and test_far_planet at 300 / 3000 spheres, no flags
  trace_rays_kernel<2, 0>, <3, 0>, <4, 0>, <5, 0>, trace_rays_warp_kernel<0>
                                      test_far_origin_rays
"""
import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import oracle_scene_from_flat
from oracle import orc
from test_gpu_grid_build import _assert_like_fresh, _grids
from test_gpu_limits import _assert_oracle, _bits
from test_gpu_mesh_paths import NLG, SHADOW_FLAGS, UNSORTED, _oracle_ref, _render, wavefront_launches

pytestmark = pytest.mark.gpu

RENDER_ACCELS = ("auto", "exact", "linear", "bvh", "bvh_mega", "grid")
TRACE_ACCELS = ("linear", "bvh", "bvh_mega", "grid", "warp", "auto")
SIZES = (40, 300, 3000)
W, H = 64, 36
# distance / radius of the planet; the last two have centres past FLT_MAX
PLANETS = [(5e16, 5e15), (2e19, 2e18), (1e20, 1e19), (1e30, 1e29), (1e39, 1e38), (1e100, 1e99)]
LIGHT_DISTANCES = (1e16, 2e19, 1e20, 1e30, 1e39)
LIGHT_DIRECTIONS = ((0.3, -1.0, -0.2), (-1.0, -0.5, 0.4))


def _base(n):
    flat = sc.synthetic_scene("c3", n_spheres=n)
    flat.lights['diffuse_colour'] = [(1.0, 0.9, 0.3), (0.2, 0.4, 1.0), (0.9, 0.2, 0.6)]
    flat.lights['specular_colour'] = [(0.8, 0.7, 0.2), (0.1, 0.9, 0.4), (0.6, 0.3, 0.9)]
    return flat


def _renumbered(flat):
    """orders in table order: lights, spheres, planes"""
    at = 0
    for t in (flat.lights, flat.spheres, flat.triangles, flat.planes):
        t['order'] = np.arange(at, at + len(t))
        at += len(t)
    return flat


def _planet(dist, radius):
    p = np.zeros(1, dtype=_lib.SPHERE_DT)
    # up and to the right of the view's middle: part of the frame, behind and beside the near spheres
    d = np.array([0.45, -0.25, 1.0])
    p['center'] = d / np.linalg.norm(d) * dist
    p['radius'] = radius
    p['material']['colour'] = (0.3, 0.8, 0.7)
    p['material']['specular_power'] = 4.0
    p['material']['shininess'] = 0.4
    p['material']['reflectivity'] = 0.5
    return p


def with_planet(flat, dist, radius):
    return _renumbered(sc.FlatScene(flat.camera, flat.lights.copy(), np.concatenate([flat.spheres, _planet(dist, radius)]),
                                    flat.triangles.copy(), flat.planes.copy()))


def with_far_light(flat, dist, direction, k=0):
    out = sc.FlatScene(flat.camera, flat.lights.copy(), flat.spheres.copy(), flat.triangles.copy(), flat.planes.copy())
    d = np.asarray(direction, float)
    out.lights['location'][k] = d / np.linalg.norm(d) * dist
    return out


def _expected_used(flat, accel, cell_grid):
    n = len(flat.spheres)
    if accel == "auto":
        return "exact" if n <= 16 else "linear" if n <= 192 else "grid" if (n >= 256 and cell_grid) else "bvh"
    if accel == "grid":
        return "grid" if cell_grid else "bvh"
    return accel


def _launches(flat, used, flags, depth, light_grids):
    if used in ("exact", "bvh_mega") or (used == "linear" and len(flat.spheres) <= 192):
        return 1
    if used == "linear":
        return wavefront_launches("scan", depth)
    fused = not (flags & NLG) and light_grids == len(flat.lights) and len(flat.lights) <= 8
    return wavefront_launches("fused" if fused else "unsorted" if flags & UNSORTED else "binned", depth)


def _check_all(flat, depths=(1, 4), flag_sets=SHADOW_FLAGS, accels=RENDER_ACCELS):
    """Every accel (and, for the walked wavefront paths, every shadow sequence) against the oracle, with the accel
    and the launch count each must have.  Returns {(accel, flags, depth): accel_used}."""
    dev = flat.upload(0)
    used = {}
    try:
        cell_grid, light_grids = _grids(dev, flat)
        for depth in depths:
            ref = _oracle_ref(flat, depth)
            for accel in accels:
                want = _expected_used(flat, accel, cell_grid)
                walked = want in ("bvh", "grid")
                for flags in (flag_sets if walked else (0,)):
                    f, st, _ = _render(dev, W, H, depth, accel, flags)
                    what = (accel, flags, depth, len(flat.spheres))
                    _assert_oracle(f, st, ref[0], ref[1], what)
                    assert st["accel_used"] == want, (what, st["accel_used"])
                    assert st["gpu_launches"] == _launches(flat, want, flags, depth, light_grids), (what, st["gpu_launches"])
                    used[(accel, flags, depth)] = st["accel_used"]
        return used, cell_grid, light_grids
    finally:
        dev.close()


def _changed(a, b, tol=1e-6):
    return float((np.abs(a - b).max(axis=2) > tol).mean())


# ---- 1. far planet -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dist,radius", PLANETS, ids=["%g" % p[0] for p in PLANETS])
@pytest.mark.parametrize("n", SIZES)
def test_far_planet(gpu, n, dist, radius):
    base = _base(n)
    flat = with_planet(base, dist, radius)
    _check_all(flat)
    # the planet is in the picture: the oracle's frame differs from the scene without it
    a, _, _ = _oracle_ref(flat, 1)
    b, _, _ = _oracle_ref(_renumbered(base), 1)
    assert _changed(a, b) > 0


# ---- 2. distant light --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("direction", LIGHT_DIRECTIONS, ids=["d0", "d1"])
@pytest.mark.parametrize("dist", LIGHT_DISTANCES, ids=["%g" % d for d in LIGHT_DISTANCES])
@pytest.mark.parametrize("n", SIZES)
def test_distant_light(gpu, n, dist, direction):
    flat = with_far_light(_base(n), dist, direction)
    used, cell_grid, light_grids = _check_all(flat, depths=(4,))
    # the distant light lights the scene: without it the frame changes
    a, _, _ = _oracle_ref(flat, 4)
    dark = sc.FlatScene(flat.camera, flat.lights[1:].copy(), flat.spheres.copy(), flat.triangles.copy(),
                        flat.planes.copy())
    b, _, _ = _oracle_ref(dark, 4)
    assert _changed(a, b) > 0
    print("distant light %g %s: %d spheres, cell grid %d, direction grids %d" % (dist, direction, n, cell_grid, light_grids))


# ---- 3. far origins ----------------------------------------------------------------------------------------------

def far_camera(flat, dist):
    """the camera `dist` behind the scene, its screen scaled so that the primary rays spread over the view"""
    cam = _lib.Camera()
    cam.location[:] = (0.0, 0.0, -dist)
    cam.rotation[:] = tuple(flat.camera.rotation)
    cam.fov = flat.camera.fov
    cam.screen_width, cam.screen_height = 4.0 * dist * 1e-3, 2.25 * dist * 1e-3
    return sc.FlatScene(cam, flat.lights.copy(), flat.spheres.copy(), flat.triangles.copy(), flat.planes.copy())


def translated(flat, shift, scale=1.0):
    """everything scaled by `scale` and moved by `shift`; the screen scaled so that the focal length stays far above
    the ulp of the camera's coordinates"""
    T = np.asarray(shift, float)
    cam = _lib.Camera()
    cam.location[:] = tuple(np.array(flat.camera.location) * scale + T)
    cam.rotation[:] = tuple(flat.camera.rotation)
    cam.fov = flat.camera.fov
    s = 1e-12 * np.abs(T).max()
    cam.screen_width, cam.screen_height = flat.camera.screen_width * s, flat.camera.screen_height * s
    out = sc.FlatScene(cam, flat.lights.copy(), flat.spheres.copy(), flat.triangles.copy(), flat.planes.copy())
    out.lights['location'] = out.lights['location'] * scale + T
    out.spheres['center'] = out.spheres['center'] * scale + T
    out.spheres['radius'] *= scale
    out.planes['distance'] = out.planes['distance'] * scale - out.planes['normal'] @ T
    return out


@pytest.mark.parametrize("n", SIZES)
def test_far_camera(gpu, n):
    _check_all(far_camera(_base(n), 1e20), depths=(4,), flag_sets=(0, NLG))


# at 1e20 the coordinates' ulp is 16384: the scene is scaled by 1e5 first, so that its spheres stay apart
@pytest.mark.parametrize("shift,scale", [((0.0, 0.0, 1e18), 1.0), ((1e20, -1e20, 1e20), 1e5)], ids=["1e18", "1e20"])
@pytest.mark.parametrize("n", SIZES)
def test_translated_scene(gpu, n, shift, scale):
    flat = translated(_base(n), shift, scale)
    _check_all(flat, depths=(4,), flag_sets=(0, NLG))
    # the scene is in the picture
    assert (_oracle_ref(flat, 1)[0].max(axis=2) > 0).mean() > 0.05


def _far_rays(flat, rng, n):
    """Rays from far origins: at sphere centres, at grazing points (impact parameter r (1 - 1e-6)), along the axes and
    with denormal direction components."""
    C = flat.spheres['center']
    r = flat.spheres['radius']
    out = []
    for o_dist in (1e16, 1e18, 2e19, 1e20, 1e30):
        for axis in range(3):
            for sign in (1.0, -1.0):
                O = np.zeros(3)
                O[axis] = sign * o_dist
                k = rng.integers(0, len(C), n)
                target = C[k].copy()
                graze = rng.random(n) < 0.5
                perp = np.zeros((n, 3))
                perp[:, (axis + 1) % 3] = 1.0
                target[graze] += perp[graze] * (r[k][graze] * (1.0 - 1e-6))[:, None]
                D = target - O
                D /= np.linalg.norm(D, axis=1, keepdims=True)
                # axis-parallel, and with a denormal component
                ax = rng.random(n) < 0.25
                D[ax] = 0.0
                D[ax, axis] = -sign
                den = rng.random(n) < 0.25
                D[den, (axis + 2) % 3] = 1e-310
                out.append(np.hstack([np.broadcast_to(O, (n, 3)), D]))
    return np.ascontiguousarray(np.concatenate(out))


def _assert_batches(dev, flat, rays):
    oe, te = dev.trace_rays(rays, accel="exact")
    _, kind, f = oracle_scene_from_flat(flat)
    oi, ot = orc.nearest_batch(rays, kind, f)
    assert np.array_equal(oi, oe) and np.array_equal(_bits(ot), _bits(te))
    for accel in TRACE_ACCELS:
        o, t = dev.trace_rays(rays, accel=accel)
        bad = np.flatnonzero((o != oe) | (_bits(t) != _bits(te)))
        assert bad.size == 0, (accel, bad.size, rays[bad[:3]], o[bad[:3]], oe[bad[:3]])
    return oe


@pytest.mark.parametrize("planet", [None, (1e20, 1e19), (1e39, 1e38)], ids=["none", "1e20", "1e39"])
@pytest.mark.parametrize("n", SIZES)
def test_far_origin_rays(gpu, n, planet):
    flat = _base(n) if planet is None else with_planet(_base(n), *planet)
    dev = flat.upload(0)
    try:
        oe = _assert_batches(dev, flat, _far_rays(flat, np.random.default_rng(n), 200))
        assert (oe >= 0).any()
        if planet is not None:
            # rays from the planet's surface back into the scene, and from the scene out to the planet
            p = flat.spheres[-1]
            rng = np.random.default_rng(n + 1)
            k = rng.integers(0, n, 2000)
            c = np.asarray(p['center'])
            u = c / np.linalg.norm(c)
            O = np.broadcast_to(c - u * p['radius'], (2000, 3)).copy()
            D = flat.spheres['center'][k] - O
            D /= np.linalg.norm(D, axis=1, keepdims=True)
            O2 = flat.spheres['center'][k]
            D2 = np.broadcast_to(u, (2000, 3)).copy()
            oe = _assert_batches(dev, flat, np.ascontiguousarray(np.vstack([np.hstack([O, D]), np.hstack([O2, D2])])))
            assert (oe == p['order']).any()
    finally:
        dev.close()


# ---- 4. updates --------------------------------------------------------------------------------------------------

def _moved_out(flat):
    out = sc.FlatScene(flat.camera, flat.lights.copy(), flat.spheres.copy(), flat.triangles.copy(), flat.planes.copy())
    out.spheres['center'][0] = _planet(2e19, 2e18)['center'][0]
    out.spheres['radius'][0] = 2e18
    out.lights['location'][0] = np.array(LIGHT_DIRECTIONS[0]) / np.linalg.norm(LIGHT_DIRECTIONS[0]) * 1e20
    return out


@pytest.mark.parametrize("n", SIZES)
def test_update_out_and_back(gpu, n):
    flat = _renumbered(_base(n))
    dev = flat.upload(0)
    try:
        for target in (_moved_out(flat), flat):
            target.update(dev, rebuild_grids=True)
            _assert_like_fresh(dev, target, accels=RENDER_ACCELS)
            ref = _oracle_ref(target, 3)
            for accel in RENDER_ACCELS:
                f, st, _ = _render(dev, W, H, 3, accel)
                _assert_oracle(f, st, ref[0], ref[1], (accel, n))
    finally:
        dev.close()
