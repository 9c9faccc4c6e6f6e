"""Every kernel that walks the triangle BVH, held to the FP64 reference.

A scene with at least kTriBvhMin (64) triangles has a triangle BVH, and every kernel that can reach its triangles
runs in its TRI=1 instantiation (scan_others / scan_others_shadow -> scan_tris_bvh).  Which instantiation runs
depends on the sphere count (16/17, 63/64, 192/193 and 256 switch the accel that AUTO picks, the megakernel or
wavefront behind LINEAR, the direction grids and the cell grid), on the number of lights and on the flags.  The
scenes here cross those thresholds with meshes cut from m3 and with small hand-built meshes:

1. mesh_case(n): m3's sheet under the view, two of its icospheres and the first n C3 spheres, for n either side of
   every threshold, and 63 / 64 triangles either side of the tree.
2. The four shadow sequences of launch_wavefront (fused, binned, unfused and unsorted, the scan), told apart by
   their launch counts (wavefront_launches).
3. The reference's triangle quirks in whole frames (raytracer.erl:442 has no sign test on t): a closed mesh behind
   the camera, around the camera, around a light and behind a light, and coincident triangles through the tree.
4. The always-list of scan_tris_bvh (huge triangles and one past 1e30) and its fallback scan, taken by every ray of
   a tree of triangles some 4e4 long and by rays with denormal direction components or components past 1e30.
5. Every frame rendered again with FLAG_COUNT_TESTS, which must change no bit; updates of mesh scenes, one of
   which grows a tree triangle so that the refitted tree's edge bound sends every ray to the fallback scan.

The references: oracle_frame (the C restatement, FP64) with assert_double_parity, equal quantise and equal ray
counts for frames; accel="exact" (the linear FP64 scan) bit for bit for m3-sized scenes and between GPU paths;
trace_rays(accel="exact") for ray batches, itself held to orc.nearest_batch.  Colours differ per object, per mesh
and per light, so that a wrong winner or a dropped light changes a colour, not a rounding.

The TRI=1 instantiations that `cuobjdump --dump-resource-usage` lists for libert_b200.so, and the tests that launch
them (C: COUNT = 0, 1, through _render's counted copy of every frame; G: GRID = 0, 1 of the wavefront kernels).
Each claim rests on an accel_used, flag or launch-count assertion of that test.

  render_free_kernel<3, C, 1>         test_few_sphere_mesh_scenes (auto and bvh_mega, accel_used == "bvh_mega",
                                      one launch), test_either_side_of_the_triangle_tree
  render_tiled_kernel<C, 1>           test_few_sphere_mesh_scenes (linear up to 192 spheres, one launch),
                                      test_the_quirks_in_whole_frames, test_the_fallback_scan_in_frames
  trace_rays_kernel<2, 1> (linear), <3, 1> (bvh_mega), <4, 1> (bvh; grid below 256 spheres), <5, 1> (grid at 3000
  spheres), trace_rays_warp_kernel<1>
                                      test_rays_the_walk_refuses_equal_exact, test_the_always_list
  wf_scan_init<0, 1, C, 1>, <0, 0, C, 1>, <1, 0, C, 1>
                                      test_few_sphere_mesh_scenes (linear at 193 spheres: 8d + 1 launches;
                                      depth 1 and 5 for the first and the later bounces)
  wf_shadow_shade<C, 1>               test_every_shadow_sequence_with_triangles (no flags, 64 and 3000 spheres:
                                      2d + 1 launches), test_the_quirks_in_whole_frames
  wf_trace_path<1, C, 1, G, 1>        every bvh / grid frame (bounce 0); G = 1 where accel_used == "grid"
  wf_trace_path<0, C, 1, G, 1>        bounce 1 of the fused and the unsorted sequences (2d + 1, 3d + 1 launches)
  wf_trace_path<0, C, 0, G, 1>        bounce 1 of the binned sequence (3 + 7(d - 1) + 1 launches: 17 and 63
                                      spheres, FLAG_NO_LIGHT_GRID, 9 lights)
  wf_trace_path_refill<C, G, 1, 1>    bounces 2-4 of the fused and unsorted sequences at depth 5
  wf_trace_path_refill<C, G, 0, 1>    bounces 2-4 of the binned sequence at depth 5
  wf_trace_shadow<C, 1, 1>            binned sequences without FLAG_NO_LIGHT_GRID: fewer than 64 spheres (no
                                      direction grids) and the 9-light m3, whose ninth light walks
  wf_trace_shadow<C, 0, 1>            FLAG_NO_LIGHT_GRID, with and without FLAG_WF_UNSORTED
                                      (test_every_shadow_sequence_with_triangles, test_the_quirks_in_whole_frames)

G = 1 needs a cell grid (256 spheres and more): the m3 cases of sections 2 and 3.  No TRI=1 instantiation is
unreachable."""
import functools

import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import oracle_frame, oracle_scene_from_flat
from oracle import orc
from test_gpu_grid_build import _assert_like_fresh
from test_gpu_limits import _assert_oracle, _bits, _lights, mesh_with_duplicates
from test_gpu_triangles import _edge_rays
from test_tri_bvh import tb  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu

RENDER_ACCELS = ("auto", "exact", "linear", "bvh", "bvh_mega", "grid")
TRACE_ACCELS = ("linear", "bvh", "bvh_mega", "grid", "warp", "auto")
NLG, UNSORTED = _lib.FLAG_NO_LIGHT_GRID, _lib.FLAG_WF_UNSORTED
SHADOW_FLAGS = (0, NLG, NLG | UNSORTED)
W, H = 64, 36
M3_LIGHTS = np.array([[5.0, -20.0, 0.0], [-30.0, -10.0, 20.0], [20.0, -40.0, 60.0]])
SHEET = 64 * 64 * 2            # m3's heightfield triangles come first in its table, then 10 icospheres of 1280


def wavefront_launches(seq, d):
    """gpu_launches of a wavefront frame of depth 1 <= d < 8 with at least one light (launch_wavefront, ert_api.cu),
    the closing wf_finalize included.  Per bounce:
      fused     path walk (emits its hits), wf_shadow_shade
      unsorted  path walk (emits its hits), wf_trace_shadow, wf_shade
      binned    bounce 0 as unsorted; later bounces path walk, wf_emit_hits, three wf_bin_* kernels, wf_trace_shadow,
                wf_shade
      scan      wf_scan_init, wf_scan, wf_scan_finish, wf_emit_hits, then the same three for the shadow rays, wf_shade
    """
    return {"fused": 2 * d, "unsorted": 3 * d, "binned": 3 + 7 * (d - 1), "scan": 8 * d}[seq] + 1


def shadow_sequence(flat, flags):
    """The sequence launch_wavefront runs for the BVH or cell-grid path walks: shadow rays and the light fold in one
    kernel when every light has a direction grid (64 spheres and more, at most 8 lights) and the hits stay in
    arrival order; otherwise walked shadow rays, binned by location unless FLAG_WF_UNSORTED."""
    walk = bool(flags & NLG) or len(flat.spheres) < 64 or len(flat.lights) > 8
    if not walk:
        return "fused"
    return "unsorted" if flags & UNSORTED else "binned"


def _accel_used(flat, accel):
    n, tree = len(flat.spheres), len(flat.triangles) >= 64
    if accel == "auto":
        if tree and n <= 192:
            return "bvh_mega"
        return "exact" if n <= 16 else "linear" if n <= 192 else "grid" if n >= 256 else "bvh"
    if accel == "grid":
        return "grid" if n >= 256 else "bvh"
    return accel


def _launches(flat, accel, flags, depth):
    used = _accel_used(flat, accel)
    if used in ("exact", "bvh_mega") or (used == "linear" and len(flat.spheres) <= 192):
        return 1
    if used == "linear":
        return wavefront_launches("scan", depth)
    return wavefront_launches(shadow_sequence(flat, flags), depth)


def _render(dev, w, h, depth, accel, flags=0):
    """The frame, and the same frame with FLAG_COUNT_TESTS, which must change no bit, ray count or launch.  Returns
    (frame, stats, counted stats)."""
    f, st = dev.render(w, h, depth, fmt="f64", accel=accel, flags=flags)
    fc, stc = dev.render(w, h, depth, fmt="f64", accel=accel, flags=flags | _lib.FLAG_COUNT_TESTS)
    assert np.array_equal(_bits(f), _bits(fc)), (accel, flags)
    for k in ("rays", "accel_used", "gpu_launches"):
        assert st[k] == stc[k], (accel, flags, k, st[k], stc[k])
    return f, st, stc


def _check_frame(dev, flat, ref, depth, accel, flags=0, w=W, h=H):
    """One render against a reference (frame, rays), with the accel and the launch sequence it must have taken."""
    f, st, stc = _render(dev, w, h, depth, accel, flags)
    what = (accel, flags, depth)
    if ref[2] == "oracle":
        _assert_oracle(f, st, ref[0], ref[1], what)
    else:
        assert np.array_equal(_bits(f), _bits(ref[0])) and st["rays"] == ref[1], what
    assert st["accel_used"] == _accel_used(flat, accel), (what, st["accel_used"])
    assert st["gpu_launches"] == _launches(flat, accel, flags, depth), (what, st["gpu_launches"])
    return f, st, stc


def _oracle_ref(flat, depth, w=W, h=H):
    ref, rays, _ = oracle_frame(flat, w, h, depth)
    return ref, rays, "oracle"


def _exact_ref(dev, depth, w=W, h=H):
    f, st = dev.render(w, h, depth, fmt="f64", accel="exact")
    return f, st["rays"], "exact"


def _changed(a, b, tol=1e-6):
    """Share of pixels whose colour differs between two frames."""
    return float((np.abs(a - b).max(axis=2) > tol).mean())


def _renumber(flat):
    """Contiguous `order` values 0, 1, ... in the list order the tables already give."""
    tabs = (flat.lights, flat.spheres, flat.triangles, flat.planes)
    orders = np.concatenate([t['order'] for t in tabs]).astype(np.int64)
    rank = np.empty(len(orders), np.int32)
    rank[np.argsort(orders, kind='stable')] = np.arange(len(orders), dtype=np.int32)
    at = 0
    for t in tabs:
        t['order'] = rank[at:at + len(t)]
        at += len(t)
    return flat


def _list_orders(flat):
    """Orders in table order: lights, spheres, triangles, plane."""
    tabs = (flat.lights, flat.spheres, flat.triangles, flat.planes)
    at = 0
    for t in tabs:
        t['order'] = np.arange(at, at + len(t))
        at += len(t)
    return flat


def _light_locs(n):
    k = np.arange(n)
    a = 2.0 * np.pi * k / max(n, 1)
    locs = np.stack([50 * np.cos(a), -36.0 - 2 * k, 45 + 50 * np.sin(a)], 1)
    locs[:min(n, 3)] = M3_LIGHTS[:min(n, 3)]
    return locs


@functools.lru_cache(maxsize=None)
def _m3():
    return sc.mesh_scene("m3")


def _with(flat, lights=None, spheres=None, triangles=None, planes=None):
    pick = lambda new, old: (old if new is None else new).copy()
    return sc.FlatScene(flat.camera, pick(lights, flat.lights), pick(spheres, flat.spheres),
                        pick(triangles, flat.triangles), pick(planes, flat.planes))


def mesh_case(n_spheres, n_lights=3, n_triangles=None):
    """m3's sheet cells under the near part of the view (centroid z < 22), its two nearest icospheres (their own
    colours) and the first n_spheres C3 spheres of m3, lit by n_lights lights of different colours (the first three
    at m3's positions); orders contiguous: lights, spheres, triangles, plane.  n_triangles keeps that many sheet
    triangles nearest the middle of the view instead (either side of the tree), in table order."""
    m3 = _m3()
    t = m3.triangles
    sheet = t[:SHEET]
    c = (sheet['v1'] + sheet['v2'] + sheet['v3']) / 3.0
    keep = (c[:, 2] < 22.0) & (np.abs(c[:, 0]) < c[:, 2] + 3.0)
    if n_triangles is None:
        icos = [t[SHEET + 1280 * k:SHEET + 1280 * (k + 1)] for k in (7, 1)]     # centres at z = 19.9 and 36.9
        tris = np.concatenate([sheet[keep]] + icos)
    else:
        cand = np.nonzero(keep)[0]
        near = np.argsort(np.linalg.norm(c[cand] - (0.0, 4.5, 11.0), axis=1), kind='stable')[:n_triangles]
        tris = sheet[np.sort(cand[near])]
    flat = sc.FlatScene(m3.camera, _first_lights(n_lights), m3.spheres[:n_spheres].copy(), tris.copy(),
                        m3.planes.copy())
    return _renumber(flat)


def _first_lights(n):
    """_lights at _light_locs, listed before everything else (orders below m3's, for _renumber)."""
    lights = _lights(_light_locs(n))
    lights['order'] -= n
    return lights


def m3_case(n_lights=3):
    return _renumber(_with(_m3(), lights=_first_lights(n_lights)))


# ---- 1. few-sphere mesh scenes across every threshold ------------------------------------------------------------

N_SPHERES = (0, 1, 16, 17, 63, 64, 192, 193)


@functools.lru_cache(maxsize=None)
def _mesh_ref(n, depth):
    return _oracle_ref(mesh_case(n), depth)


@pytest.mark.parametrize("n", N_SPHERES)
def test_few_sphere_mesh_scenes(gpu, n):
    """auto takes the megakernel with the triangle walk up to 192 spheres, linear the tiled kernel up to 192 and
    the wavefront's scan from 193; grid is bvh below 256 spheres, and the direction grids start at 64."""
    flat = mesh_case(n)
    assert len(flat.triangles) <= 4000
    ref1 = _mesh_ref(n, 1)
    bare, _, _ = oracle_frame(_with(flat, triangles=flat.triangles[:0]), W, H, 1)
    assert _changed(ref1[0], bare) >= 0.2                 # the triangles are a real share of the frame
    dev = flat.upload(0)
    try:
        for depth in (1, 5):
            ref = _mesh_ref(n, depth)
            for accel in RENDER_ACCELS:
                _check_frame(dev, flat, ref, depth, accel)
    finally:
        dev.close()


@pytest.mark.parametrize("n_spheres", [0, 16])
@pytest.mark.parametrize("n_tris", [63, 64])
def test_either_side_of_the_triangle_tree(gpu, n_spheres, n_tris):
    flat = mesh_case(n_spheres, n_triangles=n_tris)
    assert len(flat.triangles) == n_tris
    dev = flat.upload(0)
    try:
        for depth in (1, 5):
            ref = _oracle_ref(flat, depth)
            if depth == 1:
                bare, _, _ = oracle_frame(_with(flat, triangles=flat.triangles[:0]), W, H, 1)
                assert _changed(ref[0], bare) >= 0.05
            for accel in RENDER_ACCELS:
                _check_frame(dev, flat, ref, depth, accel)
    finally:
        dev.close()


# ---- 2. every shadow sequence with triangles --------------------------------------------------------------------

SEQ_SCENES = {
    "n17": lambda: mesh_case(17),
    "n63": lambda: mesh_case(63),
    "n64": lambda: mesh_case(64),
    "m3": lambda: m3_case(),
    "m3_9_lights": lambda: m3_case(9),        # lights 0-7 have direction grids, light 8 walks
}


@pytest.mark.parametrize("name", list(SEQ_SCENES))
def test_every_shadow_sequence_with_triangles(gpu, name):
    flat = SEQ_SCENES[name]()
    depth = 5
    dev = flat.upload(0)
    try:
        ref = _mesh_ref(int(name[1:]), depth) if name.startswith("n") else _exact_ref(dev, depth)
        seen = set()
        for accel in ("bvh", "grid"):
            for flags in SHADOW_FLAGS:
                _check_frame(dev, flat, ref, depth, accel, flags)
                seen.add(shadow_sequence(flat, flags))
        want = {"binned", "unsorted"} | ({"fused"} if len(flat.spheres) >= 64 and len(flat.lights) <= 8 else set())
        assert seen == want, seen
    finally:
        dev.close()


# ---- 3. the reference's triangle quirks in whole frames ---------------------------------------------------------

def _ico(level, centre, radius, colour, refl=0.3, inward=False):
    v, f = sc._icosphere(level)
    if inward:
        f = f[:, [0, 2, 1]]
    v = sc._f32(v * radius + np.asarray(centre, dtype=np.float64))
    return sc.mesh_triangles(v, f, (tuple(colour), 20.0, 0.5, refl), 0)


def quirk_base(n_spheres):
    """C3's camera and floor, three lights of different colours at m3's positions, the first n_spheres of m3's
    spheres (n_spheres = 3000: all of them) and a closed icosphere of 320 triangles in view, so that the scene has a
    triangle tree without the quirk's mesh."""
    m3 = _m3()
    front = _ico(2, (3.0, -1.0, 13.0), 3.0, (0.2, 0.7, 0.9), refl=0.4)
    return sc.FlatScene(m3.camera, _lights(M3_LIGHTS), m3.spheres[:n_spheres].copy(), front, m3.planes.copy())


def _quirk_mesh(kind):
    if kind == "behind_camera":             # primary rays meet its far side at negative Distance, and that wins
        return _ico(2, (0.5, 0.3, -9.0), 2.5, (0.95, 0.3, 0.1))
    if kind == "around_camera":             # every primary ray meets the face behind the camera
        return _ico(1, (0.3, -0.2, -1.5), 4.0, (0.6, 0.9, 0.2), refl=0.5)
    if kind == "around_light":              # light 0's shadow rays meet the face behind the light
        return _ico(1, M3_LIGHTS[0] + (0.2, 0.1, 0.1), 1.5, (0.9, 0.1, 0.8))
    if kind == "behind_light":              # light 1's shadow rays are blocked at negative Distance
        d = np.array([0.0, 0.0, 30.0]) - M3_LIGHTS[1]
        return _ico(2, M3_LIGHTS[1] - 25.0 * d / np.linalg.norm(d), 12.0, (0.3, 0.3, 0.95))
    raise KeyError(kind)


def duplicates_scene(n_spheres, with_quirk=True):
    """mesh_with_duplicates(200) (coincident sheet triangles, two copies listed before their originals) with its
    spheres cut to n_spheres; without the quirk, m3's first 200 triangles."""
    flat = mesh_with_duplicates(200) if with_quirk else sc.mesh_scene("m3", n_triangles=200)
    return _renumber(sc.FlatScene(flat.camera, _lights(M3_LIGHTS), flat.spheres[:n_spheres].copy(), flat.triangles,
                                  flat.planes))


def _coincident_rays(flat):
    """Rays from above at the centroids of coincident triangles, and the list position that must win each."""
    t = flat.triangles
    key = np.concatenate([t['v1'], t['v2'], t['v3']], 1)
    _, inv, cnt = np.unique(key, axis=0, return_inverse=True, return_counts=True)
    tied = np.nonzero(cnt[inv.reshape(-1)] > 1)[0]
    c = (t['v1'][tied] + t['v2'][tied] + t['v3'][tied]) / 3.0
    d = np.tile([0.0, 0.6, 0.8], (len(tied), 1))
    win = [int(t['order'][inv.reshape(-1) == inv.reshape(-1)[i]].min()) for i in tied]
    return np.concatenate([c - 5.0 * d, d], 1), np.array(win)


def quirk_scene(kind, n_spheres, with_quirk=True):
    if kind == "duplicates":
        return duplicates_scene(n_spheres, with_quirk)
    flat = quirk_base(n_spheres)
    if with_quirk:
        flat.triangles = np.concatenate([flat.triangles, _quirk_mesh(kind)])
    return _list_orders(flat)


QUIRKS = ("behind_camera", "around_camera", "around_light", "behind_light", "duplicates")


@pytest.mark.parametrize("n_spheres", [0, 17, 3000])
@pytest.mark.parametrize("kind", QUIRKS)
def test_the_quirks_in_whole_frames(gpu, kind, n_spheres):
    if kind == "duplicates" and n_spheres == 17:
        n_spheres = 16
    depth = 4
    flat = quirk_scene(kind, n_spheres)
    ref = _oracle_ref(flat, depth)
    without, _, _ = oracle_frame(quirk_scene(kind, n_spheres, with_quirk=False), W, H, depth)
    dev = flat.upload(0)
    try:
        if kind == "duplicates":
            # the sheet's shading normal (v1 x v2, erl:448-451) faces away from every light that can reach its front,
            # so which copy wins never shows in a colour: the ties are checked on the hits
            rays, win = _coincident_rays(flat)
            oe, _ = _assert_batches(dev, flat, rays, min_hits=0.99)
            assert np.array_equal(oe, win) and len(set(win)) == 4
            assert np.array_equal(_bits(ref[0]), _bits(without))
        else:
            assert _changed(ref[0], without) > 0.01, kind            # the quirk decides colours
        for accel in RENDER_ACCELS:
            _check_frame(dev, flat, ref, depth, accel)
        for accel in ("bvh", "grid"):
            for flags in SHADOW_FLAGS[1:]:
                _check_frame(dev, flat, ref, depth, accel, flags)
    finally:
        dev.close()


# ---- 4. the always-list and the fallback scan -------------------------------------------------------------------

def _tri(v1, v2, v3, colour, refl=0.2):
    return sc.mesh_triangles(np.array([v1, v2, v3], dtype=np.float64), np.array([[0, 1, 2]]),
                             (tuple(colour), 4.0, 0.4, refl), 0)


def always_scene(n_spheres):
    """quirk_base plus a backdrop of two triangles 2000 wide at z = 60 (edges far beyond 64 times the median) and a
    band x in [-4, 4] at z = 25 whose apex lies at y = -2e30: three triangles on the always-list."""
    flat = quirk_base(n_spheres)
    extra = [_tri((-1000.0, -1000.0, 60.0), (-1000.0, 1000.0, 60.0), (1000.0, -1000.0, 60.0), (0.8, 0.75, 0.3)),
             _tri((1000.0, 1000.0, 60.0), (1000.0, -1000.0, 60.0), (-1000.0, 1000.0, 60.0), (0.3, 0.8, 0.5)),
             _tri((-4.0, -3.0, 25.0), (0.0, -2e30, 25.0), (4.0, -3.0, 25.0), (0.9, 0.2, 0.4), refl=0.5)]
    flat.triangles = np.concatenate([flat.triangles[:100]] + extra + [flat.triangles[100:]])
    return _list_orders(flat)


def _n_always(L, tris):
    t = np.ascontiguousarray(np.concatenate([tris['v1'], tris['v2'], tris['v3']], 1))
    h = L.tb_build(t.ctypes.data, len(t))
    n = L.tb_n_always(h)
    L.tb_free(h)
    return n


def _assert_batches(dev, flat, rays, min_hits=0.3):
    """exact against the oracle's nearest_batch, every other accel against exact: (order, Distance bits)."""
    oe, te = dev.trace_rays(rays, accel="exact")
    _, kind, f = oracle_scene_from_flat(flat)
    oi, ot = orc.nearest_batch(rays, kind, f)
    assert np.array_equal(oi, oe) and np.array_equal(_bits(ot), _bits(te))
    assert (oe >= 0).mean() > min_hits, (oe >= 0).mean()
    for accel in TRACE_ACCELS:
        o, t = dev.trace_rays(rays, accel=accel)
        bad = np.flatnonzero((o != oe) | (_bits(t) != _bits(te)))
        assert bad.size == 0, (accel, bad.size, rays[bad[:3]], o[bad[:3]], oe[bad[:3]])
    return oe, te


@pytest.mark.parametrize("n_spheres", [0, 17, 3000])
def test_the_always_list(gpu, tb, n_spheres):
    flat = always_scene(n_spheres)
    assert _n_always(tb, flat.triangles) == 3 and _n_always(tb, quirk_base(0).triangles) == 0
    depth = 4
    ref = _oracle_ref(flat, depth)
    dev = flat.upload(0)
    try:
        for accel in RENDER_ACCELS:
            _check_frame(dev, flat, ref, depth, accel)
        for accel in ("bvh", "grid"):
            for flags in SHADOW_FLAGS[1:]:
                _check_frame(dev, flat, ref, depth, accel, flags)
        oe, _ = _assert_batches(dev, flat, _edge_rays(flat, 30000, 17))
        always = flat.triangles['order'][100:103]
        assert all(np.count_nonzero(oe == o) > 10 for o in always)
    finally:
        dev.close()


FALLBACK_CELL = 3.0e4


def fallback_scene(n_spheres):
    """A tree of 136 triangles whose edges are all 3e4 and more: the floor y = 3 in 8 x 8 cells of 3e4 (every
    triangle its own colour) and an awning of 8 triangles at y = -8 over x, z in [0, 6e4] that faces the lights and
    shadows part of the floor.  tri_ray_setup refuses every ray of unit length there (e_det > 0.5e-6), so every
    kernel's triangles go through the fallback loop of scan_tris_bvh."""
    rng = np.random.default_rng(77)
    m3 = _m3()
    xs = np.arange(-4, 5) * FALLBACK_CELL
    X, Z = np.meshgrid(xs, xs, indexing='ij')
    floor_v = np.stack([X, np.full_like(X, 3.0), Z], -1).reshape(-1, 3)
    aw = np.arange(0, 3) * FALLBACK_CELL
    X, Z = np.meshgrid(aw, aw, indexing='ij')
    awning_v = np.stack([X, np.full_like(X, -8.0), Z], -1).reshape(-1, 3)

    def quads(v, n):
        idx = np.arange((n + 1) * (n + 1)).reshape(n + 1, n + 1)
        p00, p10, p01, p11 = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, 1:].ravel()
        f = np.stack([np.stack([p00, p10, p01], 1), np.stack([p10, p11, p01], 1)], 1).reshape(-1, 3)
        nrm = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
        f[nrm[:, 1] > 0] = f[nrm[:, 1] > 0][:, [0, 2, 1]]          # facing up (-y), towards the lights
        return f

    tabs = []
    for v, n in ((floor_v, 8), (awning_v, 2)):
        for face in quads(v, n):
            tabs.append(sc.mesh_triangles(v, face[None], (tuple(rng.uniform(0.1, 1.0, 3)), 4.0, 0.3, 0.25), 0))
    flat = sc.FlatScene(m3.camera, _lights(M3_LIGHTS), m3.spheres[:n_spheres].copy(), np.concatenate(tabs),
                        m3.planes.copy())
    return _list_orders(flat)


def _tree_edge_max(tris):
    e = [np.linalg.norm(tris[b] - tris[a], axis=1) for a, b in (('v1', 'v2'), ('v1', 'v3'), ('v2', 'v3'))]
    return float(np.max(e))


def _e_det_unit(edge_max):
    """tri_walk.h's bound on det's rounding error for a ray of unit length (|D|_inf >= 1/sqrt(3))."""
    return 16.0 * 2.0 ** -53 * 1.7321 / np.sqrt(3.0) * edge_max ** 2


@pytest.mark.parametrize("n_spheres", [0, 17, 64])
def test_the_fallback_scan_in_frames(gpu, tb, n_spheres):
    flat = fallback_scene(n_spheres)
    assert _n_always(tb, flat.triangles) == 0
    assert _e_det_unit(_tree_edge_max(flat.triangles)) > 0.5e-6 > _e_det_unit(1e4)
    depth = 4
    ref = _oracle_ref(flat, depth)
    no_awning, _, _ = oracle_frame(_with(flat, triangles=flat.triangles[:128]), W, H, depth)
    assert _changed(ref[0], no_awning) > 0.05                    # the awning's shadow is in the frame
    dev = flat.upload(0)
    try:
        counted = {}
        for accel in RENDER_ACCELS:
            _, _, stc = _check_frame(dev, flat, ref, depth, accel)
            counted[accel] = stc["exact_other_tests"]
        for accel in ("bvh", "grid"):
            for flags in SHADOW_FLAGS[1:]:
                _check_frame(dev, flat, ref, depth, accel, flags)
        # no ray pruned: the megakernel and the tiled kernel test every triangle and plane, as the linear scan does;
        # the wavefront's shadow walks stop at the first improvement
        assert counted["bvh_mega"] == counted["linear"] == counted["exact"], counted
        assert 0 < counted["bvh"] <= counted["exact"], counted
    finally:
        dev.close()


def _refused_rays(flat, rng, n):
    """Rays tri_ray_setup refuses, aimed at points of the mesh: a denormal direction component, |D|_inf > 1e30,
    and axis-parallel rays from 2e30 away (in front of the mesh and behind it)."""
    t = flat.triangles
    k = rng.integers(0, len(t), n)
    w = rng.dirichlet((2.0, 2.0, 2.0), n)
    P = w[:, :1] * t['v1'][k] + w[:, 1:2] * t['v2'][k] + w[:, 2:] * t['v3'][k]
    O = np.stack([rng.uniform(-15, 15, n), rng.uniform(-15, 0, n), rng.uniform(-8, 2, n)], 1)
    D = P - O
    D /= np.linalg.norm(D, axis=1, keepdims=True)
    denorm = D.copy()
    j = np.argmin(np.abs(D), axis=1)
    denorm[np.arange(n), j] = np.where(D[np.arange(n), j] < 0, -1.0, 1.0) * 4e-320
    axis = np.zeros((n, 3))
    axis[np.arange(n), rng.integers(0, 3, n)] = rng.choice([-1.0, 1.0], n)
    far = P - axis * 2e30 * rng.choice([-1.0, 1.0], n)[:, None]
    return {"denormal": np.concatenate([O, denorm], 1), "huge_direction": np.concatenate([O, D * 3e31], 1),
            "huge_origin": np.concatenate([far, axis], 1)}


@pytest.mark.parametrize("n_spheres", [0, 16, 3000])
def test_rays_the_walk_refuses_equal_exact(gpu, n_spheres):
    flat = mesh_case(n_spheres)
    dev = flat.upload(0)
    try:
        for name, rays in _refused_rays(flat, np.random.default_rng(n_spheres), 4000).items():
            _assert_batches(dev, flat, rays, min_hits=0.2)
    finally:
        dev.close()


# ---- 5. updates -------------------------------------------------------------------------------------------------

def _moved_mesh_case(flat):
    out = _with(flat)
    ico = slice(len(out.triangles) - 2560, None)
    for v in ('v1', 'v2', 'v3'):
        out.triangles[v][ico] = sc._f32(out.triangles[v][ico] + (0.75, -0.5, 1.25))
        out.triangles[v][:ico.start, 1] = sc._f32(out.triangles[v][:ico.start, 1] - 0.125)
    out.lights['location'][0] += (2.0, 1.5, -1.0)
    if len(out.spheres):
        out.spheres['center'] = sc._f32(out.spheres['center'] + (-0.5, 0.25, 0.75))
    return out


@pytest.mark.parametrize("n_spheres", [0, 16])
def test_updated_mesh_scenes_equal_a_fresh_create(gpu, n_spheres):
    flat = mesh_case(n_spheres)
    dev = flat.upload(0)
    try:
        moved = _moved_mesh_case(flat)
        info = moved.update(dev, rebuild_grids=True)
        assert "refit_triangles" in info["done"] and "light_pos" in info["changed"], info
        assert ("spheres" in info["changed"]) == (n_spheres > 0), info
        _assert_like_fresh(dev, moved)
        ref = _oracle_ref(moved, 4)
        assert _changed(ref[0], oracle_frame(flat, W, H, 4)[0]) > 0.05
        for accel in ("auto", "bvh"):
            _check_frame(dev, moved, ref, 4, accel)
    finally:
        dev.close()


@pytest.mark.parametrize("n_spheres", [0, 16])
def test_a_grown_tree_triangle_engages_the_fallback(gpu, tb, n_spheres):
    """An update that stretches one tree triangle to edges of 5e4 refits it into the tree (its coordinates stay
    below 1e30) and raises the tree's edge bound: every ray then takes the fallback scan.  A fresh create of the
    same tables puts the triangle on the always-list and walks the tree; the frames must agree bit for bit."""
    flat = mesh_case(n_spheres)
    grown = _with(flat)
    c = (grown.triangles['v1'] + grown.triangles['v2'] + grown.triangles['v3']) / 3.0
    i = int(np.argmin(np.linalg.norm(c - (4.0, 4.5, 12.0), axis=1)))
    grown.triangles['v3'][i] = grown.triangles['v3'][i] + (0.0, -3.0e4, 4.0e4)
    assert _n_always(tb, flat.triangles) == 0 and _n_always(tb, grown.triangles) == 1
    assert _e_det_unit(_tree_edge_max(grown.triangles)) > 0.5e-6
    depth = 4
    dev = flat.upload(0)
    try:
        info = grown.update(dev)
        assert "refit_triangles" in info["done"] and "rebuild_tri_bvh" not in info["done"], info
        _assert_like_fresh(dev, grown)
        ref = _oracle_ref(grown, depth)
        assert _changed(ref[0], oracle_frame(flat, W, H, depth)[0]) > 0.01
        counted = {}
        for accel in RENDER_ACCELS:
            _, _, stc = _check_frame(dev, grown, ref, depth, accel)
            counted[accel] = stc["exact_other_tests"]
        assert counted["bvh_mega"] == counted["linear"] == counted["exact"], counted
        fresh = grown.upload(0)
        _, _, walked = _render(fresh, W, H, depth, "bvh_mega")
        fresh.close()
        assert walked["exact_other_tests"] < counted["exact"] // 4, (walked["exact_other_tests"], counted)
    finally:
        dev.close()
