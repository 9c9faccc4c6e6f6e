"""The kernels at the limits of their fixed-size structures, held to the FP64 reference.

1. wf_shadow_shade (shadow rays and the light fold in one kernel) at 6, 7 and 8 lights: a pair list entry is
   `slot << 3 | light`, and only 5-8 lights use all three light bits; a sparse scene fills the whole pair list.
   9 lights take the unfused sequence.
2. wf_scan (ERT_ACCEL_LINEAR frames past 192 spheres) at its tile (512), group (16) and batch (512 rays) edges, with
   exact Distance ties between spheres of different tiles, ties with the planes and triangles wf_scan_init seeds,
   and floods of candidates.
3. Triangle and plane tables that are not in list order: their `order` values decide every tie.
4. A cell holding exactly kCellGridMaxCount (127) spheres, one more, and direction cells of 512 and 513 entries,
   where the device builder switches from a warp rank to a block radix sort.
5. The f32 and rgb8 output formats through the wavefront.

The references: oracle_frame (the C restatement, FP64) with assert_double_parity and equal ray counts for frames,
accel="exact" (the per-pixel FP64 linear scan) bit for bit between GPU strategies, and trace_rays(accel="exact")
for ray batches.  Colours differ per object and per light, so that a wrong winner or a dropped or swapped light
changes the colour, not just a rounding.  The construction checks of section 4 run on the CPU."""
import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import assert_double_parity, oracle_frame, oracle_scene_from_flat, quantise
from oracle import orc
from test_grid_build_host import CAND_DT, gh, host_cell, host_light, sphere_table  # noqa: F401 (gh: fixture)
from test_gpu_grid_build import _assert_like_fresh, gd, device_cell, device_light  # noqa: F401 (gd: fixture)

RENDER_ACCELS = ("exact", "linear", "bvh", "bvh_mega", "grid", "auto")
CELL_DT = np.dtype([("f", "<f4", (6, 4)), ("sph", "<i4", 6), ("cnt", "<u4"), ("more", "<u4")])   # CellBlock


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def _assert_oracle(frame, st, ref, ref_rays, what):
    assert_double_parity(frame, ref)
    assert np.array_equal(quantise(frame), quantise(ref)), what
    assert st["rays"] == ref_rays, (what, st["rays"], ref_rays)


def _lattice(w, h, nx=12, ny=8):
    xs = np.unique(np.linspace(0, w - 1, min(w, nx)).astype(np.int32))
    ys = np.unique(np.linspace(0, h - 1, min(h, ny)).astype(np.int32))
    gx, gy = np.meshgrid(xs, ys)
    return gx.reshape(-1), gy.reshape(-1)


def _assert_oracle_lattice(flat, frame, w, h, depth, extra=()):
    xs, ys = _lattice(w, h)
    if len(extra):
        xs = np.concatenate([xs, np.asarray([p[0] for p in extra], np.int32)])
        ys = np.concatenate([ys, np.asarray([p[1] for p in extra], np.int32)])
    ref, _, _ = oracle_frame(flat, w, h, depth, pixels=(xs, ys))
    got = frame[ys, xs]
    assert_double_parity(got, ref)
    assert np.array_equal(quantise(got), quantise(ref))


def _lights(locs):
    """A light table whose diffuse and specular colours differ per light."""
    k = np.arange(len(locs), dtype=np.float64)
    t = np.zeros(len(locs), dtype=_lib.LIGHT_DT)
    t['location'] = locs
    t['diffuse_colour'] = np.stack([0.15 + 0.1 * k, 0.9 - 0.08 * k, 0.2 + 0.3 * (k % 3)], 1)
    t['specular_colour'] = np.stack([0.3 + 0.07 * k, 0.25 + 0.15 * (k % 4), 0.95 - 0.1 * k], 1)
    t['order'] = np.arange(len(locs))
    return t


def _interleave(flat, rng):
    """New `order` values: one random permutation over every element, so lights, spheres, triangles and planes
    alternate in the list."""
    tabs = (flat.lights, flat.spheres, flat.triangles, flat.planes)
    perm = rng.permutation(sum(len(t) for t in tabs)).astype(np.int32)
    at = 0
    for t in tabs:
        t['order'] = perm[at:at + len(t)]
        at += len(t)
    return flat


def _by_order(t, reverse=False):
    idx = np.argsort(t['order'], kind='stable')
    return t[idx[::-1] if reverse else idx].copy()


# ---- 1. the fused shadow stage at eight lights ------------------------------------------------------------------

def shadow_scene(n_lights, sparse=False):
    """C3's recipe with n_lights lights around and above the cloud.  The list interleaves lights with spheres and
    the plane, the light table goes to create in reversed list order, and lights 0 and 1 share a position (with
    different colours).  sparse: 320 small spheres spread thin just above the floor under the lights, so nearly
    every (hit, light) pair stays open after the triage and a chunk of 128 hits fills the 1024-entry pair list."""
    k = np.arange(n_lights)
    a = 2.0 * np.pi * k / n_lights
    if sparse:
        rng = np.random.default_rng(71)
        flat = sc.synthetic_scene("c3", n_spheres=320, seed=71)
        flat.spheres['center'] = _f32(np.stack([rng.uniform(-22, 22, 320), rng.uniform(3.2, 4.6, 320),
                                                rng.uniform(6, 40, 320)], 1))
        flat.spheres['radius'] = _f32(rng.uniform(0.15, 0.35, 320))
        locs = np.stack([14 * np.cos(a), -22.0 - 2 * k, 22 + 14 * np.sin(a)], 1)
    else:
        flat = sc.synthetic_scene("c3", n_spheres=2000)
        locs = np.stack([50 * np.cos(a), -36.0 - 2 * k, 45 + 50 * np.sin(a)], 1)
    locs[1] = locs[0]
    flat.lights = _lights(locs)
    flat = _interleave(flat, np.random.default_rng(1000 + n_lights))
    flat.lights = _by_order(flat.lights, reverse=True)
    return flat


def _one_light(flat):
    lights = _by_order(flat.lights)[:1]
    return sc.FlatScene(flat.camera, lights, flat.spheres, flat.triangles, flat.planes)


def _check_shadow_scene(flat, n_lights, w=64, h=36, depth=4):
    dev = flat.upload(0)
    one = _one_light(flat).upload(0)
    try:
        ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
        assert ref.any()
        for accel in ("grid", "bvh", "auto"):
            frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            _assert_oracle(frame, st, ref, ref_rays, accel)
            walk, sw = dev.render(w, h, depth, fmt="f64", accel=accel, flags=_lib.FLAG_NO_LIGHT_GRID)
            assert np.array_equal(_bits(walk), _bits(frame)) and sw["rays"] == st["rays"], accel
            # L <= 8 lights with a direction grid each: shadow rays and the fold in one kernel, so the frame takes as
            # many launches as with one light; a ninth light has no grid and brings the binned, unfused sequence
            _, s1 = one.render(w, h, depth, fmt="f64", accel=accel)
            if n_lights <= 8:
                assert st["gpu_launches"] == s1["gpu_launches"], (accel, st["gpu_launches"], s1["gpu_launches"])
            else:
                assert st["gpu_launches"] > s1["gpu_launches"], (accel, st["gpu_launches"], s1["gpu_launches"])
        for accel in ("linear", "exact"):
            frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            _assert_oracle(frame, st, ref, ref_rays, accel)
    finally:
        one.close()
        dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_lights", [6, 7, 8, 9])
def test_many_lights_match_the_oracle(gpu, n_lights):
    _check_shadow_scene(shadow_scene(n_lights), n_lights)


@pytest.mark.gpu
@pytest.mark.parametrize("n_lights", [6, 8])
def test_full_pair_list_of_a_sparse_scene(gpu, n_lights):
    _check_shadow_scene(shadow_scene(n_lights, sparse=True), n_lights, w=64, h=48)


# ---- 2. the brute-force scan at its tile, group and batch edges, with ties and floods ---------------------------

def scan_scene(n, seed):
    """n spheres of C3's materials packed in front of the camera, the floor and C3's three lights."""
    rng = np.random.default_rng(seed)
    flat = sc.synthetic_scene("c3", n_spheres=n, seed=seed)
    flat.spheres['center'] = _f32(np.stack([rng.uniform(-14, 14, n), rng.uniform(-9, 4, n), rng.uniform(4, 34, n)], 1))
    flat.spheres['radius'] = _f32(rng.uniform(0.3, 1.3, n))
    return flat


def _check_linear(flat, sizes, depth=4, extra=()):
    """Every frame through wf_scan: bit-equal to the exact scan with equal ray counts, and the oracle's on a
    lattice of pixels."""
    dev = flat.upload(0)
    try:
        for w, h in sizes:
            lin, sl = dev.render(w, h, depth, fmt="f64", accel="linear")
            ex, se = dev.render(w, h, depth, fmt="f64", accel="exact")
            assert sl["accel_used"] == "linear" and sl["gpu_launches"] > 1, (w, h)       # the wavefront's scan
            assert np.array_equal(_bits(lin), _bits(ex)), (w, h)
            assert sl["rays"] == se["rays"], (w, h)
            _assert_oracle_lattice(flat, lin, w, h, depth, [p for p in extra if p[0] < w and p[1] < h])
        return lin
    finally:
        dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [193, 208, 511, 512, 513, 1024, 1025, 1535])
def test_scan_tile_group_and_batch_edges(gpu, n):
    _check_linear(scan_scene(n, 300 + n), ((1, 1), (16, 32), (17, 31), (96, 54)))


TIE_COPIES = (1, 2, 17, 511, 512, 1024)        # list positions in different tiles, groups and pair halves


def tie_scene(park=()):
    """1100 spheres; those at TIE_COPIES are one big sphere in front of the others (same centre and radius, different
    colours), so every ray that meets it meets all six at the same Distance.  park: copies moved out of sight."""
    flat = scan_scene(1100, 17)
    s = flat.spheres
    assert np.array_equal(s['order'], np.arange(3, 1103))
    for k, i in enumerate(TIE_COPIES):
        s['center'][i] = (0.5, -0.5, 3.0) if i not in park else (0.0, 1.0e4, 0.0)
        s['radius'][i] = 2.5
        s['material']['colour'][i] = (k / 6.0, 1.0 - k / 6.0, 0.25 + 0.1 * k)
        s['material']['reflectivity'][i] = 0.3
    return flat


@pytest.mark.gpu
def test_scan_ties_across_tiles_go_to_the_earliest_copy(gpu):
    """The CAS fold of scan_resolve must order equal Distances by list position whichever block's candidate
    arrives first.  The earliest copy wins every path ray: parking the later copies changes no bit.  Shadow rays
    to it meet the five later copies at the same Distance and must stay lit (the oracle checks the colours)."""
    sizes = ((16, 32), (96, 54))
    lin = _check_linear(tie_scene(), sizes)
    later = [i for i in TIE_COPIES if i != TIE_COPIES[0]]
    dev = tie_scene(park=later).upload(0)
    alone, _ = dev.render(96, 54, 4, fmt="f64", accel="linear")
    dev.close()
    assert np.array_equal(_bits(lin), _bits(alone))
    dev = tie_scene(park=TIE_COPIES[:1]).upload(0)
    second, _ = dev.render(96, 54, 4, fmt="f64", accel="linear")
    dev.close()
    assert (np.abs(second - lin).max(axis=2) > 1e-3).sum() > 200        # the copies fill a good part of the frame


def _tri(v1, v2, v3, colour, order, refl=0.3):
    t = np.zeros(1, dtype=_lib.TRIANGLE_DT)
    t['v1'], t['v2'], t['v3'] = v1, v2, v3
    t['material']['colour'] = colour
    t['material']['specular_power'] = 4.0
    t['material']['shininess'] = 0.5
    t['material']['reflectivity'] = refl
    t['order'] = order
    return t


def _plane(normal, dist, colour, order, refl=0.2):
    p = np.zeros(1, dtype=_lib.PLANE_DT)
    p['normal'] = normal
    p['distance'] = dist
    p['material']['colour'] = colour
    p['material']['specular_power'] = 1.0
    p['material']['shininess'] = 0.0
    p['material']['reflectivity'] = refl
    p['order'] = order
    return p


def seeded_tie_scene(sphere_first):
    """The centre pixel of an even-sized frame looks along +z from (0, 0, -2).  A sphere of radius 4 at z = 10, the
    plane z = 6 and a triangle in that plane all meet that ray at exactly t = 8.  wf_scan_init seeds the ray with
    the triangle or the plane; the sphere arrives as a scan candidate and must win (sphere_first) or lose the tie
    by list position.  300 small spheres stand off the axis in front of the plane."""
    rng = np.random.default_rng(44)
    n = 300
    flat = sc.synthetic_scene("c3", n_spheres=n + 1, seed=44)
    c = np.stack([rng.uniform(-5, 5, n), rng.uniform(-3.5, 3.5, n), rng.uniform(1.5, 5.0, n)], 1)
    c[:, 0] = np.where(np.abs(c[:, 0]) < 1.2, c[:, 0] + np.sign(c[:, 0] + 1e-9) * 1.2, c[:, 0])
    flat.spheres['center'] = _f32(np.concatenate([[[0.0, 0.0, 10.0]], c]))
    flat.spheres['radius'] = _f32(np.concatenate([[4.0], rng.uniform(0.1, 0.4, n)]))
    flat.spheres['material']['colour'][0] = (0.9, 0.1, 0.2)
    flat.lights = _lights(np.array([[4.0, -6.0, -1.0], [-5.0, -3.0, 2.0]]))
    # orders: lights 0, 1; then sphere 0, the triangle and the plane in the order asked for; then the rest
    first, tri_o, plane_o = (2, 3, 4) if sphere_first else (4, 2, 3)
    flat.spheres['order'] = np.concatenate([[first], np.arange(5, 5 + n)])
    flat.triangles = _tri((-3.0, 3.0, 6.0), (3.0, 3.0, 6.0), (0.0, -3.0, 6.0), (0.1, 0.8, 0.3), tri_o)
    flat.planes = _plane((0.0, 0.0, -1.0), 6.0, (0.2, 0.3, 0.9), plane_o)
    return flat


@pytest.mark.gpu
@pytest.mark.parametrize("sphere_first", [True, False])
def test_scan_ties_with_the_seeded_plane_and_triangle(gpu, sphere_first):
    flat = seeded_tie_scene(sphere_first)
    cam, kind, f = oracle_scene_from_flat(flat)
    ray = np.array([[0.0, 0.0, -2.0, 0.0, 0.0, 1.0]])
    for o in (int(flat.spheres['order'][0]), int(flat.triangles['order'][0]), int(flat.planes['order'][0])):
        _, t = orc.nearest_batch(ray, kind[[o]], f[[o]])
        assert t[0] == 8.0, o                                  # the three meet the axis at the same Distance
    oi, _ = orc.nearest_batch(ray, kind, f)
    assert oi[0] == min(o for o in (2, 3, 4))
    _check_linear(flat, ((16, 32), (96, 54)), extra=((8, 16), (48, 27)))


def nest_scene():
    """The camera inside 600 concentric spheres: the FP32 filter passes every (ray, sphere) pair, the literal test
    (erl:381) rejects them all.  Lights are inside too; 40 small spheres and the floor are what the rays see."""
    rng = np.random.default_rng(9)
    flat = scan_scene(640, 9)
    s = flat.spheres
    s['center'][:600] = (0.0, 0.0, -2.0)
    s['radius'][:600] = 60.0 + 0.25 * np.arange(600)
    s['material']['colour'][:600] = rng.uniform(0, 1, (600, 3))
    flat.lights['location'] = [(3.0, -4.0, -1.0), (-4.0, 2.0, 0.0), (0.0, -8.0, 10.0)]
    return flat


def crowd_scene():
    """600 big overlapping spheres ahead, each met by every primary ray: hundreds of candidates per ray, concurrent
    swaps on one result slot and many drains per group."""
    rng = np.random.default_rng(10)
    flat = scan_scene(600, 10)
    s = flat.spheres
    s['center'] = _f32(np.array([0.0, 0.0, 300.0]) + rng.uniform(-4, 4, (600, 3)))
    s['radius'] = _f32(250.0 + rng.uniform(-3, 3, 600))
    flat.lights['location'] = [(3.0, -4.0, -1.0), (-4.0, 2.0, 0.0), (1.0, 1.0, -1.5)]
    return flat


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["nest", "crowd"])
def test_scan_candidate_floods(gpu, name):
    flat = nest_scene() if name == "nest" else crowd_scene()
    w, h = 32, 18
    _check_linear(flat, ((w, h),))
    dev = flat.upload(0)
    _, st = dev.render(w, h, 4, fmt="f64", accel="linear", flags=_lib.FLAG_COUNT_TESTS)
    dev.close()
    assert st["exact_sphere_tests"] >= 500 * w * h, st["exact_sphere_tests"]


# ---- 3. triangle and plane tables out of list order -------------------------------------------------------------

def small_tri_scene():
    """300 spheres, 12 triangles and 3 planes, every `order` interleaved.  Two pairs of coincident triangles with
    different materials, a triangle in the floor plane and one in the back wall (exact triangle-plane ties: the
    centre ray meets the wall and its triangle at t = 42)."""
    rng = np.random.default_rng(23)
    n = 300
    flat = sc.synthetic_scene("c3", n_spheres=n, seed=23)
    flat.spheres['center'] = _f32(np.stack([rng.uniform(-12, 12, n), rng.uniform(-8, 4, n), rng.uniform(12, 38, n)], 1))
    flat.spheres['radius'] = _f32(rng.uniform(0.2, 0.8, n))
    tris = []
    for _ in range(6):
        c = np.array([rng.uniform(-6, 6), rng.uniform(-4, 3), rng.uniform(7, 20)])
        v = _f32(c + rng.uniform(-3, 3, (3, 3)))
        if np.cross(v[1] - v[0], v[2] - v[0])[2] > 0:                 # face the camera
            v = v[[0, 2, 1]]
        tris.append(v)
    pairs = [tris[0], tris[1]]
    tris += pairs                                                     # coincident copies
    tris.append(np.array([[-6.0, 5.0, 9.0], [0.0, 5.0, 24.0], [6.0, 5.0, 9.0]]))      # in the floor y = 5
    tris.append(np.array([[-4.0, -3.0, 40.0], [0.0, 4.0, 40.0], [4.0, -3.0, 40.0]]))  # in the wall z = 40
    for v in tris[-2:]:
        if np.cross(v[1] - v[0], v[2] - v[0]) @ np.array([0.0, 0.3, 1.0]) > 0:
            v[[1, 2]] = v[[2, 1]]
    tris.append(_f32(np.array([[-9.0, -6.0, 14.0], [-7.0, 0.0, 14.5], [-5.0, -6.0, 15.0]])))
    tris.append(_f32(np.array([[9.0, -6.0, 14.0], [5.0, -6.0, 15.0], [7.0, 0.0, 14.5]])))
    flat.triangles = np.concatenate([_tri(v[0], v[1], v[2], rng.uniform(0, 1, 3), 0, rng.choice([0.05, 0.3, 0.6]))
                                     for v in tris])
    flat.planes = np.concatenate([_plane((0.0, -1.0, 0.0), 5.0, (1.0, 1.0, 1.0), 0, 0.1),
                                  _plane((0.0, 0.0, -1.0), 40.0, (0.3, 0.6, 0.9), 0, 0.3),
                                  _plane((-1.0, 0.0, -0.2), 18.0, (0.8, 0.4, 0.1), 0, 0.05)])
    flat.lights = _lights(np.array([[5.0, -20.0, 0.0], [-14.0, -10.0, 12.0], [2.0, -3.0, 30.0]]))
    flat = _interleave(flat, rng)
    # the copy listed later gets the earlier list position, so the table order and the list order disagree
    o = flat.triangles['order']
    for a, b in ((0, 6), (1, 7)):
        if o[a] < o[b]:
            o[a], o[b] = o[b], o[a]
    return flat


def mesh_with_duplicates(n_triangles):
    """mesh_scene("m3") cut to n_triangles (a triangle BVH from 64 on) plus four duplicated triangles in other
    colours, two listed before their originals and two after; orders renumbered in that list order."""
    flat = sc.mesh_scene("m3", n_triangles=n_triangles)
    t = _by_order(flat.triangles)
    rng = np.random.default_rng(n_triangles)
    dup = rng.choice(len(t), 4, replace=False)
    rows = []
    for i in range(len(t)):
        if i in dup:
            c = t[i:i + 1].copy()
            c['material']['colour'] = rng.uniform(0, 1, 3)
            rows += [c, t[i:i + 1]] if i in dup[:2] else [t[i:i + 1], c]
        else:
            rows.append(t[i:i + 1])
    t = np.concatenate(rows)
    first = int(flat.triangles['order'].min())
    t['order'] = np.arange(first, first + len(t))
    flat.planes['order'] = first + len(t)
    flat.triangles = t
    return flat


def permuted(flat, seed):
    """The same scene with its triangle and plane tables shuffled; every pair of coincident triangles ends up with
    the later-listed one first in the table."""
    rng = np.random.default_rng(seed)
    tris = flat.triangles[rng.permutation(len(flat.triangles))].copy()
    key = np.concatenate([tris['v1'], tris['v2'], tris['v3']], 1)
    for i in range(len(tris)):
        for j in range(i + 1, len(tris)):
            if np.array_equal(key[i], key[j]) and tris['order'][i] < tris['order'][j]:
                tris[[i, j]] = tris[[j, i]]
                key[[i, j]] = key[[j, i]]
    planes = flat.planes[rng.permutation(len(flat.planes))].copy()
    if len(planes) > 1 and np.all(np.diff(planes['order']) > 0):
        planes = planes[::-1].copy()
    return sc.FlatScene(flat.camera, flat.lights, flat.spheres, tris, planes)


def in_list_order(flat):
    return sc.FlatScene(flat.camera, _by_order(flat.lights), _by_order(flat.spheres), _by_order(flat.triangles),
                        _by_order(flat.planes))


def _tie_rays(flat, rng, n=3000):
    """Rays from random origins in front of the scene: half at random points, half at the centroids of
    coincident triangles and at points of triangles that lie in a plane."""
    t = flat.triangles
    key = np.concatenate([t['v1'], t['v2'], t['v3']], 1)
    _, inv, cnt = np.unique(key, axis=0, return_inverse=True, return_counts=True)
    tied = np.nonzero(cnt[inv.reshape(-1)] > 1)[0].tolist()
    for p in flat.planes:
        s = t['v1'] @ p['normal'] + p['distance'], t['v2'] @ p['normal'] + p['distance'], t['v3'] @ p['normal'] + p['distance']
        tied += np.nonzero((s[0] == 0) & (s[1] == 0) & (s[2] == 0))[0].tolist()
    assert tied
    w = rng.dirichlet((2.0, 2.0, 2.0), n // 2)
    k = rng.choice(tied, n // 2)
    aim = w[:, :1] * t['v1'][k] + w[:, 1:2] * t['v2'][k] + w[:, 2:] * t['v3'][k]
    aim = np.concatenate([aim, np.stack([rng.uniform(-30, 30, n - n // 2), rng.uniform(-20, 5, n - n // 2),
                                         rng.uniform(5, 60, n - n // 2)], 1)])
    o = np.stack([rng.uniform(-15, 15, n), rng.uniform(-15, 0, n), rng.uniform(-8, 2, n)], 1)
    d = aim - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d], 1)


TRI_SCENES = {
    "small": small_tri_scene,
    "m3_64": lambda: mesh_with_duplicates(64),
    "m3_200": lambda: mesh_with_duplicates(200),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRI_SCENES))
def test_permuted_triangle_and_plane_tables(gpu, name):
    flat = permuted(TRI_SCENES[name](), 5)
    ordered = in_list_order(flat)
    assert not np.array_equal(flat.triangles['order'], ordered.triangles['order'])
    w, h, depth = 64, 48, 4
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    dev, dev_o = flat.upload(0), ordered.upload(0)
    try:
        for accel in RENDER_ACCELS:
            frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            _assert_oracle(frame, st, ref, ref_rays, accel)
            same, so = dev_o.render(w, h, depth, fmt="f64", accel=accel)
            assert np.array_equal(_bits(frame), _bits(same)) and so["rays"] == st["rays"], accel
        rays = _tie_rays(flat, np.random.default_rng(8))
        oe, te = dev.trace_rays(rays, accel="exact")
        cam, kind, f = oracle_scene_from_flat(flat)
        oi, ot = orc.nearest_batch(rays, kind, f)
        assert np.array_equal(oi, oe) and np.array_equal(_bits(ot), _bits(te))
        assert (oe >= 0).mean() > 0.4
        for accel in RENDER_ACCELS[1:] + ("warp",):
            for d in (dev, dev_o):
                o, t = d.trace_rays(rays, accel=accel)
                assert np.array_equal(o, oe) and np.array_equal(_bits(t), _bits(te)), accel
    finally:
        dev.close()
        dev_o.close()


def _moved(flat):
    out = sc.FlatScene(flat.camera, flat.lights.copy(), flat.spheres.copy(), flat.triangles.copy(), flat.planes.copy())
    out.spheres['center'] = out.spheres['center'] + (0.25, -0.125, 0.5)
    for v in ('v1', 'v2', 'v3'):
        out.triangles[v] = out.triangles[v] + (-0.375, 0.25, 0.125)
    out.planes['distance'] = out.planes['distance'] + 0.5
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small", "m3_200"])
def test_update_with_permuted_tables(gpu, name):
    flat = TRI_SCENES[name]()
    ordered, shuffled = in_list_order(flat), permuted(flat, 6)
    dev = ordered.upload(0)
    try:
        want = {a: dev.render(64, 36, 3, fmt="f64", accel=a) for a in RENDER_ACCELS}
        info = shuffled.update(dev)
        assert info["changed"] == [], info
        for a in RENDER_ACCELS:
            got, st = dev.render(64, 36, 3, fmt="f64", accel=a)
            assert np.array_equal(_bits(got), _bits(want[a][0])) and st["rays"] == want[a][1]["rays"], a
        moved = permuted(_moved(flat), 7)
        info = moved.update(dev, rebuild_grids=True)
        assert "triangles" in info["changed"] and "planes" in info["changed"], info
        _assert_like_fresh(dev, moved)
    finally:
        dev.close()


# ---- 4. full cell lists and direction cells at the sort switch --------------------------------------------------

def _cell_counts(L, sph):
    enabled, geo, blocks, *_ = host_cell(L, sph, 0.35)
    res = np.frombuffer(geo[:12], np.int32)
    lo = np.frombuffer(geo[12:24], np.float32).astype(np.float64)
    cs = float(np.frombuffer(geo[36:40], np.float32)[0])
    cnt = np.frombuffer(blocks, CELL_DT)['cnt'][::2] if enabled else None
    return enabled, res, lo, cs, cnt


def knot_scene(L, k):
    """C3 with spheres moved into a knot of tiny ones at the centre of a cell the host builder lists as empty, so
    that the cell lists exactly k spheres.  The moved spheres define none of the bounds, so the grid's geometry
    stays C3's.  Returns (flat, cell, knot centre)."""
    flat = sc.synthetic_scene("c3")
    sph = sphere_table(flat)
    enabled, res, lo, cs, cnt = _cell_counts(L, sph)
    assert enabled
    ids = np.arange(len(cnt))
    centres = lo + (np.stack([ids % res[0], ids // res[0] % res[1], ids // (res[0] * res[1])], 1) + 0.5) * cs
    r = np.abs(sph[:, 3])
    b_lo, b_hi = (sph[:, :3] - r[:, None]).min(0), (sph[:, :3] + r[:, None]).max(0)
    inner = np.nonzero((cnt == 0) & np.all(centres > b_lo + cs, 1) & np.all(centres < b_hi - cs, 1))[0]
    cell = int(inner[len(inner) // 2])
    centre = centres[cell]
    extreme = set(np.argmin(sph[:, :3] - r[:, None], 0).tolist()) | set(np.argmax(sph[:, :3] + r[:, None], 0).tolist())
    idx = [i for i in range(len(sph)) if i not in extreme][100:100 + k]
    rng = np.random.default_rng(k)
    flat.spheres['center'][idx] = _f32(centre + rng.uniform(-0.08, 0.08, (k, 3)) * cs)
    flat.spheres['radius'][idx] = _f32(rng.uniform(0.005, 0.02, k))
    return flat, cell, centre


@pytest.mark.parametrize("k", [127, 128])
def test_cell_list_at_its_limit(gh, k):
    flat, cell, _ = knot_scene(gh, k)
    base = _cell_counts(gh, sphere_table(sc.synthetic_scene("c3")))
    enabled, res, lo, cs, cnt = _cell_counts(gh, sphere_table(flat))
    if k == 127:
        assert enabled and cnt[cell] == 127
        assert np.array_equal(res, base[1]) and np.array_equal(lo, base[2]) and cs == base[3]
    else:
        assert not enabled                  # a refused grid keeps no geometry: the knot is the only change from 127


LIGHT = np.array([5.0, -20.0, 0.0])


def cluster_table(L, k, res=32):
    """2000 C3 spheres plus k tiny ones 120 units from LIGHT, around the centre direction of a cube-face cell that
    no C3 sphere reaches.  Returns (sphere table, that cell)."""
    base = sphere_table(sc.synthetic_scene("c3", n_spheres=2000))
    d = np.array([-1 + 2 * 20.5 / res, -1 + 2 * 12.5 / res, -1.0])        # -z face, cell (20, 12)
    d /= np.linalg.norm(d)
    cell = int(L.gh_light_cell(np.ascontiguousarray(d).ctypes.data, res))
    rng = np.random.default_rng(k)
    c = LIGHT + 120.0 * d + rng.uniform(-0.3, 0.3, (k, 3))
    knot = np.concatenate([c, rng.uniform(0.01, 0.03, (k, 1))], 1)
    return np.ascontiguousarray(_f32(np.concatenate([base, knot]))), base, cell


def _dir_cell_len(grid, cell):
    off = np.frombuffer(grid[0], np.uint32)
    return int(off[cell + 1]) - int(off[cell]), int(off[-1])


@pytest.mark.parametrize("k", [512, 513])
def test_direction_cell_at_the_sort_switch(gh, k):
    sph, base, cell = cluster_table(gh, k)
    before, n0 = _dir_cell_len(host_light(gh, np.ascontiguousarray(_f32(base)), LIGHT, 32), cell)
    n, total = _dir_cell_len(host_light(gh, sph, LIGHT, 32), cell)
    assert before == 0 and n == k and total == n0 + k


@pytest.mark.gpu
def test_device_builders_at_the_limits(gd):
    for k in (127, 128):
        sph = sphere_table(knot_scene(gd, k)[0])
        host, dev = host_cell(gd, sph, 0.35), device_cell(gd, sph, 0.35)
        assert host[0] == dev[0] == (k == 127), k
        assert dev[1:] == host[1:] or k == 128, k
    for k in (512, 513):
        sph, _, cell = cluster_table(gd, k)
        host = host_light(gd, sph, LIGHT, 32, packed=True)
        dev = device_light(gd, sph, LIGHT, 32)
        assert _dir_cell_len(host, cell)[0] == k
        cell_off, _, _, always, cand, head = host
        assert (dev[0], dev[1], dev[2], dev[3]) == (cell_off, cand, head, always), k


def _knot_rays(centre, knot, rng, n=4000):
    """Rays aimed at the knot's spheres from around it, and rays that start inside the knot."""
    o = centre + rng.normal(size=(n, 3)) * 6.0
    d = knot[rng.integers(0, len(knot), n)] + rng.uniform(-0.01, 0.01, (n, 3)) - o
    inside = np.concatenate([centre + rng.uniform(-0.3, 0.3, (n, 3)), rng.normal(size=(n, 3))], 1)
    out = np.concatenate([np.concatenate([o, d], 1), inside])
    out[:, 3:] /= np.linalg.norm(out[:, 3:], axis=1, keepdims=True)
    return out


@pytest.mark.gpu
def test_full_cell_renders_like_the_linear_scan(gpu, gd):
    flat, _, centre = knot_scene(gd, 127)
    dev = flat.upload(0)
    try:
        in_knot = flat.spheres['radius'] < 0.05
        rays = _knot_rays(centre, flat.spheres['center'][in_knot], np.random.default_rng(4))
        og, tg = dev.trace_rays(rays, accel="grid")
        ol, tl = dev.trace_rays(rays, accel="linear")
        assert np.array_equal(og, ol) and np.array_equal(_bits(tg), _bits(tl))
        assert np.isin(og, flat.spheres['order'][in_knot]).sum() > 250
        cam = _lib.Camera()
        cam.location[:] = centre + (0.0, 0.0, -1.5)
        cam.fov, cam.screen_width, cam.screen_height = 90.0, 4.0, 2.25
        for camera in (None, cam):
            g, sg = dev.render(96, 54, 3, fmt="f64", accel="grid", camera=camera)
            e, se = dev.render(96, 54, 3, fmt="f64", accel="exact", camera=camera)
            assert sg["accel_used"] == "grid"
            assert np.array_equal(_bits(g), _bits(e)) and sg["rays"] == se["rays"]
    finally:
        dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [127, 128])
def test_update_into_a_full_cell(gpu, gd, k):
    flat = knot_scene(gd, k)[0]
    fresh = flat.upload(0)
    _, st = fresh.render(16, 9, 1, fmt="f64", accel="auto")
    fresh.close()
    assert st["has_cell_grid"] == (k == 127)
    dev = sc.synthetic_scene("c3").upload(0)
    info = flat.update(dev, rebuild_grids=True)
    assert info["has_cell_grid"] == (k == 127) and "rebuild_cell_grid" in info["done"], info
    _assert_like_fresh(dev, flat)
    dev.close()


# ---- 5. output formats through the wavefront --------------------------------------------------------------------

@pytest.mark.gpu
def test_f32_and_rgb8_frames_and_band_parts(gpu):
    flat = sc.synthetic_scene("c3", n_spheres=2000)
    rng = np.random.default_rng(12)
    flat.spheres['material']['colour'] = _f32(rng.uniform(-0.8, 1.8, (2000, 3)))
    dev = flat.upload(0)
    w, h, depth = 80, 40, 3
    try:
        ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
        assert ref.min() < 0 and ref.max() > 1
        for accel in ("grid", "bvh", "linear"):
            f64, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            _assert_oracle(f64, st, ref, ref_rays, accel)
            want = {"f64": f64, "f32": f64.astype(np.float32), "rgb8": np.clip(quantise(f64), 0, 255).astype(np.uint8)}
            for fmt in ("f32", "rgb8"):
                got, _ = dev.render(w, h, depth, fmt=fmt, accel=accel)
                assert got.dtype == want[fmt].dtype and np.array_equal(got, want[fmt]), (accel, fmt)
            for fmt in ("f64", "f32", "rgb8"):
                out = np.zeros((h, w, 3), dtype=want[fmt].dtype)
                for part in range(3):
                    dev.render(w, h, depth, fmt=fmt, accel=accel, band_rows=8, n_parts=3, part=part, out=out)
                assert np.array_equal(out, want[fmt]), (accel, fmt)
    finally:
        dev.close()
