"""CPU tests of the triangle BVH (eraytracer_b200/csrc/bvh_build.cpp, tri_walk.h) and of the mesh workloads.

The walk only prunes: what it must guarantee is that every triangle the literal FP64 test (raytracer.erl:402-455)
accepts, and that could still win under (Distance, list position), lies in a leaf the walk enters.  The walk is
restated in tests/tribvh/shim.cpp over the device's own bound code (tri_walk.h) and checked with the incumbent's
cull at the triangle's own Distance, the tightest cull under which it still wins its tie."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "tribvh", "_build")
SO = os.path.join(BUILD, "libtribvh_test.so")
# node array + leaf order of the C3 sphere tree as the sphere-only builder made it before the builder took boxes
C3_SPHERE_TREE_SHA256 = "750cde9469d972a09606cd004524d4228d9ba52094461b460f72c89002ee641e"
vp, ll = ctypes.c_void_p, ctypes.c_longlong


@pytest.fixture(scope="module")
def tb():
    os.makedirs(BUILD, exist_ok=True)
    src = [os.path.join(HERE, "tribvh", "shim.cpp"), os.path.join(ROOT, "eraytracer_b200", "csrc", "bvh_build.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO] + src
                          + ["-lpthread"])
    L = ctypes.CDLL(SO)
    L.tb_build.restype = vp
    L.tb_build.argtypes = [vp, ll]
    L.tb_free.argtypes = [vp]
    for name in ("tb_n_always", "tb_n_tree"):
        getattr(L, name).restype = ll
        getattr(L, name).argtypes = [vp]
    L.tb_depth.argtypes = [vp]
    L.tb_constants.argtypes = [vp, vp]
    L.tb_check.argtypes = [vp, vp, ll, vp, ll, ctypes.c_int, vp]
    L.tb_sphere_tree.restype = ll
    L.tb_sphere_tree.argtypes = [vp, vp, ll, vp, ll]
    return L


def _check(L, tris, rays, margins=True):
    tris = np.ascontiguousarray(tris, dtype=np.float64).reshape(-1, 9)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    h = L.tb_build(tris.ctypes.data, len(tris))
    stats = np.zeros(4, dtype=np.int64)
    L.tb_check(h, tris.ctypes.data, len(tris), rays.ctypes.data, len(rays), 1 if margins else 0, stats.ctypes.data)
    n_always = L.tb_n_always(h)
    L.tb_free(h)
    return stats, n_always


def _mesh(rng, n, scale, offset, f32):
    """n small triangles in a box of side `scale` around `offset`, some in axis planes, some degenerate."""
    c = offset + rng.uniform(-scale, scale, (n, 3))
    e = rng.normal(0, scale / 20, (n, 2, 3))
    tris = np.concatenate([c, c + e[:, 0], c + e[:, 1]], axis=1)
    ax = rng.integers(0, 3, n)
    flat = rng.uniform(0, 1, n) < 0.3                   # in an axis plane: a zero-thickness box
    for k in range(3):
        tris[flat, 3 * k + ax[flat]] = c[flat, ax[flat]]
    deg = rng.uniform(0, 1, n) < 0.05                    # collinear vertices
    tris[deg, 6:9] = tris[deg, 0:3] + 2.0 * (tris[deg, 3:6] - tris[deg, 0:3])
    if f32:
        tris = tris.astype(np.float32).astype(np.float64)
    return tris


def _rays(rng, tris, n):
    """Rays at the triangles' hard cases: det just above 1e-6 (grazing), through edges and vertices, in the plane,
    axis-parallel and non-unit directions, hits far behind the origin."""
    k = rng.integers(0, len(tris), n)
    v1, v2, v3 = tris[k, 0:3], tris[k, 3:6], tris[k, 6:9]
    e1, e2 = v2 - v1, v3 - v1
    nrm = np.cross(e1, e2)
    nn = np.linalg.norm(nrm, axis=1)
    nn[nn == 0] = 1.0
    nrm /= nn[:, None]
    a, b = rng.uniform(0, 1, n), rng.uniform(0, 1, n)
    cls = rng.integers(0, 6, n)
    a = np.where(cls == 1, np.round(a), a)               # on an edge / vertex
    b = np.where(cls == 1, 1.0 - a, b)
    sw = a + b > 1
    a, b = np.where(sw, 1 - a, a), np.where(sw, 1 - b, b)
    P = v1 + a[:, None] * e1 + b[:, None] * e2 + rng.normal(0, 1e-9, (n, 3)) * np.abs(v1).max(axis=1)[:, None]
    # det = D . (E2 x E1) = -D . n |E1 x E2|: the grazing class has det a few ulps to a few percent above 1e-6
    area2 = nn
    t = e1 / np.maximum(np.linalg.norm(e1, axis=1), 1e-300)[:, None]
    D = np.where((cls == 0)[:, None], t - nrm * (1e-6 * (1 + rng.choice([1e-12, 1e-6, 0.05], n)) / area2)[:, None],
                 -nrm + rng.normal(0, 0.3, (n, 3)))
    D = np.where((cls == 2)[:, None], e1, D)             # in the plane
    axd = np.zeros((n, 3))
    axd[np.arange(n), rng.integers(0, 3, n)] = rng.choice([-1.0, 1.0], n)
    D = np.where((cls == 3)[:, None], axd, D)            # axis-parallel
    D *= rng.choice([1.0, 1e-3, 3.0, 1e3], n)[:, None] * np.where(cls == 0, 1.0, 1.0)[:, None]
    D[cls == 0] /= np.linalg.norm(D[cls == 0], axis=1)[:, None]
    s = rng.uniform(-5, 5, n)
    s = np.where(cls == 4, -rng.uniform(1e2, 1e5, n), s)  # the hit far behind the origin
    O = P - s[:, None] * D
    return np.concatenate([O, D], axis=1)


CASES = [
    # (n triangles, extent, offset, float32 vertices)
    (400, 1.0, 0.0, True),
    (400, 50.0, 1e4, True),
    (400, 50.0, -9.7e3, False),
    (300, 0.01, 3.0, False),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_walk_enters_every_accepted_triangle(tb, case):
    n, ext, off, f32 = CASES[case]
    rng = np.random.default_rng(100 + case)
    tris = _mesh(rng, n, ext, off, f32)
    rays = _rays(rng, tris, 20000)
    stats, _ = _check(tb, tris, rays)
    assert stats[0] > 2000, stats
    assert stats[1] == 0, stats
    assert stats[2] < 0.01 * len(rays), stats


def test_walk_misses_hits_without_margins(tb):
    """The same cases with every rounding term of tri_walk.h dropped: the walk loses accepted triangles."""
    missed = 0
    for case, (n, ext, off, f32) in enumerate(CASES):
        rng = np.random.default_rng(100 + case)
        tris = _mesh(rng, n, ext, off, f32)
        stats, _ = _check(tb, tris, _rays(rng, tris, 20000), margins=False)
        missed += int(stats[1])
    assert missed > 0


def test_huge_and_far_triangles_go_to_the_always_list(tb):
    rng = np.random.default_rng(7)
    tris = _mesh(rng, 200, 1.0, 0.0, True)
    huge = np.array([[-1e4, 0, -1e4, 1e4, 0, -1e4, 0, 0, 1e4]], dtype=np.float64)
    far = np.array([[1e31, 0, 0, 1e31, 1, 0, 1e31, 0, 1]], dtype=np.float64)
    tris = np.concatenate([tris, huge, far])
    rays = _rays(rng, tris[:200], 5000)
    stats, n_always = _check(tb, tris, rays)
    assert n_always == 2
    assert stats[1] == 0, stats


def test_c3_sphere_tree_unchanged(tb):
    f = sc.synthetic_scene("c3")
    c = np.ascontiguousarray(f.spheres['center'])
    r = np.ascontiguousarray(f.spheres['radius'])
    buf = np.zeros(1 << 22, dtype=np.uint8)
    n = tb.tb_sphere_tree(c.ctypes.data, r.ctypes.data, len(r), buf.ctypes.data, len(buf))
    assert 0 < n <= len(buf)
    assert hashlib.sha256(buf[:n].tobytes()).hexdigest() == C3_SPHERE_TREE_SHA256


# ---- the mesh workloads ------------------------------------------------------------------------------------


def _digest(flat):
    h = hashlib.sha256()
    for tab in (flat.lights, flat.spheres, flat.triangles, flat.planes):
        h.update(np.ascontiguousarray(tab).tobytes())
    return h.hexdigest()


def test_mesh_scene_is_pinned():
    flat = sc.mesh_scene("m3")
    assert len(flat.triangles) == 20992 and len(flat.spheres) == 3000
    assert _digest(flat) == "d056577ce854579609a8d3ee290566c43863f80ff0ebbb8a13a62866c919f739"
    for k in ("v1", "v2", "v3"):
        v = flat.triangles[k]
        assert np.array_equal(v, v.astype(np.float32).astype(np.float64))
    orders = np.concatenate([flat.lights['order'], flat.spheres['order'], flat.triangles['order'], flat.planes['order']])
    assert np.array_equal(np.sort(orders), np.arange(len(orders)))
    assert flat.triangles['order'].min() == 3 + 3000 and flat.planes['order'][0] == orders.max()


def test_mesh_faces_wound_outwards():
    """Front faces towards the camera and the outside: the literal test's det >= 1e-6 for a ray from the camera."""
    flat = sc.mesh_scene("m3")
    tr = flat.triangles
    n = np.cross(tr['v2'] - tr['v1'], tr['v3'] - tr['v1'])
    sheet = tr[:2 * 64 * 64]
    assert (np.cross(sheet['v2'] - sheet['v1'], sheet['v3'] - sheet['v1'])[:, 1] < 0).all()
    ico = slice(2 * 64 * 64, None)
    cen = np.concatenate([(tr['v1'][ico] + tr['v2'][ico] + tr['v3'][ico]) / 3])
    per = 1280
    centres = cen.reshape(-1, per, 3).mean(axis=1)
    out = cen - np.repeat(centres, per, axis=0)
    assert (np.einsum('ij,ij->i', n[ico], out) > 0).all()


def test_mesh_triangles_equal_flatten():
    rng = np.random.default_rng(3)
    v = rng.uniform(-5, 5, (30, 3)).astype(np.float32).astype(np.float64)
    f = rng.integers(0, 30, (40, 3))
    mat = ((0.25, 0.5, 1), 20, 0.5, 0.25)
    t = sc.mesh_triangles(v, f, mat, 3)
    cam = ('camera', ('vector', 0, 0, -2), ('vector', 0, 0, 0), 90, ('screen', 4, 3))
    lights = [('point_light', ('colour', 1, 1, 1), ('vector', k, 0, 0), ('colour', 1, 1, 1)) for k in range(3)]
    recs = [('triangle',) + tuple(('vector',) + tuple(v[i]) for i in face)
            + (('material', ('colour',) + mat[0], mat[1], mat[2], mat[3]),) for face in f]
    ref = sc.flatten([cam] + lights + recs).triangles
    assert t.tobytes() == ref.tobytes()
    with pytest.raises(_lib.BadArg):
        sc.mesh_triangles(v, np.array([[0, 1, 30]]), mat, 0)
