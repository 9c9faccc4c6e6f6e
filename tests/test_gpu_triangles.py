"""Triangle meshes through the triangle BVH: every accel against ERT_ACCEL_EXACT (the linear FP64 scan of every
triangle, the GPU statement of raytracer.erl:300-346) and against the CPU oracle."""
import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc
from helpers import assert_double_parity, oracle_frame, quantise

pytestmark = pytest.mark.gpu

TRACE_ACCELS = ("linear", "bvh", "bvh_mega", "grid", "warp", "auto")
RENDER_ACCELS = ("exact", "linear", "bvh", "bvh_mega", "grid", "auto")


@pytest.fixture(scope="module")
def m3(gpu):
    flat = sc.mesh_scene("m3")
    dev = flat.upload(0)
    yield flat, dev
    dev.close()


def _edge_rays(flat, n, seed):
    """Rays aimed at the mesh's hard cases: through edges and vertices, lying in a triangle's plane, grazing with
    det just above 1e-6, axis-parallel and non-unit directions, starting inside the closed meshes, on a triangle,
    and far in front of a mesh (its hits then have negative Distance)."""
    rng = np.random.default_rng(seed)
    tr = flat.triangles
    k = rng.integers(0, len(tr), n)
    v1, v2, v3 = tr['v1'][k], tr['v2'][k], tr['v3'][k]
    e1, e2 = v2 - v1, v3 - v1
    nrm = np.cross(e1, e2)
    nrm /= np.linalg.norm(nrm, axis=1)[:, None]
    cls = rng.integers(0, 8, n)
    a = rng.uniform(0, 1, n)
    b = rng.uniform(0, 1, n)
    # target point: inside, on an edge, or on a vertex
    on_edge = cls == 1
    on_vert = cls == 2
    a = np.where(on_edge, a, np.where(on_vert, 0.0, a))
    b = np.where(on_edge, 1.0 - a, np.where(on_vert, 0.0, b))
    swap = a + b > 1
    a, b = np.where(swap, 1 - a, a), np.where(swap, 1 - b, b)
    P = v1 + a[:, None] * e1 + b[:, None] * e2
    O = P - nrm * rng.uniform(0.5, 60, n)[:, None] * 1.0 + rng.normal(0, 3, (n, 3))
    D = P - O
    # in the triangle's plane
    inplane = cls == 3
    O[inplane] = P[inplane] - e1[inplane] * 2.0
    D[inplane] = e1[inplane]
    # grazing: a direction almost in the plane, det = D . (E2 x E1) about 1e-6
    graze = cls == 4
    t = e1[graze] / np.linalg.norm(e1[graze], axis=1)[:, None]
    s2 = np.linalg.norm(np.cross(e2[graze], e1[graze]), axis=1)
    D[graze] = t - nrm[graze] * (1.05e-6 / s2)[:, None]
    O[graze] = P[graze] - D[graze] * 3.0
    # axis-parallel
    ax = cls == 5
    axis = rng.integers(0, 3, int(ax.sum()))
    Dax = np.zeros((int(ax.sum()), 3))
    Dax[np.arange(len(axis)), axis] = rng.choice([-1.0, 1.0], len(axis)) * rng.uniform(0.3, 3.0, len(axis))
    D[ax] = Dax
    O[ax] = P[ax] - Dax * rng.uniform(-20, 20, len(axis))[:, None]
    # starting on a triangle, or inside a closed mesh, in any direction
    on = cls == 6
    O[on] = P[on]
    D[on] = rng.normal(0, 1, (int(on.sum()), 3))
    # far in front: the mesh is far behind the origin of a ray pointing away from it
    far = cls == 7
    D[far] = -D[far]
    O[far] = P[far] + D[far] * rng.uniform(100, 1e4, int(far.sum()))[:, None]
    # non-unit directions everywhere but the grazing class
    scale = np.where(graze, 1.0, rng.choice([1.0, 0.01, 7.0, 1e3], n))
    D = D * scale[:, None]
    return np.ascontiguousarray(np.concatenate([O, D], axis=1))


def test_trace_rays_equal_exact(m3):
    flat, dev = m3
    rays = _edge_rays(flat, 240_000, 5)
    ref_o, ref_t = dev.trace_rays(rays, accel="exact")
    assert (ref_o >= 0).mean() > 0.5
    for accel in TRACE_ACCELS:
        o, t = dev.trace_rays(rays, accel=accel)
        bad = np.flatnonzero((o != ref_o) | (t.view(np.int64) != ref_t.view(np.int64)))
        assert bad.size == 0, (accel, bad.size, rays[bad[:3]], o[bad[:3]], ref_o[bad[:3]], t[bad[:3]], ref_t[bad[:3]])
    # the negative-Distance class is there
    assert (ref_t < 0).sum() > 1000


@pytest.mark.parametrize("depth", [1, 5])
def test_m3_frames_match_oracle(m3, depth):
    flat, dev = m3
    w, h = 48, 27
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    for accel in RENDER_ACCELS:
        f64, st = dev.render(w, h, depth, fmt="f64", accel=accel)
        rgb8, _ = dev.render(w, h, depth, fmt="rgb8", accel=accel)
        assert st["rays"] == ref_rays, accel
        assert np.array_equal(rgb8.astype(np.int64), quantise(ref)), accel
        assert_double_parity(f64, ref)


def test_auto_never_picks_exact(m3):
    flat, dev = m3
    _, st = dev.render(16, 9, 1, accel="auto")
    assert st["accel_used"] != "exact"
    small = sc.mesh_scene("m3", n_triangles=64)
    d2 = small.upload(0)
    for accel in RENDER_ACCELS[1:]:
        a, _ = d2.render(40, 24, 3, fmt="f64", accel=accel)
        b, _ = d2.render(40, 24, 3, fmt="f64", accel="exact")
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), accel
    d2.close()


def test_counts(m3):
    flat, dev = m3
    _, ex = dev.render(64, 36, 1, accel="exact", flags=_lib.FLAG_COUNT_TESTS)
    _, au = dev.render(64, 36, 1, accel="auto", flags=_lib.FLAG_COUNT_TESTS)
    assert ex["rays"] == au["rays"]
    n_obj = len(flat.triangles) + len(flat.planes)
    # every ray tests every triangle and plane (a shadow ray skips its target, and one whose target is missed
    # tests nothing)
    assert 0.9 * ex["rays"] * n_obj <= ex["exact_other_tests"] <= ex["rays"] * n_obj
    assert au["exact_other_tests"] < 0.01 * ex["exact_other_tests"]
    assert au["box_tests"] > 0


def test_m4_bands_auto_equal_exact(gpu):
    flat = sc.mesh_scene("m4")
    dev = flat.upload(0)
    W, H, depth = 3840, 2160, 5
    for band in (0, 130, 269):
        # rows [8 band, 8 band + 8) of the full frame: one part of n_parts bands of 8 rows
        n_parts = H // 8
        a, _ = dev.render(W, H, depth, fmt="f64", accel="auto", band_rows=8, n_parts=n_parts, part=band)
        b, _ = dev.render(W, H, depth, fmt="f64", accel="exact", band_rows=8, n_parts=n_parts, part=band)
        rows = slice(8 * band, 8 * band + 8)
        assert np.array_equal(a[rows].view(np.int64), b[rows].view(np.int64)), band
    dev.close()


def test_clone_and_parts(m3):
    flat, dev = m3
    w, h, depth = 96, 54, 3
    full, _ = dev.render(w, h, depth, fmt="f64")
    clone = dev.clone(0)
    c, _ = clone.render(w, h, depth, fmt="f64")
    assert np.array_equal(c.view(np.int64), full.view(np.int64))
    for n_parts in (2, 8):
        out = np.zeros_like(full)
        for part in range(n_parts):
            f, _ = clone.render(w, h, depth, fmt="f64", band_rows=8, n_parts=n_parts, part=part)
            for b in range(part, (h + 7) // 8, n_parts):
                out[8 * b:8 * b + 8] = f[8 * b:8 * b + 8]
        assert np.array_equal(out.view(np.int64), full.view(np.int64)), n_parts
    clone.close()
