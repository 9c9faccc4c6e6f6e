"""CPU tests of the host grid builders after their per-element arithmetic moved to grid_math.h (shared with the
device builders of grid_build.cuh): the cell grid and the direction grids of C3 keep the bytes they had before the
move, and pack_light_grid gives the layout the shadow kernels walk.  Built through tests/gridbuild/host_shim.cpp."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from eraytracer_b200 import scene as sc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "gridbuild", "_build")
SO = os.path.join(BUILD, "libgridhost_test.so")
CSRC = os.path.join(ROOT, "eraytracer_b200", "csrc")
vp, ll = ctypes.c_void_p, ctypes.c_longlong

# SHA-256 of C3's grids as the builders made them before grid_math.h: the cell grid (geometry, blocks, over_filter,
# over_sph, big) per density, the direction grids (cell_off, entries, fs, always) of the three lights at res 128
C3_CELL_SHA256 = {
    0.35: "63f45b0ba3adcb005f5bda8df5b9271af984f4b7a7c2ce34164cd1b334e1a1cc",
    1.0: "7183f1d7d11ee5b65038efd9f6f4d727e2f4757b633801893f82eea13ca9369d",
}
C3_LIGHT_SHA256 = (
    "df5b1e8a056a8b7079fe007409b86f35769a74a29794eaa671d50bfc13d8d562",
    "c82db5fe34e012314184b0188864547408d1e982ad4c4ba17ed2f89042dad932",
    "d429c22c41c3495edd03a2ac18ba9e7d2667ed485299497cfa7e8f7ec9a69ba7",
)
CAND_DT = np.dtype([("f", "<f4", 4), ("sphere", "<i4"), ("dmin", "<f4"), ("pad", "<i4", 2)])


def declare(L):
    """ctypes signatures of host_shim.cpp (shared with the GPU test)."""
    for f in ("gh_cell", "gh_light", "gh_cell_blocks", "gh_cell_over_filter", "gh_cell_over_sph", "gh_cell_big",
              "gh_light_cell_off", "gh_light_entries", "gh_light_fs", "gh_light_always"):
        getattr(L, f).restype = vp
    L.gh_cell.argtypes = [vp, ll, ctypes.c_double]
    L.gh_light.argtypes = [vp, ll, vp, ctypes.c_int]
    for f in ("gh_cell_n_blocks", "gh_cell_n_over", "gh_cell_n_big", "gh_light_n_cells", "gh_light_n_entries",
              "gh_light_n_always"):
        getattr(L, f).restype = ll
        getattr(L, f).argtypes = [vp]
    for f in ("gh_cell_blocks", "gh_cell_over_filter", "gh_cell_over_sph", "gh_cell_big", "gh_light_cell_off",
              "gh_light_entries", "gh_light_fs", "gh_light_always", "gh_cell_enabled", "gh_cell_free",
              "gh_light_free"):
        getattr(L, f).argtypes = [vp]
    L.gh_cell_geometry.argtypes = [vp, vp, vp, vp, vp]
    L.gh_light_packed.argtypes = [vp, vp, vp]
    L.gh_light_cell.restype = ll
    L.gh_light_cell.argtypes = [vp, ctypes.c_int]
    L.gh_light_cell_f32.restype = ll
    L.gh_light_cell_f32.argtypes = [vp, ctypes.c_int]
    return L


@pytest.fixture(scope="module")
def gh():
    os.makedirs(BUILD, exist_ok=True)
    src = [os.path.join(HERE, "gridbuild", "host_shim.cpp"), os.path.join(CSRC, "cell_grid.cpp"),
           os.path.join(CSRC, "light_grid.cpp")]
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO] + src
                          + ["-lpthread"])
    return declare(ctypes.CDLL(SO))


def sphere_table(flat):
    """{cx, cy, cz, r} in list order, as ert_scene_create keeps the spheres."""
    s = flat.spheres[np.argsort(flat.spheres['order'], kind='stable')]
    return np.ascontiguousarray(np.concatenate([s['center'], s['radius'][:, None]], 1), dtype=np.float64)


def scene_lights(flat):
    return [np.ascontiguousarray(l['location'], dtype=np.float64)
            for l in flat.lights[np.argsort(flat.lights['order'])]]


def raw(p, n):
    return ctypes.string_at(p, n) if n else b""


def host_cell(L, sph, density):
    """(enabled, geometry bytes, blocks, over_filter, over_sph, big) of the host builder."""
    g = L.gh_cell(sph.ctypes.data, len(sph), density)
    res, lo, hi, cs = np.zeros(3, np.int32), np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(3, np.float32)
    L.gh_cell_geometry(g, res.ctypes.data, lo.ctypes.data, hi.ctypes.data, cs.ctypes.data)
    n_over = L.gh_cell_n_over(g)
    out = (bool(L.gh_cell_enabled(g)), res.tobytes() + lo.tobytes() + hi.tobytes() + cs.tobytes(),
           raw(L.gh_cell_blocks(g), 128 * L.gh_cell_n_blocks(g)), raw(L.gh_cell_over_filter(g), 16 * n_over),
           raw(L.gh_cell_over_sph(g), 4 * n_over), raw(L.gh_cell_big(g), 4 * L.gh_cell_n_big(g)))
    L.gh_cell_free(g)
    return out


def host_light(L, sph, light, res, packed=False):
    """(cell_off, entries, fs, always) of the host builder, or None over the entry budget; with packed, also
    (cand, head) in the device layout."""
    light = np.ascontiguousarray(light, dtype=np.float64)
    g = L.gh_light(sph.ctypes.data, len(sph), light.ctypes.data, res)
    if not g:
        return None
    nc, ne, na = L.gh_light_n_cells(g), L.gh_light_n_entries(g), L.gh_light_n_always(g)
    out = (raw(L.gh_light_cell_off(g), 4 * (nc + 1)), raw(L.gh_light_entries(g), 8 * ne),
           raw(L.gh_light_fs(g), 16 * ne), raw(L.gh_light_always(g), 4 * na))
    if packed:
        cand, head = np.zeros(ne, CAND_DT), np.zeros(nc, CAND_DT)
        L.gh_light_packed(g, cand.ctypes.data, head.ctypes.data)
        out = out + (cand.tobytes(), head.tobytes())
    L.gh_light_free(g)
    return out


def sha(parts):
    h = hashlib.sha256()
    for p in parts:
        h.update(p)
    return h.hexdigest()


@pytest.mark.parametrize("density", [0.35, 1.0])
def test_c3_cell_grid_bytes_are_unchanged(gh, density):
    enabled, *parts = host_cell(gh, sphere_table(sc.synthetic_scene("c3")), density)
    assert enabled
    assert sha(parts) == C3_CELL_SHA256[density]


def test_c3_direction_grid_bytes_are_unchanged(gh):
    flat = sc.synthetic_scene("c3")
    sph = sphere_table(flat)
    lights = scene_lights(flat)
    assert len(lights) == len(C3_LIGHT_SHA256)
    for light, want in zip(lights, C3_LIGHT_SHA256):
        assert sha(host_light(gh, sph, light, 128)) == want


def test_packed_direction_grid_is_the_host_grid(gh):
    """pack_light_grid: every entry with its filter sphere, and per cell the nearest one with the range of the rest."""
    flat = sc.synthetic_scene("c3", n_spheres=2000)
    sph = sphere_table(flat)
    off, ent, fs, always, cand, head = host_light(gh, sph, scene_lights(flat)[0], 32, packed=True)
    off = np.frombuffer(off, np.uint32)
    ent = np.frombuffer(ent, np.dtype([("sphere", "<i4"), ("dmin", "<f4")]))
    fs = np.frombuffer(fs, np.float32).reshape(-1, 4)
    cand, head = np.frombuffer(cand, CAND_DT), np.frombuffer(head, CAND_DT)
    assert np.array_equal(cand["sphere"], ent["sphere"]) and np.array_equal(cand["dmin"], ent["dmin"])
    assert np.array_equal(cand["f"], fs) and not cand["pad"].any()
    e0, e1 = off[:-1].astype(np.int64), off[1:].astype(np.int64)
    full = e1 > e0
    assert full.any() and (~full).any()
    assert np.array_equal(head["sphere"][full], ent["sphere"][e0[full]])
    assert np.array_equal(head["pad"][full], np.stack([e0[full] + 1, e1[full]], 1))
    assert np.all(head["sphere"][~full] == -1) and np.all(np.isinf(head["dmin"][~full]))
    assert np.all(head["f"][~full][:, 3] == np.float32(-3.0e38)) and not head["pad"][~full].any()
