"""CPU checks of ERT_FLAG_CAMERA_ROTATION (include/ert_b200.h, DESIGN.md "Camera rotation").

Three restatements of the rotation are held to each other bit for bit: the library's host matrix (scene_tables.cpp
through tests/camrot/shim.cpp), the C oracle's (tests/camrot/rot_oracle.c over oracle/oracle.c) and a pure-Python one
over oracle/pyoracle.py (tests/camrot_oracle.py).  The rotated frames of the two oracles must agree too, and
look_at must aim the centre pixel at its target.  The Python look_at is held to raytracer_gpu:look_at/2 evaluated by
oracle/erlref.py, and the NIF's Opts decoder to the flag."""
import ctypes
import inspect
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import camrot_oracle as cr
from eraytracer_b200 import _lib, raytracer
from eraytracer_b200 import scene as sc
from erl_scenes import stress_scene
from helpers import oracle_scene_from_flat
from oracle import pyoracle

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

QUARTERS = [q * s for q in (0.0, 90.0, 180.0, 270.0, 360.0) for s in (1.0, -1.0)]


def _angles():
    rng = np.random.default_rng(2026)
    near90 = [float(np.nextafter(90.0, 0.0)), float(np.nextafter(90.0, 180.0)), 90.0 + 1e-12, 89.999999,
              -90.00000001, 450.0000001, float(np.nextafter(-270.0, 0.0))]
    big = [720.0, -1080.0, 3600.0, 1e300, -1e300, 1e-300, -1e-300, -0.0, 5e-324, 1e17, 2.0 ** 60 + 90.0]
    return QUARTERS + near90 + big + [float(a) for a in rng.uniform(-720.0, 720.0, 40)] + \
        [float(a) for a in rng.uniform(-1e6, 1e6, 10)]


def _rotations():
    angles = _angles()
    rng = np.random.default_rng(7)
    rots = [(a, 0.0, 0.0) for a in angles] + [(0.0, a, 0.0) for a in angles] + [(0.0, 0.0, a) for a in angles]
    rots += [tuple(float(x) for x in rng.choice(angles, 3)) for _ in range(300)]
    rots += [tuple(float(x) for x in rng.choice(QUARTERS, 3)) for _ in range(100)]
    return rots


def test_three_matrices_are_bit_equal():
    for rot in _rotations():
        m_lib, id_lib = cr.library_matrix(rot)
        m_orc, id_orc = cr.oracle_matrix(rot)
        m_py, id_py = cr.py_matrix(rot)
        assert m_lib.tobytes() == m_orc.tobytes() == m_py.tobytes(), rot
        assert id_lib == id_orc == id_py, rot
        assert id_lib == bool(np.array_equal(m_lib, np.eye(3))), rot


def test_quarter_turns_are_exact_permutations():
    for rx in QUARTERS:
        for ry in QUARTERS:
            for rz in QUARTERS:
                m, ident = cr.library_matrix((rx, ry, rz))
                assert set(np.unique(m)) <= {-1.0, 0.0, 1.0}, (rx, ry, rz)
                assert np.array_equal(np.abs(m).sum(axis=0), np.ones(3))
                assert np.array_equal(np.abs(m).sum(axis=1), np.ones(3))
                assert abs(np.linalg.det(m) - 1.0) == 0.0
    for rot in [(0.0, 0.0, 0.0), (360.0, -720.0, 0.0), (180.0, 180.0, 180.0), (-0.0, -0.0, -0.0), (1e-300 * 0, 0, 0),
                (-180.0, 180.0, -180.0), (720.0, 0.0, -360.0)]:
        m, ident = cr.library_matrix(rot)
        assert ident and np.array_equal(m, np.eye(3)), rot
    for rot in [(1e-300, 0.0, 0.0), (0.0, float(np.nextafter(360.0, 0.0)), 0.0), (180.0, 180.0, 0.0), (90.0, 0, 0)]:
        assert not cr.library_matrix(rot)[1], rot


def test_orientation_examples_of_the_header():
    fwd = np.array([0.0, 0.0, 1.0])
    for rot, want in [((0, 90, 0), (1, 0, 0)), ((0, 180, 0), (0, 0, -1)), ((90, 0, 0), (0, -1, 0)),
                      ((-90, 0, 0), (0, 1, 0)), ((0, -90, 0), (-1, 0, 0))]:
        m, _ = cr.library_matrix(rot)
        assert np.array_equal(m @ fwd, np.array(want, dtype=float)), rot
    # rz rolls about the view axis: the forward axis stays, screen x turns towards screen y
    m, _ = cr.library_matrix((0, 0, 90))
    assert np.array_equal(m @ fwd, fwd) and np.array_equal(m @ np.array([1.0, 0, 0]), np.array([0.0, 1, 0]))


def test_non_finite_rotations_are_reported():
    L = cr.host_lib()
    for rot in [(math.nan, 0, 0), (0, math.inf, 0), (0, 0, -math.inf)]:
        r = np.array(rot, dtype=float)
        assert L.cr_check_rotation(r.ctypes.data_as(cr._dp)) == b"camera rotation has a non-finite field"
    r = np.array([1e308, -1e308, 0.0])
    assert L.cr_check_rotation(r.ctypes.data_as(cr._dp)) == b""


def _with_rotation(scene_list, rot):
    cam = scene_list[0]
    return [(cam[0], cam[1], ('vector',) + tuple(rot), cam[3], cam[4])] + list(scene_list[1:])


SMALL_POSES = [(0.0, 90.0, 0.0), (90.0, 0.0, 0.0), (-30.0, 200.0, 15.0), (12.5, -47.0, 0.0), (0.0, 180.0, 90.0)]


@pytest.mark.parametrize("name", ["demo", "stress"])
def test_c_oracle_and_pyoracle_frames_are_bit_equal(name):
    base = pyoracle.scene() if name == "demo" else stress_scene()
    from oracle import orc
    kind, f = orc.flatten(base[1:])
    for rot in SMALL_POSES + [sc.look_at(base[0][1], ('vector', -4.5, -2.5, 14))]:
        scene_list = _with_rotation(base, rot)
        cam9 = orc.camera_array(scene_list[0])
        for depth in (1, 3):
            c_rgb, _ = cr.render(cam9, kind, f, 12, 9, depth, rotate=True)
            py_rgb = cr.py_render(scene_list, 12, 9, depth, rotate=True)
            assert c_rgb.reshape(9, 12, 3).tobytes() == py_rgb.tobytes(), (name, rot, depth)


def test_identity_rotation_renders_the_unrotated_frame():
    from oracle import orc
    for scene_list in (pyoracle.scene(), stress_scene()):
        kind, f = orc.flatten(scene_list[1:])
        plain, plain_rays, _ = orc.render(orc.camera_array(scene_list[0]), kind, f, 20, 15, 5)
        for rot in [(0, 0, 0), (360, -720, 0), (180, 180, 180)]:
            cam9 = orc.camera_array(_with_rotation(scene_list, rot)[0])
            got, rays = cr.render(cam9, kind, f, 20, 15, 5, rotate=True)
            assert got.tobytes() == plain.tobytes() and rays == plain_rays, rot
            off, off_rays = cr.render(cam9, kind, f, 20, 15, 5, rotate=False)
            assert off.tobytes() == plain.tobytes() and off_rays == plain_rays
        # without the switch the rotation is not read
        cam9 = orc.camera_array(_with_rotation(scene_list, (33, 44, 55))[0])
        assert cr.render(cam9, kind, f, 20, 15, 5, rotate=False)[0].tobytes() == plain.tobytes()


def test_look_at_centre_pixel_hits_the_target_sphere():
    flat = sc.synthetic_scene("c3", n_spheres=400)
    cam0, kind, f = oracle_scene_from_flat(flat)
    L = cr.oracle_lib()
    picked = [0, 17, 123, 399]
    for loc in [(0.0, 0.0, -2.0), (60.0, -20.0, 45.0), (0.0, -80.0, 45.0), (-70.0, 4.5, 90.0), (1.5, -3.0, 30.0)]:
        for i in picked:
            c = flat.spheres['center'][i]
            rot = sc.look_at(loc, tuple(float(x) for x in c))
            cam9 = np.array(list(loc) + list(rot) + [90.0, 4.0, 2.25])
            ray = np.zeros(6)
            L.orc_ray_through_pixel_rot(0.5, 0.5, cam9.ctypes.data_as(cr._dp), 1, ray.ctypes.data_as(cr._dp))
            d = c - np.array(loc)
            assert np.allclose(ray[3:], d / np.linalg.norm(d), atol=1e-12)
            # pixel (W/2, H/2) of an even W x H is the screen's centre; nothing in front of the sphere's centre
            # but what the oracle's nearest hit says: that sphere, unless another one covers it
            hit = np.zeros(7)
            from oracle import orc
            idx = orc.lib().orc_nearest_object_intersecting_ray(ray.ctypes.data_as(cr._dp), len(kind),
                                                                kind.ctypes.data_as(cr._ip), f.ctypes.data_as(cr._dp),
                                                                hit.ctypes.data_as(cr._dp))
            order = int(flat.spheres['order'][i])
            if idx != order:
                # another sphere is in the way: it must be nearer than the target's centre
                assert 0 < hit[0] < np.linalg.norm(d)
            else:
                assert idx == order
    # a lone target from afar: the centre pixel must hit it
    one = sc.synthetic_scene("c3", n_spheres=1)
    _, kind1, f1 = oracle_scene_from_flat(one)
    c = tuple(float(x) for x in one.spheres['center'][0])
    for loc in [(30.0, -40.0, -10.0), (c[0], c[1] - 50.0, c[2]), (c[0] + 0.1, c[1] + 3.0, c[2] + 20.0)]:
        rot = sc.look_at(loc, c)
        cam9 = np.array(list(loc) + list(rot) + [90.0, 4.0, 2.25])
        rgb, _ = cr.render(cam9, kind1, f1, 64, 36, 1, rotate=True, pixels=([32], [18]))
        ray = np.zeros(6)
        L.orc_ray_through_pixel_rot(0.5, 0.5, cam9.ctypes.data_as(cr._dp), 1, ray.ctypes.data_as(cr._dp))
        from oracle import orc
        hit = np.zeros(7)
        idx = orc.lib().orc_nearest_object_intersecting_ray(ray.ctypes.data_as(cr._dp), len(kind1),
                                                            kind1.ctypes.data_as(cr._ip), f1.ctypes.data_as(cr._dp),
                                                            hit.ctypes.data_as(cr._dp))
        assert idx == int(one.spheres['order'][0]), loc


def _erl_module():
    from oracle import erlref
    sys.setrecursionlimit(200000)
    with open(os.path.join(ROOT, "erl", "raytracer_gpu.erl")) as fh:
        m = erlref.Module(fh.read(), name="raytracer_gpu")
    base = m.apply_remote

    def apply_remote(mod, fname, args):
        # math:atan2/2 is the platform libm's atan2, as BEAM's BIF is
        if mod == "math" and fname == "atan2":
            return math.atan2(args[0], args[1])
        return base(mod, fname, args)
    m.apply_remote = apply_remote
    return erlref, m


def test_look_at_matches_the_erlang_function():
    erlref, m = _erl_module()
    rng = np.random.default_rng(5)
    pairs = [((0, 0, -2), (4, 0, 10)), ((0, 0, -2), (0, 0, 10)), ((0, 0, 0), (0, 5, 0)), ((0, 0, 0), (0, -5, 0)),
             ((1, 2, 3), (1, 2, -7)), ((0.5, -1.25, 3.0), (0.5, -1.25, 3.0)), ((0.0, 0.0, 0.0), (-3.0, 0.0, 0.0)),
             ((0, 0, 0), (0, 0, -1)), ((0.0, 0.0, 0.0), (0.0, -0.0, 1.0))]
    pairs += [(tuple(float(x) for x in rng.uniform(-100, 100, 3)), tuple(float(x) for x in rng.uniform(-100, 100, 3)))
              for _ in range(60)]
    for loc, tgt in pairs:
        want = sc.look_at(loc, tgt)
        V = erlref.Atom('vector')
        got = m.call("look_at", (V,) + tuple(loc), (V,) + tuple(tgt))
        got = erlref.to_py(got) if hasattr(erlref, "to_py") else got
        assert got[0] == 'vector'
        assert np.array(got[1:], dtype=float).tobytes() == np.array(want, dtype=float).tobytes(), (loc, tgt)
        # records and 3-sequences are the same input
        assert sc.look_at(('vector',) + tuple(loc), ('vector',) + tuple(tgt)) == want


def test_python_entry_points_default_to_the_references_camera():
    for fn in (_lib.Scene.render, _lib.Scene.render_async, raytracer.render_frame, raytracer.render_frame_multi_gpu):
        assert inspect.signature(fn).parameters["camera_rotation"].default is False, fn.__qualname__
    for fn in (raytracer.raytraced_pixel_list_gpu, raytracer.raytraced_pixel_list_gpu_distributed):
        assert list(inspect.signature(fn).parameters) == ["width", "height", "scene_list", "recursion_depth"]
    s = _lib.Scene(None, 0)
    assert s._params(16, 8, 1, "rgb8", "auto", 0, 1, 0, 0, None, 1).flags == 0
    assert s._params(16, 8, 1, "rgb8", "auto", 0, 1, 0, 1, None, 1, True).flags == 1 | 16


def test_flag_matches_the_header(tmp_path):
    src = tmp_path / "flag.c"
    src.write_text('#include <stdio.h>\n#include "ert_b200.h"\n'
                   'int main(void) { printf("%u %d\\n", ERT_FLAG_CAMERA_ROTATION, (int)ERT_ABI_VERSION); return 0; }\n')
    exe = tmp_path / "flag"
    subprocess.check_call(["gcc", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    flag, abi = map(int, subprocess.check_output([str(exe)], text=True).split())
    assert flag == _lib.FLAG_CAMERA_ROTATION == 16
    assert abi == 3
    for other in (_lib.FLAG_COUNT_TESTS, _lib.FLAG_WF_UNSORTED, _lib.FLAG_NO_LIGHT_GRID, _lib.FLAG_TIME_KERNELS):
        assert other & flag == 0


def test_nif_decodes_the_camera_rotation_option(tmp_path, monkeypatch):
    import nif_mock
    so = str(tmp_path / "raytracer_gpu_opts.so")
    lib_dir = os.path.join(ROOT, "eraytracer_b200", "lib")
    if not os.path.exists(os.path.join(lib_dir, "libert_b200.so")):
        pytest.skip("the library is not built")
    subprocess.check_call(
        ["gcc", "-Wall", "-Wextra", "-Werror", "-O1", "-fPIC", "-shared",
         "-I" + os.path.join(ROOT, "tests", "mock_erl"), "-I" + os.path.join(ROOT, "include"),
         os.path.join(HERE, "camrot", "nif_opts.c"), os.path.join(ROOT, "tests", "mock_erl", "mock_erl_nif.c"),
         "-L" + lib_dir, "-lert_b200", "-Wl,-rpath," + lib_dir, "-o", so])
    monkeypatch.setattr(nif_mock, "SO", so)
    beam = nif_mock.MockBeam()
    L = beam.L
    L.camrot_decode_opts.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint)]
    L.camrot_decode_opts.restype = ctypes.c_int

    def decode(opts):
        flags = ctypes.c_uint(0)
        ok = L.camrot_decode_opts(beam.env, beam.term(opts), ctypes.byref(flags))
        return flags.value if ok else None
    assert decode([]) == 0
    assert decode([("camera_rotation", True)]) == _lib.FLAG_CAMERA_ROTATION
    assert decode([("camera_rotation", False)]) == 0
    assert decode([("camera_rotation", True), ("camera_rotation", False)]) == 0
    assert decode([("format", "f64"), ("camera_rotation", True), ("supersample", 2)]) == _lib.FLAG_CAMERA_ROTATION
    for bad in (1, 0, "yes", "undefined", 1.0, (True,), [True]):
        assert decode([("camera_rotation", bad)]) is None, bad
    assert decode([("camera_rotation",)]) is None
