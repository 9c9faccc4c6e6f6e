"""Test infrastructure for ERT_FLAG_CAMERA_ROTATION: the C oracle with the rotation restated on top of it
(tests/camrot/rot_oracle.c, which includes oracle/oracle.c unchanged), a pure-Python restatement over
oracle/pyoracle.py, and the library's own host matrix through a shim of scene_tables.cpp.  Each restates the rule of
include/ert_b200.h independently; the tests hold all three to each other bit for bit."""
import ctypes
import math
import os
import subprocess

import numpy as np

from oracle import orc, pyoracle

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "camrot", "_build")
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int32)
_libs = {}


def _build(name, cmd, src, libs=()):
    so = os.path.join(BUILD, name)
    if name not in _libs:
        os.makedirs(BUILD, exist_ok=True)
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
            subprocess.check_call(cmd + ["-o", so] + src[:1] + [s for s in src[1:] if s.endswith(".cpp")] + list(libs))
        _libs[name] = ctypes.CDLL(so)
    return _libs[name]


def oracle_lib():
    src = [os.path.join(HERE, "camrot", "rot_oracle.c"), os.path.join(ROOT, "oracle", "oracle.c")]
    L = _build("librot_oracle.so", ["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC",
                                     "-fvisibility=hidden", "-Wall", "-std=c11", "-D_GNU_SOURCE", "-shared"], src,
               ["-lm", "-lpthread"])
    L.orc_camera_matrix.argtypes = [_dp, _dp]
    L.orc_camera_matrix.restype = ctypes.c_int
    L.orc_ray_through_pixel_rot.argtypes = [ctypes.c_double, ctypes.c_double, _dp, ctypes.c_int, _dp]
    L.orc_ray_through_pixel_rot.restype = None
    L.orc_render_rot.argtypes = [_dp, ctypes.c_int, _ip, _dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_int64, _ip, _ip, _dp, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64)]
    L.orc_render_rot.restype = ctypes.c_int
    return L


def host_lib():
    csrc = os.path.join(ROOT, "eraytracer_b200", "csrc")
    src = [os.path.join(HERE, "camrot", "shim.cpp"), os.path.join(csrc, "scene_tables.cpp"),
           os.path.join(csrc, "scene_tables.h"), os.path.join(ROOT, "include", "ert_b200.h")]
    L = _build("libcamrot_host.so", ["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-Wall", "-shared", "-fPIC"],
               src)
    L.cr_camera_matrix.argtypes = [_dp, _dp]
    L.cr_camera_matrix.restype = ctypes.c_int
    L.cr_check_rotation.argtypes = [_dp]
    L.cr_check_rotation.restype = ctypes.c_char_p
    return L


def _arr(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.float64))


def library_matrix(rot):
    """(M as a (3, 3) array, identity?) from the library's host code."""
    r, m = _arr(rot), np.zeros(9)
    ident = host_lib().cr_camera_matrix(r.ctypes.data_as(_dp), m.ctypes.data_as(_dp))
    return m.reshape(3, 3), bool(ident)


def oracle_matrix(rot):
    r, m = _arr(rot), np.zeros(9)
    ident = oracle_lib().orc_camera_matrix(r.ctypes.data_as(_dp), m.ctypes.data_as(_dp))
    return m.reshape(3, 3), bool(ident)


# ---- pure Python, over pyoracle ------------------------------------------------------------------------------
_QUARTER = {0.0: (0.0, 1.0), 90.0: (1.0, 0.0), -270.0: (1.0, 0.0), 180.0: (0.0, -1.0), -180.0: (0.0, -1.0),
            270.0: (-1.0, 0.0), -90.0: (-1.0, 0.0)}


def py_sin_cos(deg):
    a = math.fmod(float(deg), 360.0)
    if a in _QUARTER:                       # -0.0 == 0.0 finds the entry of 0
        return _QUARTER[a]
    r = a * (math.pi / 180.0)
    return math.sin(r), math.cos(r)


def py_matrix(rot):
    (sx, cx), (sy, cy), (sz, cz) = (py_sin_cos(a) for a in rot)
    rx = ((1.0, 0.0, 0.0), (0.0, cx, -sx), (0.0, sx, cx))
    ry = ((cy, 0.0, sy), (0.0, 1.0, 0.0), (-sy, 0.0, cy))
    rz = ((cz, -sz, 0.0), (sz, cz, 0.0), (0.0, 0.0, 1.0))

    def mul(a, b):
        return tuple(tuple((a[i][0] * b[0][j] + a[i][1] * b[1][j]) + a[i][2] * b[2][j] for j in range(3))
                     for i in range(3))
    m = mul(ry, mul(rx, rz))
    ident = all(m[i][j] == (1.0 if i == j else 0.0) for i in range(3) for j in range(3))
    return np.array(m), ident


def py_ray_through_pixel(x, y, camera, rotate):
    """raytracer.erl:510-511 with the rotation; camera is the #camera{} tuple."""
    if not rotate:
        return pyoracle.ray_through_pixel(x, y, camera)
    m, _ = py_matrix(camera[2][1:])
    loc = camera[1]
    _, vx, vy, vz = pyoracle.vector_sub(pyoracle.point_on_screen(x, y, camera), loc)
    d = tuple((float(m[i][0]) * vx + float(m[i][1]) * vy) + float(m[i][2]) * vz for i in range(3))
    return ('ray', loc, pyoracle.vector_normalize(('vector',) + d))


def py_render(scene_list, width, height, depth, rotate):
    """The frame (H, W, 3) of pyoracle with rotated primary rays."""
    camera, rest = scene_list[0], scene_list[1:]
    out = np.zeros((height, width, 3))
    for y in range(height):
        for x in range(width):
            c = pyoracle.pixel_colour_from_ray(py_ray_through_pixel(x / width, y / height, camera, rotate), rest,
                                               depth)
            out[y, x] = c[1:]
    return out


# ---- C oracle renders ----------------------------------------------------------------------------------------
def render(cam9, kind, f, width, height, depth, rotate=True, pixels=None, nthreads=None):
    """orc.render with the rotate switch: (rgb float64[npix, 3], rays)."""
    L = oracle_lib()
    cam9 = _arr(cam9)
    kind = np.ascontiguousarray(kind, dtype=np.int32)
    f = _arr(f)
    nthreads = nthreads or os.cpu_count() or 1
    if pixels is None:
        npix, xp, yp = width * height, None, None
    else:
        xs = np.ascontiguousarray(pixels[0], dtype=np.int32)
        ys = np.ascontiguousarray(pixels[1], dtype=np.int32)
        npix, xp, yp = len(xs), xs.ctypes.data_as(_ip), ys.ctypes.data_as(_ip)
    out = np.zeros((npix, 3))
    counters = (ctypes.c_uint64 * 2)()
    rc = L.orc_render_rot(cam9.ctypes.data_as(_dp), len(kind), kind.ctypes.data_as(_ip), f.ctypes.data_as(_dp),
                          width, height, depth, 1 if rotate else 0, npix, xp, yp, out.ctypes.data_as(_dp),
                          int(nthreads), counters)
    if rc != 0:
        raise ValueError("orc_render_rot rejected its arguments")
    return out, int(counters[0])


def camera_array(camera, rotation=None):
    """_lib.Camera -> the oracle's cam[9], with `rotation` in place of the camera's own if given."""
    rot = list(camera.rotation) if rotation is None else list(rotation)
    return np.array(list(camera.location) + rot + [camera.fov, camera.screen_width, camera.screen_height])


def oracle_frame(flat, width, height, depth, rotation=None, camera=None, pixels=None):
    """The rotated frame of a FlatScene: (rgb (H, W, 3) or (npix, 3), rays)."""
    from helpers import oracle_scene_from_flat
    _, kind, f = oracle_scene_from_flat(flat)
    cam9 = camera_array(flat.camera if camera is None else camera, rotation)
    rgb, rays = render(cam9, kind, f, width, height, depth, rotate=True, pixels=pixels)
    return (rgb.reshape(height, width, 3) if pixels is None else rgb), rays


__all__ = ["library_matrix", "oracle_matrix", "py_matrix", "py_render", "render", "oracle_frame", "camera_array",
           "orc"]
