"""Scene model of the host side: Erlang-shaped records -> flat tables for the C ABI.

Records are the tagged tuples of raytracer.erl:72-81 as `scene_test` pins them
(raytracer.erl:760-801), e.g.
    ('sphere', 4, ('vector', 4, 0, 10), ('material', ('colour', 0, 0.5, 1), 20, 1, 0.1))
A scene is a list with the camera first (raytracer.erl:617-619).  Every numeric
field may be an int or a float (Erlang scene literals mix both, erl:619-664).
"""
import functools
import math

import numpy as np

from . import _lib


def demo_scene():
    """The built-in scene of scene/0, raytracer.erl:618-665, values as written there."""
    return [
        ('camera', ('vector', 0, 0, -2), ('vector', 0, 0, 0), 90, ('screen', 4, 3)),
        ('point_light', ('colour', 1, 1, 0.5), ('vector', 5, -2, 0), ('colour', 1, 1, 1)),
        ('point_light', ('colour', 1, 0, 0.5), ('vector', -10, 0, 7), ('colour', 1, 0, 0.5)),
        ('sphere', 4, ('vector', 4, 0, 10),
         ('material', ('colour', 0, 0.5, 1), 20, 1, 0.1)),
        ('sphere', 4, ('vector', -5, 3, 9),
         ('material', ('colour', 1, 0.5, 0), 4, 0.25, 0.5)),
        ('sphere', 4, ('vector', -4.5, -2.5, 14),
         ('material', ('colour', 0.5, 1, 0), 20, 0.25, 0.7)),
        ('triangle', ('vector', -2, 5, 5), ('vector', 4, 5, 10), ('vector', 4, -5, 10),
         ('material', ('colour', 1, 0.5, 0), 4, 0.25, 0.5)),
        ('plane', ('vector', 0, -1, 0), 5,
         ('material', ('colour', 1, 1, 1), 1, 0, 0.01)),
    ]


def _num(x):
    # Erlang numbers only; the atom 'undefined' (hand-built records, erl:1016-1020) is badarg
    if isinstance(x, bool) or not isinstance(x, (int, float, np.integer, np.floating)):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "not a number in a scene record: %r" % (x,))
    return float(x)


def _v3(rec, tag):
    if not (isinstance(rec, tuple) and len(rec) == 4 and rec[0] == tag):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "expected a #%s{} record, got %r" % (tag, rec))
    return (_num(rec[1]), _num(rec[2]), _num(rec[3]))


def _material(rec):
    if not (isinstance(rec, tuple) and len(rec) == 5 and rec[0] == 'material'):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "expected a #material{} record, got %r" % (rec,))
    return (_v3(rec[1], 'colour'), _num(rec[2]), _num(rec[3]), _num(rec[4]))


def camera_struct(rec):
    """#camera{location, rotation, fov, screen=#screen{width,height}} -> _lib.Camera."""
    if isinstance(rec, _lib.Camera):
        return rec
    if not (isinstance(rec, tuple) and len(rec) == 5 and rec[0] == 'camera'):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "the first scene element must be a #camera{} record")
    scr = rec[4]
    if not (isinstance(scr, tuple) and len(scr) == 3 and scr[0] == 'screen'):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "expected a #screen{} record in the camera")
    cam = _lib.Camera()
    cam.location[:] = _v3(rec[1], 'vector')
    cam.rotation[:] = _v3(rec[2], 'vector')
    cam.fov = _num(rec[3])
    cam.screen_width = _num(scr[1])
    cam.screen_height = _num(scr[2])
    return cam


class FlatScene:
    """The four element tables plus the camera, ready for ert_scene_create."""

    def __init__(self, camera, lights, spheres, triangles, planes):
        self.camera = camera
        self.lights = lights
        self.spheres = spheres
        self.triangles = triangles
        self.planes = planes

    def upload(self, device=0):
        return _lib.Scene.create(self.camera, self.lights, self.spheres, self.triangles,
                                 self.planes, device=device)

    def update(self, dev, rebuild_grids=False, rebuild=False):
        """Puts these tables into the device scene `dev` (an upload of a scene with the same list shape).  With
        rebuild_grids, cell and direction grids the change made stale (or an earlier update dropped) are built again
        on the device, byte-identical to what a fresh upload of these tables builds; without, they are dropped."""
        return dev.update(self.camera, self.lights, self.spheres, self.triangles, self.planes,
                          rebuild_grids=rebuild_grids, rebuild=rebuild)

    @property
    def n_elements(self):
        return len(self.lights) + len(self.spheres) + len(self.triangles) + len(self.planes)


def _set_mat(row, mat):
    colour, sp, sh, refl = mat
    row['material']['colour'] = colour
    row['material']['specular_power'] = sp
    row['material']['shininess'] = sh
    row['material']['reflectivity'] = refl


def flatten(scene):
    """[Camera | Rest] (raytracer.erl:180) -> FlatScene.  List positions after the camera
    become `order`; elements that are no known record are skipped like erl:357-358."""
    if not isinstance(scene, (list, tuple)) or len(scene) == 0:
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "scene must be a non-empty list, camera first")
    camera = camera_struct(scene[0])
    lights, spheres, tris, planes = [], [], [], []
    for order, e in enumerate(scene[1:]):
        tag = e[0] if isinstance(e, tuple) and len(e) else None
        if tag == 'point_light' and len(e) == 4:
            lights.append((order, _v3(e[1], 'colour'), _v3(e[2], 'vector'), _v3(e[3], 'colour')))
        elif tag == 'sphere' and len(e) == 4:
            spheres.append((order, _num(e[1]), _v3(e[2], 'vector'), _material(e[3])))
        elif tag == 'triangle' and len(e) == 5:
            tris.append((order, _v3(e[1], 'vector'), _v3(e[2], 'vector'), _v3(e[3], 'vector'),
                         _material(e[4])))
        elif tag == 'plane' and len(e) == 4:
            planes.append((order, _v3(e[1], 'vector'), _num(e[2]), _material(e[3])))
        # anything else: not an object, not a light — ignored by the reference
    lt = np.zeros(len(lights), dtype=_lib.LIGHT_DT)
    for i, (o, dc, loc, sc) in enumerate(lights):
        lt[i]['diffuse_colour'] = dc
        lt[i]['location'] = loc
        lt[i]['specular_colour'] = sc
        lt[i]['order'] = o
    st = np.zeros(len(spheres), dtype=_lib.SPHERE_DT)
    for i, (o, r, c, m) in enumerate(spheres):
        st[i]['radius'] = r
        st[i]['center'] = c
        _set_mat(st[i], m)
        st[i]['order'] = o
    tt = np.zeros(len(tris), dtype=_lib.TRIANGLE_DT)
    for i, (o, v1, v2, v3, m) in enumerate(tris):
        tt[i]['v1'], tt[i]['v2'], tt[i]['v3'] = v1, v2, v3
        _set_mat(tt[i], m)
        tt[i]['order'] = o
    pt = np.zeros(len(planes), dtype=_lib.PLANE_DT)
    for i, (o, n, d, m) in enumerate(planes):
        pt[i]['normal'] = n
        pt[i]['distance'] = d
        _set_mat(pt[i], m)
        pt[i]['order'] = o
    return FlatScene(camera, lt, st, tt, pt)


# ---------------------------------------------------------------------------
# Synthetic scenes (SURVEY.md §8(d), configs C3/C4): "randomly generated scene
# (not done)" is on the reference's own to-do list (raytracer.erl:35).
# ---------------------------------------------------------------------------
_MASK = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64_uniform(seed, count):
    """count doubles in [0,1): u_k = (splitmix64 output k >> 11) * 2^-53."""
    k = np.arange(1, count + 1, dtype=np.uint64)
    with np.errstate(over='ignore'):
        z = np.uint64(seed) + k * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) * (2.0 ** -53)


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


SYNTH_CONFIGS = {
    # name: (n_spheres, (xlo,xhi), (ylo,yhi), (zlo,zhi), (rlo,rhi), seed)
    "c3": (10_000, (-40.0, 40.0), (-30.0, 4.0), (5.0, 85.0), (0.2, 0.8), 0xE7A9C0DE00000003),
    "c4": (1_000_000, (-200.0, 200.0), (-150.0, 4.0), (5.0, 405.0), (0.2, 1.0), 0xE7A9C0DE00000004),
}


def synthetic_scene(name="c3", n_spheres=None, seed=None):
    """Random-sphere scene of SURVEY §8(d): camera (0,0,-2) fov 90 screen 4x2.25, the demo
    floor plane, three point lights, n spheres.  Every value is rounded to float32 so that a
    double-precision CPU evaluation and the GPU start from identical inputs.  List order: lights, spheres, plane."""
    n0, xr, yr, zr, rr, seed0 = SYNTH_CONFIGS[name]
    n = n0 if n_spheres is None else int(n_spheres)
    seed = seed0 if seed is None else seed
    u = splitmix64_uniform(seed, n * 10).reshape(n, 10)
    cam = _lib.Camera()
    cam.location[:] = (0.0, 0.0, -2.0)
    cam.rotation[:] = (0.0, 0.0, 0.0)
    cam.fov = 90.0
    cam.screen_width, cam.screen_height = 4.0, 2.25

    lights = np.zeros(3, dtype=_lib.LIGHT_DT)
    lights['location'] = [(5, -20, 0), (-30, -10, 20), (20, -40, 60)]
    lights['diffuse_colour'] = [(1, 1, 0.5), (1, 0, 0.5), (1, 1, 1)]
    lights['specular_colour'] = [(1, 1, 1), (1, 0, 0.5), (1, 1, 1)]
    lights['order'] = [0, 1, 2]

    sp = np.zeros(n, dtype=_lib.SPHERE_DT)
    sp['center'][:, 0] = _f32(xr[0] + u[:, 0] * (xr[1] - xr[0]))
    sp['center'][:, 1] = _f32(yr[0] + u[:, 1] * (yr[1] - yr[0]))
    sp['center'][:, 2] = _f32(zr[0] + u[:, 2] * (zr[1] - zr[0]))
    sp['radius'] = _f32(rr[0] + u[:, 3] * (rr[1] - rr[0]))
    sp['material']['colour'][:, 0] = _f32(u[:, 4])
    sp['material']['colour'][:, 1] = _f32(u[:, 5])
    sp['material']['colour'][:, 2] = _f32(u[:, 6])
    powers = np.array([1.0, 4.0, 20.0, 50.0])
    sp['material']['specular_power'] = powers[np.minimum((u[:, 7] * 4).astype(np.int64), 3)]
    sp['material']['shininess'] = _f32(u[:, 8])
    sp['material']['reflectivity'] = _f32(u[:, 9] * 0.7)
    sp['order'] = np.arange(3, 3 + n, dtype=np.int32)

    planes = np.zeros(1, dtype=_lib.PLANE_DT)
    planes['normal'] = [(0, -1, 0)]
    planes['distance'] = 5
    planes['material']['colour'] = [(1, 1, 1)]
    planes['material']['specular_power'] = 1
    planes['material']['shininess'] = 0
    planes['material']['reflectivity'] = _f32(0.01)
    planes['order'] = 3 + n
    return FlatScene(cam, lights, sp, np.zeros(0, dtype=_lib.TRIANGLE_DT), planes)


def pose_camera(k, n_poses=64):
    """Camera of pose k for the C5 batch (SURVEY §8(d)): only the location varies, because
    the reference ignores rotation (raytracer.erl:487)."""
    cam = _lib.Camera()
    a = 2.0 * math.pi * k / n_poses
    cam.location[:] = (4.0 * math.sin(a), -1.0 + math.cos(a) / 2.0, -2.0 - k / 16.0)
    cam.rotation[:] = (0.0, 0.0, 0.0)
    cam.fov = 90.0
    cam.screen_width, cam.screen_height = 4.0, 3.0
    return cam


# ---------------------------------------------------------------------------
# Triangle meshes.  A mesh of a million faces goes straight from index arrays to the
# triangle table, without one Erlang-shaped tuple per face.
# ---------------------------------------------------------------------------
def mesh_triangles(vertices, faces, material, first_order):
    """vertices (V, 3) numbers, faces (F, 3) vertex indices, material ((r, g, b), specular_power, shininess,
    reflectivity) -> a TRIANGLE_DT table whose rows are the faces in order, list positions first_order,
    first_order + 1, ...  Equal to flatten() of the same faces written as #triangle{} records."""
    v = np.asarray(vertices, dtype=np.float64)
    f = np.asarray(faces)
    if v.ndim != 2 or v.shape[1] != 3 or f.ndim != 2 or f.shape[1] != 3:
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "vertices and faces must be (n, 3) arrays")
    if not np.issubdtype(f.dtype, np.integer):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "faces must hold vertex indices")
    if len(f) and (f.min() < 0 or f.max() >= len(v)):
        raise _lib.BadArg(_lib.ERT_ERR_BADARG, "a face refers to a vertex that does not exist")
    colour, sp, sh, refl = material
    t = np.zeros(len(f), dtype=_lib.TRIANGLE_DT)
    t['v1'], t['v2'], t['v3'] = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    t['material']['colour'] = [_num(c) for c in colour]
    t['material']['specular_power'] = _num(sp)
    t['material']['shininess'] = _num(sh)
    t['material']['reflectivity'] = _num(refl)
    t['order'] = np.arange(first_order, first_order + len(f), dtype=np.int32)
    return t


@functools.lru_cache(maxsize=None)
def _icosphere(level):
    """Unit icosphere: (vertices, faces), faces wound so that (v2 - v1) x (v3 - v1) points outwards."""
    p = (1.0 + math.sqrt(5.0)) / 2.0
    verts = [(-1, p, 0), (1, p, 0), (-1, -p, 0), (1, -p, 0), (0, -1, p), (0, 1, p), (0, -1, -p), (0, 1, -p),
             (p, 0, -1), (p, 0, 1), (-p, 0, -1), (-p, 0, 1)]
    verts = [tuple(c / math.sqrt(1 + p * p) for c in v) for v in verts]
    faces = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2),
             (10, 7, 6), (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11),
             (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    for _ in range(level):
        mid = {}

        def m(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                x = [(verts[a][k] + verts[b][k]) / 2 for k in range(3)]
                n = math.sqrt(sum(c * c for c in x))
                verts.append(tuple(c / n for c in x))
                mid[key] = len(verts) - 1
            return mid[key]
        nf = []
        for a, b, c in faces:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        faces = nf
    v = np.array(verts)
    f = np.array(faces, dtype=np.int64)
    n = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    inward = np.einsum('ij,ij->i', n, v[f].mean(axis=1)) < 0
    f[inward] = f[inward][:, [0, 2, 1]]
    return v, f


def _f1(x):
    return float(np.float32(x))


MESH_CONFIGS = {
    # name: (C3 spheres, heightfield cells per side, icospheres, icosphere level, seed)
    "m3": (3000, 64, 10, 3, 0xE7A9C0DE00000103),
    "m4": (10_000, 512, 24, 5, 0xE7A9C0DE00000104),
}


def mesh_scene(name="m3", n_triangles=None, frame=0):
    """Triangle-mesh workload: the camera, lights and plane of synthetic_scene, the spheres of the C3 recipe,
    a heightfield sheet over the floor and closed icosphere meshes among the spheres (their back faces put
    entry faces behind reflection and shadow rays).  Both meshes face the camera and the outside.  Every value
    is float32-rounded and drawn from splitmix64_uniform.  List order: lights, spheres, triangles, plane.
    n_triangles keeps the first that many triangles (scenes either side of the triangle-BVH threshold).  frame k
    (animated_scene) moves the spheres, shifts the sheet's waves by the phase 2 pi k / 64 and moves every icosphere
    rigidly; frame 0 is the still scene."""
    n_sph, cells, n_ico, level, seed = MESH_CONFIGS[name]
    base = synthetic_scene("c3", n_spheres=n_sph)
    u = splitmix64_uniform(seed, 4 + 8 * n_ico)
    # heightfield sheet 0.5 above the floor (y = 5): y grows downwards, so faces wound with (e1 x e2).y < 0
    xs = np.linspace(-40.0, 40.0, cells + 1)
    zs = np.linspace(5.0, 85.0, cells + 1)
    X, Z = np.meshgrid(xs, zs, indexing='ij')
    phase, swing = _frame_motion(frame)
    Y = 4.5 - 0.4 * (np.sin(X * (0.3 + u[0] * 0.2) + phase) * np.cos(Z * (0.3 + u[1] * 0.2)) + 1.0)
    sheet_v = _f32(np.stack([X, Y, Z], axis=-1).reshape(-1, 3))
    idx = np.arange((cells + 1) * (cells + 1)).reshape(cells + 1, cells + 1)
    p00, p10, p01, p11 = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, 1:].ravel()
    sheet_f = np.stack([np.stack([p00, p10, p01], 1), np.stack([p10, p11, p01], 1)], 1).reshape(-1, 3)
    first = 3 + n_sph
    tabs = [mesh_triangles(sheet_v, sheet_f, ((_f1(0.6), _f1(0.55), _f1(0.5)), 4.0, _f1(0.2), _f1(0.1)), first)]
    first += len(sheet_f)
    ico_v, ico_f = _icosphere(level)
    ico_dir = _directions(seed ^ ANIM_SEED, n_ico)
    for k in range(n_ico):
        r = u[4 + 8 * k: 12 + 8 * k]
        c = np.array((-35.0 + 70.0 * r[0], -25.0 + 26.0 * r[1], 10.0 + 70.0 * r[2])) + swing * ANIM_AMPLITUDE * ico_dir[k]
        rad = 2.0 + 3.0 * r[3]
        mat = ((_f1(r[4]), _f1(r[5]), _f1(r[6])), 20.0, _f1(0.5), _f1(0.2 + 0.5 * r[7]))
        tabs.append(mesh_triangles(_f32(ico_v * rad + c), ico_f, mat, first))
        first += len(ico_f)
    tris = np.concatenate(tabs)
    if n_triangles is not None:
        tris = tris[:int(n_triangles)].copy()
    planes = base.planes.copy()
    planes['order'] = 3 + n_sph + len(tris)
    return FlatScene(base.camera, base.lights, _moved_spheres(base.spheres, seed0_of("c3"), frame), tris, planes)


# ---------------------------------------------------------------------------
# Animation: frame k of a scene whose values move and whose list shape stays (ert_scene_update).
# ---------------------------------------------------------------------------
ANIM_SEED = 0xA11E0000A11E0000      # xor-ed into a scene's seed for the motion directions
ANIM_AMPLITUDE = 1.0                # scene units
ANIM_PERIOD = 64                    # frames


def seed0_of(name):
    return SYNTH_CONFIGS[name][5]


def _frame_motion(k):
    """(sheet phase, sphere / icosphere displacement factor) of frame k: both periodic in ANIM_PERIOD frames."""
    a = 2.0 * math.pi * k / ANIM_PERIOD
    return a, math.sin(a)


def _directions(seed, n):
    """n unit vectors from splitmix64_uniform (uniform in the cube, normalised)."""
    d = splitmix64_uniform(seed, 3 * n).reshape(n, 3) * 2.0 - 1.0
    return d / np.maximum(np.linalg.norm(d, axis=1), 1e-12)[:, None]


def _moved_spheres(spheres, seed, k):
    """Every sphere displaced by ANIM_AMPLITUDE sin(2 pi k / 64) along its own direction, float32-rounded."""
    out = spheres.copy()
    _, swing = _frame_motion(k)
    if swing:
        d = _directions(seed ^ ANIM_SEED, len(spheres))
        out['center'] = _f32(spheres['center'] + swing * ANIM_AMPLITUDE * d)
    return out


def animated_scene(name, k):
    """Frame k of the animation of c3 / c4 (synthetic_scene) or m3 / m4 (mesh_scene): the same list as frame 0 (the
    still scene) with moved spheres, a travelling wave on the heightfield sheet and rigidly moved icospheres."""
    if name in MESH_CONFIGS:
        return mesh_scene(name, frame=k)
    base = synthetic_scene(name)
    return FlatScene(base.camera, base.lights, _moved_spheres(base.spheres, seed0_of(name), k), base.triangles,
                     base.planes)
