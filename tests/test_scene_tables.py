"""CPU tests of the scene's element tables (eraytracer_b200/csrc/scene_tables.cpp): the checks and the one packer that
ert_scene_create and ert_scene_update share, through a host shim (tests/scenetables/shim.cpp).

A moved scene equals a fresh create only while both entry points write the same bytes: the packed tables are held to
a numpy restatement of the layouts, a shuffled descriptor packed through the update's mapping must give the create's
bytes, and every single-defect descriptor must get the messages both entry points have always returned.  Create's
messages are also taken from the real library: ert_scene_create checks the descriptor before it looks for a device."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from eraytracer_b200 import _lib, scene as sc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "eraytracer_b200", "csrc")
BUILD = os.path.join(HERE, "scenetables", "_build")
SO = os.path.join(BUILD, "libscenetables_test.so")
vp = ctypes.c_void_p
KINDS = ["lights", "planes", "triangles", "spheres"]          # ElemKind order
LAYOUT = {"lights": 9, "planes": 4, "plane_mat": 6, "tris": 9, "tri_mat": 6, "sph_exact": 4, "sph_mat": 6,
          "sph_refl": 1}


@pytest.fixture(scope="module")
def st():
    os.makedirs(BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", SO,
                           os.path.join(HERE, "scenetables", "shim.cpp"), os.path.join(CSRC, "scene_tables.cpp")])
    L = ctypes.CDLL(SO)
    L.st_table.restype = ctypes.c_char_p
    L.st_table.argtypes = [ctypes.c_int, vp, vp, vp]
    L.st_create.restype = ctypes.c_char_p
    L.st_create.argtypes = [vp, vp, vp]
    L.st_update.restype = ctypes.c_char_p
    L.st_update.argtypes = [vp, vp, vp, vp]
    tables = []
    for t in range(L.st_n_tables()):
        kind, per, changed = ctypes.c_int(), ctypes.c_int(), ctypes.c_uint()
        name = L.st_table(t, ctypes.byref(kind), ctypes.byref(per), ctypes.byref(changed)).decode()
        tables.append((name, kind.value, per.value, changed.value))
    L.tables = tables
    return L


def _mixed(seed=7, nl=5, ns=300, nt=120, npl=4):
    """A scene of every kind with interleaved, shuffled list positions and random values."""
    rng = np.random.default_rng(seed)
    order = rng.permutation(nl + ns + nt + npl).astype(np.int32)
    f = sc.FlatScene(sc.synthetic_scene("c3", n_spheres=1).camera, np.zeros(nl, _lib.LIGHT_DT),
                     np.zeros(ns, _lib.SPHERE_DT), np.zeros(nt, _lib.TRIANGLE_DT), np.zeros(npl, _lib.PLANE_DT))
    o = 0
    for tab in (f.lights, f.spheres, f.triangles, f.planes):
        tab['order'] = order[o:o + len(tab)]
        o += len(tab)
        for name in tab.dtype.names:
            if name in ('order', 'reserved'):
                continue
            if name == 'material':
                for m in tab.dtype['material'].names:
                    tab['material'][m] = rng.normal(0, 10, tab['material'][m].shape)
            else:
                tab[name] = rng.normal(0, 10, tab[name].shape)
    return f


SCENES = {"c3": lambda: sc.synthetic_scene("c3"), "m3": lambda: sc.mesh_scene("m3"), "mixed": _mixed}


def _tabs(f):
    return {"lights": f.lights, "spheres": f.spheres, "triangles": f.triangles, "planes": f.planes}


def _desc(f, tabs=None):
    t = tabs or _tabs(f)
    return _lib.Scene._desc(f.camera, t["lights"], t["spheres"], t["triangles"], t["planes"])


def _restated(f):
    """The tables and list positions in scene element order, restated from the layouts: lights and spheres by list
    position, planes and triangles as listed."""
    L = f.lights[np.argsort(f.lights['order'], kind='stable')]
    S = f.spheres[np.argsort(f.spheres['order'], kind='stable')]
    P, T = f.planes, f.triangles

    def mat(m):
        return np.column_stack([m['colour'], m['specular_power'], m['shininess'], m['reflectivity']])
    tabs = {"lights": np.column_stack([L['diffuse_colour'], L['location'], L['specular_colour']]),
            "planes": np.column_stack([P['normal'], P['distance']]), "plane_mat": mat(P['material']),
            "tris": np.column_stack([T['v1'], T['v2'], T['v3']]), "tri_mat": mat(T['material']),
            "sph_exact": np.column_stack([S['center'], S['radius']]), "sph_mat": mat(S['material']),
            "sph_refl": S['material']['reflectivity']}
    return {k: np.ascontiguousarray(v, dtype=np.float64).tobytes() for k, v in tabs.items()}, \
        [L['order'], P['order'], T['order'], S['order']]


def _counts(f):
    return [len(_tabs(f)[k]) for k in KINDS]


def _split(st, buf, counts):
    out, o = {}, 0
    for name, kind, per, _ in st.tables:
        n = counts[kind] * per
        out[name] = buf[o:o + n].tobytes()
        o += n
    return out


def _create(st, f, desc=None):
    """(message, tables by name, list positions per kind) of the create path"""
    counts = _counts(f)
    tab = np.full(sum(counts[k] * per for _, k, per, _ in st.tables), np.nan)
    order = np.full(sum(counts), -7, dtype=np.int32)
    if desc is None:
        desc, keep = _desc(f)
    msg = st.st_create(ctypes.byref(desc) if desc is not False else None, tab.ctypes.data, order.ctypes.data).decode()
    return msg, _split(st, tab, counts), np.split(order, np.cumsum(counts)[:-1])


def _update(st, f, orders, desc):
    """(message, tables by name) of the update path of the scene created from f, for the descriptor desc"""
    counts = _counts(f)
    staging = np.full(sum(counts[k] * per for _, k, per, _ in st.tables), np.nan)
    flat = np.ascontiguousarray(np.concatenate(orders), dtype=np.int32)
    n = np.array(counts, dtype=np.int64)
    msg = st.st_update(ctypes.byref(desc) if desc is not False else None, flat.ctypes.data, n.ctypes.data,
                       staging.ctypes.data).decode()
    return msg, _split(st, staging, counts)


def test_table_list(st):
    """The eight tables: DevScene's arrays of the same names, their layouts and their ert_update_info.changed bits."""
    changed = {"lights": "LIGHTS", "planes": "PLANES", "plane_mat": "PLANES", "tris": "TRIANGLES",
               "tri_mat": "TRIANGLE_MAT", "sph_exact": "SPHERES", "sph_mat": "SPHERE_MAT", "sph_refl": "SPHERE_MAT"}
    kind = {"lights": 0, "planes": 1, "plane_mat": 1, "tris": 2, "tri_mat": 2, "sph_exact": 3, "sph_mat": 3,
            "sph_refl": 3}
    assert [t[0] for t in st.tables] == list(LAYOUT)
    device = open(os.path.join(CSRC, "ert_device.cuh")).read()
    for name, k, per, bit in st.tables:
        assert (k, per) == (kind[name], LAYOUT[name]), name
        assert bit == 1 << _lib.UPDATE_CHANGED.index(changed[name].lower()), name
        assert re.search(r"const double4? \*%s;" % name, device), name


@pytest.mark.parametrize("name", list(SCENES))
def test_create_packs_the_layouts(st, name):
    f = SCENES[name]()
    msg, tabs, orders = _create(st, f)
    assert msg == ""
    want, want_orders = _restated(f)
    assert tabs == want
    for got, exp in zip(orders, want_orders):
        assert np.array_equal(got, exp)


@pytest.mark.parametrize("name", list(SCENES))
def test_update_of_a_shuffled_descriptor_packs_the_create_bytes(st, name):
    f = SCENES[name]()
    _, created, orders = _create(st, f)
    rng = np.random.default_rng(len(name))
    shuffled = {k: v[rng.permutation(len(v))] for k, v in _tabs(f).items()}
    for tabs in (None, shuffled):
        desc, keep = _desc(f, tabs)
        msg, staged = _update(st, f, orders, desc)
        assert msg == ""
        assert staged == created


# (name, change, create's message, update's message); None: the path accepts the descriptor
NAN, INF = float("nan"), float("inf")
NOT_FINITE = {"lights": "point_light has a non-finite field", "planes": "plane has a non-finite field",
              "triangles": "triangle has a non-finite field", "spheres": "sphere has a non-finite field"}
FIELDS = {"lights": ["diffuse_colour", "location", "specular_colour"], "planes": ["normal", "distance"],
          "triangles": ["v1", "v2", "v3"], "spheres": ["center", "radius"]}
MATERIAL = ["colour", "specular_power", "shininess", "reflectivity"]
NO_POSITIONS = "the %s do not have the list positions of the scene's create"
COUNTS = "element counts differ from the scene's (a new list shape needs ert_scene_create)"
CAMERA = "camera has a non-finite field"
DUP, DUP_KIND = "duplicate list position in `order`", "duplicate list position in `order` among the %s"


def _set(kind, field, value, i=1):
    def change(t, d):
        if field in MATERIAL:
            t[kind]['material'][field][i] = value
        elif t[kind][field].ndim > 1:
            t[kind][field][i, 1] = value
        else:
            t[kind][field][i] = value
    return change


def _set_desc(**fields):
    def change(t, d):
        d.update(fields)
    return change


def _camera(field, value):
    def change(t, d):
        d["camera." + field] = value
    return change


def _order(kind, i, value):
    def change(t, d):
        t[kind]['order'][i] = value(t) if callable(value) else value
    return change


def _both(*changes):
    def change(t, d):
        for c in changes:
            c(t, d)
    return change


def _defects():
    out = []
    for field in ("location", "fov", "screen_width", "screen_height"):
        for v in (NAN, -INF):
            out.append(("camera %s %r" % (field, v), _camera(field, v), CAMERA, CAMERA))
    for kind in KINDS:
        out.append(("NULL %s" % kind, _set_desc(**{kind: None}), "element table pointer is NULL",
                    "element table pointer is NULL"))
        for field in FIELDS[kind] + (MATERIAL if kind != "lights" else []):
            for v in (NAN, INF):
                out.append(("%s %s %r" % (kind, field, v), _set(kind, field, v), NOT_FINITE[kind], NOT_FINITE[kind]))
    out += [
        ("duplicate sphere order", _order("spheres", 3, lambda t: t["spheres"]['order'][4]), DUP, DUP_KIND % "spheres"),
        ("duplicate light order", _order("lights", 0, lambda t: t["lights"]['order'][1]), DUP, DUP_KIND % "lights"),
        ("sphere with a plane's order", _order("spheres", 3, lambda t: t["planes"]['order'][0]), DUP,
         NO_POSITIONS % "spheres"),
        ("triangle with a light's order", _order("triangles", 2, lambda t: t["lights"]['order'][0]), DUP,
         NO_POSITIONS % "triangles"),
        ("plane order not in the scene", _order("planes", 1, 10 ** 6), None, NO_POSITIONS % "planes"),
        ("negative sphere order", _order("spheres", 5, -3), "negative list position in `order`",
         NO_POSITIONS % "spheres"),
        ("one sphere fewer", _set_desc(n_spheres=299), None, COUNTS),
        ("negative count", _set_desc(n_planes=-1), "negative element count", COUNTS),
        ("too many spheres", _set_desc(n_spheres=1 << 28), "too many elements", COUNTS),
        ("NULL descriptor", False, "scene descriptor is NULL", "scene descriptor is NULL"),
        # several defects: the first in the order header, list positions, lights, planes, triangles, spheres
        ("negative count and NULL", _set_desc(n_planes=-1, spheres=None), "negative element count", COUNTS),
        ("NULL and too many", _set_desc(lights=None, n_spheres=1 << 28), "element table pointer is NULL", COUNTS),
        ("too many and camera", _both(_set_desc(n_triangles=1 << 28), _camera("fov", NAN)), "too many elements",
         COUNTS),
        ("counts and camera", _both(_set_desc(n_spheres=299), _camera("fov", NAN)), CAMERA, COUNTS),
        ("NULL and camera", _both(_set_desc(planes=None), _camera("fov", NAN)), "element table pointer is NULL",
         "element table pointer is NULL"),
        ("camera and duplicate order", _both(_camera("fov", NAN), _order("spheres", 3, lambda t: t["spheres"]['order'][4])),
         CAMERA, CAMERA),
        ("duplicate order and NaN", _both(_order("spheres", 3, lambda t: t["spheres"]['order'][4]),
                                          _set("lights", "location", NAN)), DUP, DUP_KIND % "spheres"),
        ("plane and sphere positions", _both(_order("planes", 1, 10 ** 6), _order("spheres", 5, 10 ** 6 + 1)), None,
         NO_POSITIONS % "spheres"),
        ("light and sphere positions", _both(_order("lights", 1, 10 ** 6), _order("spheres", 5, 10 ** 6 + 1)), None,
         NO_POSITIONS % "lights"),
        ("light and sphere NaN", _both(_set("spheres", "radius", NAN), _set("lights", "location", NAN)),
         NOT_FINITE["lights"], NOT_FINITE["lights"]),
        ("plane and triangle NaN", _both(_set("triangles", "v2", NAN), _set("planes", "shininess", NAN)),
         NOT_FINITE["planes"], NOT_FINITE["planes"]),
        ("triangle and sphere NaN", _both(_set("spheres", "center", NAN), _set("triangles", "colour", NAN)),
         NOT_FINITE["triangles"], NOT_FINITE["triangles"]),
    ]
    return out


DEFECTS = _defects()


def _defective(name):
    """(the mixed scene, the descriptor with the defect `name`, the tables it points into)"""
    f = _mixed()
    change = next(c for n, c, _, _ in DEFECTS if n == name)
    if change is False:
        return f, False, None
    tabs = {k: v.copy() for k, v in _tabs(f).items()}
    fields = {}
    change(tabs, fields)
    desc, keep = _desc(f, tabs)
    for k, v in fields.items():
        if k == "camera.location":
            desc.camera.location[2] = v
        elif k.startswith("camera."):
            setattr(desc.camera, k[7:], v)
        else:
            setattr(desc, k, v)
    return f, desc, keep


@pytest.mark.parametrize("name,create,update", [(n, c, u) for n, _, c, u in DEFECTS], ids=[d[0] for d in DEFECTS])
def test_messages_of_single_and_first_defects(st, name, create, update):
    f, desc, keep = _defective(name)
    _, _, orders = _create(st, f)
    assert _create(st, f, desc)[0] == (create or "")
    assert _update(st, f, orders, desc)[0] == (update or "")


@pytest.mark.parametrize("name,create", [(n, c) for n, _, c, _ in DEFECTS if c], ids=[d[0] for d in DEFECTS if d[2]])
def test_create_messages_of_the_library(ert, name, create):
    """ert_scene_create checks the descriptor before it looks for a device: the same messages, with or without one."""
    f, desc, keep = _defective(name)
    h = ctypes.c_void_p()
    rc = _lib.load().ert_scene_create(ctypes.byref(desc) if desc is not False else None, 0, ctypes.byref(h))
    assert rc == _lib.ERT_ERR_BADARG and not h.value
    assert _lib.load().ert_last_error().decode() == create


@pytest.mark.gpu
def test_update_messages_of_the_library(gpu):
    """ert_scene_update of a scene made from the mixed scene returns the shim's messages and keeps the scene."""
    f = _mixed()
    dev = f.upload(0)
    for name, _, _, update in DEFECTS:
        if not update:
            continue
        _, desc, keep = _defective(name)
        rc = _lib.load().ert_scene_update(dev.handle, ctypes.byref(desc) if desc is not False else None, 0, None)
        assert rc == _lib.ERT_ERR_BADARG, name
        assert _lib.load().ert_last_error().decode() == update, name
    info = f.update(dev)
    assert info["changed"] == [], info
    dev.close()
