"""ctypes binding of libert_b200.so (include/ert_b200.h).

There is no CPU fallback: if the shared object is missing this module raises,
and every call that needs a GPU raises ErtError when none is usable.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# ERT_B200_LIB selects another build of the same library (tuning experiments only)
LIB_PATH = os.environ.get("ERT_B200_LIB") or os.path.join(HERE, "lib", "libert_b200.so")

ERT_OK, ERT_ERR_BADARG, ERT_ERR_NO_DEVICE, ERT_ERR_CUDA, ERT_ERR_NOMEM = 0, 1, 2, 3, 4
FMT_RGB8, FMT_F32, FMT_F64 = 0, 1, 2
ACCEL_AUTO, ACCEL_EXACT, ACCEL_LINEAR, ACCEL_BVH, ACCEL_BVH_MEGAKERNEL, ACCEL_GRID, ACCEL_WARP = 0, 1, 2, 3, 4, 5, 6
FLAG_COUNT_TESTS = 1
FLAG_WF_UNSORTED = 2
FLAG_NO_LIGHT_GRID = 4
FLAG_TIME_KERNELS = 8
MAX_SLOTS = 4
UPDATE_REBUILD_GRIDS = 1
UPDATE_REBUILD = 2
# ert_update_info.changed / .done bits (include/ert_b200.h)
UPDATE_CHANGED = ["camera", "lights", "light_pos", "spheres", "sphere_mat", "triangles", "triangle_mat", "planes"]
UPDATE_DONE = ["refit_spheres", "refit_triangles", "drop_cell_grid", "drop_light_grids", "rebuild_cell_grid",
               "rebuild_light_grids", "rebuild_tri_bvh", "rebuild"]

FORMATS = {"rgb8": FMT_RGB8, "f32": FMT_F32, "f64": FMT_F64}
FORMAT_DTYPES = {FMT_RGB8: np.uint8, FMT_F32: np.float32, FMT_F64: np.float64}
ACCELS = {"auto": ACCEL_AUTO, "exact": ACCEL_EXACT, "linear": ACCEL_LINEAR, "bvh": ACCEL_BVH,
          "bvh_mega": ACCEL_BVH_MEGAKERNEL, "grid": ACCEL_GRID, "warp": ACCEL_WARP}
ACCEL_NAMES = {v: k for k, v in ACCELS.items()}


class ErtError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("ert_b200 error %d: %s" % (code, message))
        self.code = code


class BadArg(ErtError, ValueError):
    """ERT_ERR_BADARG — what the NIF turns into `badarg`."""


class Camera(ctypes.Structure):
    _fields_ = [("location", ctypes.c_double * 3), ("rotation", ctypes.c_double * 3),
                ("fov", ctypes.c_double), ("screen_width", ctypes.c_double),
                ("screen_height", ctypes.c_double)]


class SceneDesc(ctypes.Structure):
    _fields_ = [("camera", Camera),
                ("n_lights", ctypes.c_int64), ("lights", ctypes.c_void_p),
                ("n_spheres", ctypes.c_int64), ("spheres", ctypes.c_void_p),
                ("n_triangles", ctypes.c_int64), ("triangles", ctypes.c_void_p),
                ("n_planes", ctypes.c_int64), ("planes", ctypes.c_void_p)]


class RenderParams(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int32), ("height", ctypes.c_int32), ("depth", ctypes.c_int32),
                ("format", ctypes.c_int32), ("accel", ctypes.c_int32), ("band_rows", ctypes.c_int32),
                ("n_parts", ctypes.c_int32), ("part", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("reserved", ctypes.c_int32), ("camera", ctypes.POINTER(Camera))]


class Stats(ctypes.Structure):
    _fields_ = [("kernel_ms", ctypes.c_double), ("total_ms", ctypes.c_double),
                ("rays", ctypes.c_uint64), ("pixels", ctypes.c_uint64),
                ("gpu_launches", ctypes.c_uint64), ("d2h_bytes", ctypes.c_uint64),
                ("h2d_bytes", ctypes.c_uint64), ("sphere_filter_tests", ctypes.c_uint64),
                ("box_tests", ctypes.c_uint64), ("exact_sphere_tests", ctypes.c_uint64),
                ("exact_other_tests", ctypes.c_uint64), ("accel_used", ctypes.c_int32),
                ("reserved", ctypes.c_int32),
                ("path_box_tests", ctypes.c_uint64), ("path_filter_tests", ctypes.c_uint64),
                ("shadow_box_tests", ctypes.c_uint64), ("shadow_filter_tests", ctypes.c_uint64),
                ("path_ms", ctypes.c_double), ("shadow_ms", ctypes.c_double), ("other_ms", ctypes.c_double),
                ("path_launches", ctypes.c_uint64), ("shadow_launches", ctypes.c_uint64),
                ("cell_steps", ctypes.c_uint64), ("has_cell_grid", ctypes.c_int32),
                ("bounces_recorded", ctypes.c_int32),
                ("bounce_path_rays", ctypes.c_uint64 * 16), ("bounce_hits", ctypes.c_uint64 * 16)]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if not n.startswith("reserved")}
        nb = d["bounces_recorded"]
        d["bounce_path_rays"] = [int(v) for v in self.bounce_path_rays[:nb]]
        d["bounce_hits"] = [int(v) for v in self.bounce_hits[:nb]]
        return d


class UpdateInfo(ctypes.Structure):
    _fields_ = [("changed", ctypes.c_uint32), ("done", ctypes.c_uint32), ("has_cell_grid", ctypes.c_int32),
                ("light_grids", ctypes.c_int32), ("light_grids_rebuilt", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("h2d_bytes", ctypes.c_uint64), ("host_ms", ctypes.c_double), ("device_ms", ctypes.c_double),
                ("sphere_area_ratio", ctypes.c_double), ("triangle_area_ratio", ctypes.c_double)]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}
        d["changed"] = [n for k, n in enumerate(UPDATE_CHANGED) if self.changed >> k & 1]
        d["done"] = [n for k, n in enumerate(UPDATE_DONE) if self.done >> k & 1]
        return d


# numpy views of the element records (same layout as the C structs)
MATERIAL_DT = np.dtype([("colour", "<f8", 3), ("specular_power", "<f8"), ("shininess", "<f8"),
                        ("reflectivity", "<f8")])
LIGHT_DT = np.dtype([("diffuse_colour", "<f8", 3), ("location", "<f8", 3),
                     ("specular_colour", "<f8", 3), ("order", "<i4"), ("reserved", "<i4")])
SPHERE_DT = np.dtype([("radius", "<f8"), ("center", "<f8", 3), ("material", MATERIAL_DT),
                      ("order", "<i4"), ("reserved", "<i4")])
TRIANGLE_DT = np.dtype([("v1", "<f8", 3), ("v2", "<f8", 3), ("v3", "<f8", 3),
                        ("material", MATERIAL_DT), ("order", "<i4"), ("reserved", "<i4")])
PLANE_DT = np.dtype([("normal", "<f8", 3), ("distance", "<f8"), ("material", MATERIAL_DT),
                     ("order", "<i4"), ("reserved", "<i4")])
assert MATERIAL_DT.itemsize == 48 and LIGHT_DT.itemsize == 80 and SPHERE_DT.itemsize == 88
assert TRIANGLE_DT.itemsize == 128 and PLANE_DT.itemsize == 88

EXPORTS = [
    "ert_abi_version", "ert_last_error", "ert_device_count", "ert_scene_create", "ert_scene_clone",
    "ert_scene_destroy", "ert_render", "ert_render_async", "ert_wait", "ert_download",
    "ert_get_stats", "ert_trace_rays", "ert_host_alloc", "ert_host_free", "ert_host_register",
    "ert_host_unregister", "ert_fp32_peak", "ert_fp32_peak_rrr", "ert_fp64_peak", "ert_d2h_peak", "ert_l2_flush",
    "ert_scene_update",
]

_lib = None


def load():
    """Loads the shared object; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `make -C eraytracer_b200/csrc` "
            "(or __graft_entry__.build()); eraytracer_b200 has no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp = ctypes.c_void_p
    L.ert_abi_version.restype = ctypes.c_int
    L.ert_last_error.restype = ctypes.c_char_p
    L.ert_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
    L.ert_scene_create.argtypes = [ctypes.POINTER(SceneDesc), ctypes.c_int, ctypes.POINTER(vp)]
    L.ert_scene_clone.argtypes = [vp, ctypes.c_int, ctypes.POINTER(vp)]
    L.ert_scene_destroy.argtypes = [vp]
    L.ert_scene_update.argtypes = [vp, ctypes.POINTER(SceneDesc), ctypes.c_uint32, ctypes.POINTER(UpdateInfo)]
    L.ert_render.argtypes = [vp, ctypes.POINTER(RenderParams), vp, ctypes.c_size_t]
    L.ert_render_async.argtypes = [vp, ctypes.POINTER(RenderParams), ctypes.c_int, vp,
                                   ctypes.c_size_t]
    L.ert_wait.argtypes = [vp, ctypes.c_int]
    L.ert_download.argtypes = [vp, ctypes.c_int, vp, ctypes.c_size_t]
    L.ert_get_stats.argtypes = [vp, ctypes.c_int, ctypes.POINTER(Stats)]
    L.ert_trace_rays.argtypes = [vp, ctypes.c_int64, vp, ctypes.c_int, vp, vp]
    L.ert_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp)]
    L.ert_host_free.argtypes = [vp]
    L.ert_host_register.argtypes = [vp, ctypes.c_size_t]
    L.ert_host_unregister.argtypes = [vp]
    L.ert_fp32_peak.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    L.ert_fp32_peak_rrr.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    L.ert_fp64_peak.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    L.ert_d2h_peak.argtypes = [ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(ctypes.c_double)]
    L.ert_l2_flush.argtypes = [ctypes.c_int]
    for name in EXPORTS:
        if name not in ("ert_last_error",):
            getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc == ERT_OK:
        return
    msg = load().ert_last_error().decode("utf-8", "replace")
    if rc == ERT_ERR_BADARG:
        raise BadArg(rc, msg)
    raise ErtError(rc, msg)


def device_count():
    n = ctypes.c_int(0)
    check(load().ert_device_count(ctypes.byref(n)))
    return n.value


class PinnedFrame:
    """A pinned host buffer exposed as a numpy array (freed on close())."""

    def __init__(self, nbytes):
        self.ptr = ctypes.c_void_p()
        check(load().ert_host_alloc(nbytes, ctypes.byref(self.ptr)))
        self.nbytes = nbytes
        self._buf = (ctypes.c_uint8 * nbytes).from_address(self.ptr.value)

    def array(self, dtype, shape):
        return np.frombuffer(self._buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if self.ptr:
            self._buf = None
            load().ert_host_free(self.ptr)
            self.ptr = None


class Scene:
    """Device-resident scene (ert_scene*)."""

    def __init__(self, handle, device, tables=None):
        self.handle = handle
        self.device = device
        self._tables = tables        # keeps the numpy tables alive during create

    @staticmethod
    def _desc(camera, lights, spheres, triangles, planes):
        """(SceneDesc, the contiguous tables it points into: keep them alive for the call)."""
        desc = SceneDesc()
        desc.camera = camera
        tabs = []
        for name, arr, dt in (("lights", lights, LIGHT_DT), ("spheres", spheres, SPHERE_DT),
                              ("triangles", triangles, TRIANGLE_DT), ("planes", planes, PLANE_DT)):
            arr = np.ascontiguousarray(arr, dtype=dt)
            tabs.append(arr)
            setattr(desc, "n_" + name, len(arr))
            setattr(desc, name, arr.ctypes.data if len(arr) else None)
        return desc, tabs

    @classmethod
    def create(cls, camera, lights, spheres, triangles, planes, device=0):
        desc, tabs = cls._desc(camera, lights, spheres, triangles, planes)
        h = ctypes.c_void_p()
        check(load().ert_scene_create(ctypes.byref(desc), int(device), ctypes.byref(h)))
        return cls(h, device)

    def update(self, camera, lights, spheres, triangles, planes, rebuild_grids=False, rebuild=False):
        """ert_scene_update: new values for the scene's elements (same counts, same `order` values per kind, tables in
        any order).  rebuild_grids builds stale cell / direction grids again on the device (the grids of a fresh
        create of the same tables); rebuild runs the whole create path in place.  Returns the ert_update_info as a
        dict; raises BadArg (scene untouched) on a shape mismatch, a non-finite value or a duplicate `order`."""
        desc, tabs = self._desc(camera, lights, spheres, triangles, planes)
        flags = (UPDATE_REBUILD_GRIDS if rebuild_grids else 0) | (UPDATE_REBUILD if rebuild else 0)
        info = UpdateInfo()
        check(load().ert_scene_update(self.handle, ctypes.byref(desc), flags, ctypes.byref(info)))
        return info.as_dict()

    def clone(self, device):
        h = ctypes.c_void_p()
        check(load().ert_scene_clone(self.handle, int(device), ctypes.byref(h)))
        return Scene(h, device)

    def close(self):
        if self.handle:
            load().ert_scene_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _params(self, width, height, depth, fmt, accel, band_rows, n_parts, part, flags, camera):
        p = RenderParams()
        p.width, p.height, p.depth = int(width), int(height), int(depth)
        p.format = FORMATS[fmt] if isinstance(fmt, str) else int(fmt)
        p.accel = ACCELS[accel] if isinstance(accel, str) else int(accel)
        p.band_rows, p.n_parts, p.part = int(band_rows), int(n_parts), int(part)
        p.flags = int(flags)
        self._cam_keep = camera
        p.camera = ctypes.pointer(camera) if camera is not None else None
        return p

    def render(self, width, height, depth, fmt="f64", accel="auto", band_rows=0, n_parts=1,
               part=0, flags=0, camera=None, out=None):
        """Synchronous render into a numpy frame (H, W, 3); returns (frame, stats dict)."""
        p = self._params(width, height, depth, fmt, accel, band_rows, n_parts, part, flags, camera)
        if p.width <= 0 or p.height <= 0:
            # let the library produce the error (mirrors the guards at raytracer.erl:89)
            check(load().ert_render(self.handle, ctypes.byref(p), None, 0))
        dt = FORMAT_DTYPES[p.format]
        if out is None:
            out = np.zeros((p.height, p.width, 3), dtype=dt)
        assert out.dtype == dt and out.flags["C_CONTIGUOUS"]
        check(load().ert_render(self.handle, ctypes.byref(p), out.ctypes.data, out.nbytes))
        return out, self.stats(0)

    def render_async(self, width, height, depth, slot=0, fmt="rgb8", accel="auto", band_rows=0,
                     n_parts=1, part=0, flags=0, camera=None, host_ptr=None, host_bytes=0):
        p = self._params(width, height, depth, fmt, accel, band_rows, n_parts, part, flags, camera)
        check(load().ert_render_async(self.handle, ctypes.byref(p), int(slot), host_ptr,
                                      int(host_bytes)))

    def wait(self, slot=0):
        check(load().ert_wait(self.handle, int(slot)))

    def stats(self, slot=0):
        st = Stats()
        check(load().ert_get_stats(self.handle, int(slot), ctypes.byref(st)))
        d = st.as_dict()
        d["accel_used"] = ACCEL_NAMES.get(d["accel_used"], d["accel_used"])
        return d

    def trace_rays(self, rays6, accel="auto"):
        rays6 = np.ascontiguousarray(rays6, dtype=np.float64).reshape(-1, 6)
        n = len(rays6)
        order = np.full(n, -1, dtype=np.int32)
        t = np.zeros(n, dtype=np.float64)
        a = ACCELS[accel] if isinstance(accel, str) else int(accel)
        check(load().ert_trace_rays(self.handle, n, rays6.ctypes.data, a, order.ctypes.data,
                                    t.ctypes.data))
        return order, t


def fp32_peak(device=0):
    v = ctypes.c_double(0)
    check(load().ert_fp32_peak(int(device), ctypes.byref(v)))
    return v.value


def fp32_peak_rrr(device=0):
    v = ctypes.c_double(0)
    check(load().ert_fp32_peak_rrr(int(device), ctypes.byref(v)))
    return v.value


def fp64_peak(device=0):
    v = ctypes.c_double(0)
    check(load().ert_fp64_peak(int(device), ctypes.byref(v)))
    return v.value


def d2h_peak(device=0, nbytes=256 << 20):
    v = ctypes.c_double(0)
    check(load().ert_d2h_peak(int(device), int(nbytes), ctypes.byref(v)))
    return v.value


def l2_flush(device=0):
    check(load().ert_l2_flush(int(device)))
