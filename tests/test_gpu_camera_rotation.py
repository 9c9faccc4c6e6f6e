"""Rotated cameras (ERT_FLAG_CAMERA_ROTATION, DESIGN.md "Camera rotation") held bit for bit to the FP64 reference
with the rotation restated in tests/camrot/rot_oracle.c: every accel on the scenes of test_gpu_supersample.py, from
quarter turns, generic angles and look_at poses on every side (above, below the floor plane, inside the sphere field,
behind), at depths 0, 1 and 5.  Identity rotations must give today's frame, and the flag composes with supersampling,
parts, slots, per-call cameras, updates, several GPUs and the NIF."""
import numpy as np
import pytest

import camrot_oracle as cr
from eraytracer_b200 import _lib, raytracer
from eraytracer_b200 import scene as sc
from erl_scenes import stress_scene
from helpers import assert_double_parity, clustered_scene
from test_gpu_supersample import fold, in_format

ACCELS = ["exact", "linear", "bvh", "bvh_mega", "grid", "auto"]
SCENES = {
    "demo": lambda: sc.flatten(sc.demo_scene()),
    "c3_1200": lambda: sc.synthetic_scene("c3", n_spheres=1200),
    "clustered": lambda: clustered_scene()[0],
    "m3_300": lambda: sc.mesh_scene("m3", n_triangles=300),
    "stress": lambda: sc.flatten(stress_scene()),
}
RAY_COUNTS = ("rays", "bounce_path_rays", "bounce_hits")
IDENTITIES = [(0.0, 0.0, 0.0), (360.0, -720.0, 0.0), (180.0, 180.0, 180.0)]
W, H = 40, 24

_flats = {}
_oracle = {}


def flat_of(name):
    if name not in _flats:
        _flats[name] = SCENES[name]()
    return _flats[name]


def camera(base, location=None, rotation=(0.0, 0.0, 0.0)):
    cam = _lib.Camera()
    cam.location[:] = tuple(base.location) if location is None else location
    cam.rotation[:] = rotation
    cam.fov, cam.screen_width, cam.screen_height = base.fov, base.screen_width, base.screen_height
    return cam


def centre_of(flat):
    if len(flat.spheres):
        c = flat.spheres['center']
        return tuple(float(x) for x in (c.min(axis=0) + c.max(axis=0)) / 2.0)
    return (0.0, 0.0, 10.0)


def poses(flat):
    """(label, camera) pairs: quarter turns and generic angles at the scene's camera, then look_at poses."""
    base = flat.camera
    cx, cy, cz = centre_of(flat)
    out = [("q%s" % (r,), camera(base, rotation=r)) for r in
           [(0.0, 90.0, 0.0), (90.0, 0.0, 0.0), (0.0, 180.0, 0.0), (-90.0, 270.0, 90.0)]]
    out += [("g%s" % (r,), camera(base, rotation=r)) for r in [(-30.0, 200.0, 15.0), (12.5, -47.0, 33.0)]]
    spots = {"above": (cx + 1.0, cy - 60.0, cz - 3.0), "below_floor": (cx - 2.0, 9.0, cz - 10.0),
             "inside": (cx + 3.0, cy + 1.5, cz - 4.0), "behind": (cx, cy - 4.0, cz + 70.0), "side": (cx - 70.0, cy, cz)}
    for label, loc in spots.items():
        out.append((label, camera(base, location=loc, rotation=sc.look_at(loc, (cx, cy, cz)))))
    return out


def zero_reflectivity(flat):
    """A hit with reflectivity 0 ends the path on the GPU (0 * child adds nothing), so such scenes trace fewer rays
    than the reference, with the same colours (test_gpu_edges.check_scene)."""
    return any(len(t) and (t['material']['reflectivity'] == 0).any()
               for t in (flat.spheres, flat.triangles, flat.planes))


def oracle(name, label, cam, depth, w=W, h=H):
    key = (name, label, depth, w, h)
    if key not in _oracle:
        _oracle[key] = cr.oracle_frame(flat_of(name), w, h, depth, camera=cam)
    return _oracle[key]


@pytest.fixture(scope="module")
def scenes(gpu):
    made = {}

    def get(name):
        if name not in made:
            made[name] = flat_of(name).upload(0)
        return made[name]
    yield get
    for d in made.values():
        d.close()


@pytest.mark.gpu
@pytest.mark.parametrize("accel", ACCELS)
@pytest.mark.parametrize("scene", list(SCENES))
def test_identity_rotations_are_todays_frame(scenes, scene, accel):
    dev = scenes(scene)
    for rot in IDENTITIES:
        cam = camera(flat_of(scene).camera, rotation=rot)
        for fmt in ("f64", "rgb8"):
            plain, st0 = dev.render(W, H, 5, fmt=fmt, accel=accel, camera=cam)
            got, st = dev.render(W, H, 5, fmt=fmt, accel=accel, camera=cam, camera_rotation=True)
            assert got.tobytes() == plain.tobytes(), (rot, fmt)
            for key, v in st0.items():
                if not key.endswith("_ms"):
                    assert st[key] == v, (key, rot, fmt)


@pytest.mark.gpu
@pytest.mark.parametrize("accel", ACCELS)
@pytest.mark.parametrize("scene", list(SCENES))
def test_rotated_frames_match_the_oracle(scenes, scene, accel):
    dev = scenes(scene)
    for label, cam in poses(flat_of(scene)):
        for depth in (0, 1, 5):
            want, want_rays = oracle(scene, label, cam, depth)
            got, st = dev.render(W, H, depth, fmt="f64", accel=accel, camera=cam, camera_rotation=True)
            assert_double_parity(got, want)
            if zero_reflectivity(flat_of(scene)):
                assert st["rays"] <= want_rays, (label, depth, st["rays"], want_rays)
            else:
                assert st["rays"] == want_rays, (label, depth, st["rays"], want_rays)
            got8, _ = dev.render(W, H, depth, fmt="rgb8", accel=accel, camera=cam, camera_rotation=True)
            assert np.array_equal(got8, in_format(want, "rgb8")), (label, depth)
            ref, st_ref = dev.render(W, H, depth, fmt="f64", accel="exact", camera=cam, camera_rotation=True)
            assert got.tobytes() == ref.tobytes(), (label, depth)
            assert st["rays"] == st_ref["rays"], (label, depth)
            if depth == 5:
                cnt, st_c = dev.render(W, H, depth, fmt="f64", accel=accel, camera=cam, camera_rotation=True,
                                       flags=_lib.FLAG_COUNT_TESTS)
                assert cnt.tobytes() == got.tobytes() and st_c["rays"] == st["rays"], label


@pytest.mark.gpu
def test_rotation_is_read_only_with_the_flag(scenes):
    dev = scenes("c3_1200")
    base = flat_of("c3_1200").camera
    plain, _ = dev.render(W, H, 5, fmt="f64", camera=camera(base))
    turned = camera(base, rotation=(10.0, 20.0, 30.0))
    assert dev.render(W, H, 5, fmt="f64", camera=turned)[0].tobytes() == plain.tobytes()
    assert dev.render(W, H, 5, fmt="f64", camera=turned, camera_rotation=True)[0].tobytes() != plain.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["demo", "clustered", "m3_300"])
def test_supersampled_rotated_frame_is_the_fold(scenes, scene):
    dev = scenes(scene)
    flat = flat_of(scene)
    for label, cam in poses(flat)[::3]:
        for accel in ("auto", "bvh", "exact"):
            big, big_st = dev.render(2 * 21, 2 * 13, 5, fmt="f64", accel=accel, camera=cam, camera_rotation=True)
            want = fold(big, 2)
            for fmt in ("f64", "rgb8"):
                got, st = dev.render(21, 13, 5, fmt=fmt, accel=accel, camera=cam, camera_rotation=True, supersample=2)
                assert np.array_equal(got, in_format(want, fmt)), (label, accel, fmt)
                for key in RAY_COUNTS:
                    assert st[key] == big_st[key], (key, label, accel)
    # and the fold of the oracle's rotated 3x frame
    label, cam = poses(flat)[-1]
    ref, _ = cr.oracle_frame(flat, 3 * 16, 3 * 9, 5, camera=cam)
    got, _ = dev.render(16, 9, 5, fmt="f64", camera=cam, camera_rotation=True, supersample=3)
    assert_double_parity(got, fold(ref, 3))


@pytest.mark.gpu
def test_parts_slots_and_cameras(scenes):
    dev = scenes("c3_1200")
    flat = flat_of("c3_1200")
    _, cam = poses(flat)[6]                     # from above
    for fmt in ("rgb8", "f64"):
        whole, _ = dev.render(50, 31, 5, fmt=fmt, camera=cam, camera_rotation=True)
        out = np.zeros_like(whole)
        for part in range(3):
            dev.render(50, 31, 5, fmt=fmt, camera=cam, camera_rotation=True, band_rows=5, n_parts=3, part=part,
                       out=out)
        assert np.array_equal(out, whole)
    # slots, pinned frames and ert_download
    w, h = 41, 26
    cams = [c for _, c in poses(flat)[4:8]]
    wants = [dev.render(w, h, 5, fmt="f64", camera=c, camera_rotation=True)[0] for c in cams]
    pinned = [_lib.PinnedFrame(w * h * 3 * 8) for _ in range(3)]
    try:
        for slot in range(3):
            dev.render_async(w, h, 5, slot=slot, fmt="f64", camera=cams[slot], camera_rotation=True,
                             host_ptr=pinned[slot].ptr, host_bytes=pinned[slot].nbytes)
        dev.render_async(w, h, 5, slot=3, fmt="f64", camera=cams[3], camera_rotation=True)
        for slot in range(3):
            dev.wait(slot)
            assert np.array_equal(pinned[slot].array(np.float64, (h, w, 3)), wants[slot]), slot
        out = np.zeros((h, w, 3))
        _lib.check(_lib.load().ert_download(dev.handle, 3, out.ctypes.data, out.nbytes))
        assert np.array_equal(out, wants[3])
    finally:
        for p in pinned:
            p.close()
    # a per-call camera's rotation overrides the stored one; without a per-call camera the stored one is turned
    stored = _lib.Camera.from_buffer_copy(cams[0])
    moved = sc.FlatScene(stored, flat.lights, flat.spheres, flat.triangles, flat.planes)
    dev2 = moved.upload(0)
    try:
        got, _ = dev2.render(w, h, 5, fmt="f64", camera_rotation=True)
        assert np.array_equal(got, wants[0])
        got, _ = dev2.render(w, h, 5, fmt="f64", camera=cams[1], camera_rotation=True)
        assert np.array_equal(got, wants[1])
    finally:
        dev2.close()


@pytest.mark.gpu
def test_multi_gpu_rotated_frame_equals_one_gpu(gpu):
    flat = sc.synthetic_scene("c3", n_spheres=1200)
    loc = (30.0, -25.0, 10.0)
    flat.camera.location[:] = loc
    flat.camera.rotation[:] = sc.look_at(loc, centre_of(flat))
    one, _ = raytracer.render_frame(96, 54, flat, 5, fmt="f64", camera_rotation=True)
    many, _ = raytracer.render_frame_multi_gpu(96, 54, flat, 5, fmt="f64", camera_rotation=True, band_rows=4)
    assert np.array_equal(one, many)
    ref, _ = cr.oracle_frame(flat, 96, 54, 5)
    assert_double_parity(one, ref)


@pytest.mark.gpu
def test_update_of_the_rotation_only(gpu):
    a = sc.synthetic_scene("c3", n_spheres=1200)
    dev = a.upload(0)
    try:
        for rot in [(0.0, 90.0, 0.0), (-20.0, 35.0, 5.0), (0.0, 0.0, 0.0)]:
            b = sc.synthetic_scene("c3", n_spheres=1200)
            b.camera.rotation[:] = rot
            info = b.update(dev)
            assert info["changed"] == ["camera"], (rot, info)
            fresh = b.upload(0)
            try:
                for accel in ("auto", "bvh", "linear"):
                    got, _ = dev.render(W, H, 5, fmt="f64", accel=accel, camera_rotation=True)
                    want, _ = fresh.render(W, H, 5, fmt="f64", accel=accel, camera_rotation=True)
                    assert got.tobytes() == want.tobytes(), (rot, accel)
            finally:
                fresh.close()
    finally:
        dev.close()


@pytest.mark.gpu
def test_non_finite_rotation_is_badarg_only_with_the_flag(scenes):
    dev = scenes("demo")
    base = flat_of("demo").camera
    plain, _ = dev.render(16, 8, 2, fmt="f64", camera=camera(base))
    for bad in [(float("nan"), 0.0, 0.0), (0.0, float("inf"), 0.0), (0.0, 0.0, float("-inf"))]:
        cam = camera(base, rotation=bad)
        with pytest.raises(_lib.BadArg, match="camera rotation has a non-finite field"):
            dev.render(16, 8, 2, camera=cam, camera_rotation=True)
        with pytest.raises(_lib.BadArg):
            dev.render_async(16, 8, 2, slot=1, camera=cam, camera_rotation=True)
        got, _ = dev.render(16, 8, 2, fmt="f64", camera=cam)
        assert got.tobytes() == plain.tobytes()
        # a stored non-finite rotation: accepted at create, refused only when a render reads it
        flat = sc.flatten(sc.demo_scene())
        flat.camera.rotation[:] = bad
        d2 = flat.upload(0)
        try:
            assert d2.render(16, 8, 2, fmt="f64")[0].tobytes() == plain.tobytes()
            with pytest.raises(_lib.BadArg):
                d2.render(16, 8, 2, camera_rotation=True)
        finally:
            d2.close()
    assert dev.render(16, 8, 2, fmt="f64", camera=camera(base))[0].tobytes() == plain.tobytes()


def _lattice(w, h, nx, ny):
    xs = np.linspace(0, w - 1, nx).round().astype(np.int32)
    ys = np.linspace(0, h - 1, ny).round().astype(np.int32)
    X, Y = np.meshgrid(xs, ys)
    return X.ravel(), Y.ravel()


@pytest.mark.gpu
def test_full_size_c3_from_four_poses(gpu):
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    cx, cy, cz = centre_of(flat)
    try:
        for loc in [(0.0, -70.0, 40.0), (90.0, -10.0, 45.0), (-20.0, -5.0, 140.0), (5.0, -12.0, 30.0)]:
            cam = camera(flat.camera, location=loc, rotation=sc.look_at(loc, (cx, cy, cz)))
            frame, st = dev.render(3840, 2160, 5, fmt="f64", accel="auto", camera=cam, camera_rotation=True)
            assert st["accel_used"] == "grid" and st["has_cell_grid"] == 1, (loc, st["accel_used"])
            y0, x0 = 1048, 1888
            X, Y = np.meshgrid(np.arange(x0, x0 + 64, dtype=np.int32), np.arange(y0, y0 + 64, dtype=np.int32))
            for xs, ys in ((X.ravel(), Y.ravel()), _lattice(3840, 2160, 48, 27)):
                want, _ = cr.oracle_frame(flat, 3840, 2160, 5, camera=cam, pixels=(xs, ys))
                assert_double_parity(frame[ys, xs], want)
    finally:
        dev.close()


@pytest.mark.gpu
def test_full_size_c4_orbit_pose(gpu):
    flat = sc.synthetic_scene("c4")
    dev = flat.upload(0)
    try:
        cx, cy, cz = centre_of(flat)
        loc = (cx + 300.0, cy - 150.0, cz - 200.0)
        cam = camera(flat.camera, location=loc, rotation=sc.look_at(loc, (cx, cy, cz)))
        grid, st = dev.render(3840, 2160, 5, fmt="f64", accel="grid", camera=cam, camera_rotation=True)
        bvh, st_b = dev.render(3840, 2160, 5, fmt="f64", accel="bvh", camera=cam, camera_rotation=True)
        assert grid.tobytes() == bvh.tobytes() and st["rays"] == st_b["rays"]
        xs, ys = _lattice(3840, 2160, 32, 32)
        want, _ = cr.oracle_frame(flat, 3840, 2160, 5, camera=cam, pixels=(xs, ys))
        assert_double_parity(grid[ys, xs], want)
    finally:
        dev.close()


@pytest.mark.gpu
def test_nif_camera_rotation_option(gpu, tmp_path, monkeypatch):
    import nif_mock
    monkeypatch.setattr(nif_mock, "SO", str(tmp_path / "raytracer_gpu_nif.so"))
    beam = nif_mock.MockBeam()
    demo = sc.demo_scene()
    rot = sc.look_at((6.0, -3.0, -4.0), (-4.5, -2.5, 14.0))
    c0 = demo[0]
    turned = ('camera', ('vector', 6.0, -3.0, -4.0), ('vector',) + rot, c0[3], c0[4])
    scene_list = [turned] + demo[1:]
    ok, handle = beam.call("scene_upload", scene_list, 0)
    assert ok == "ok"
    dev = sc.flatten(scene_list).upload(0)
    try:
        want8, _ = dev.render(40, 30, 5, fmt="rgb8", camera_rotation=True)
        want64, _ = dev.render(40, 30, 5, fmt="f64", camera_rotation=True)
        ok, frame = beam.call("render", handle, 40, 30, 5, [("camera_rotation", True)])
        assert ok == "ok" and frame == want8.tobytes()
        ok, frame = beam.call("render", handle, 40, 30, 5, [("format", "f64"), ("camera_rotation", True)])
        assert frame == want64.tobytes()
        ok, frame = beam.call("render", handle, 40, 30, 5, [("camera_rotation", False)])
        assert frame == dev.render(40, 30, 5, fmt="rgb8")[0].tobytes()
        # a per-call camera through the NIF is turned too
        ok, frame = beam.call("render", handle, 40, 30, 5, [("camera", demo[0]), ("camera_rotation", True)])
        assert frame == dev.render(40, 30, 5, fmt="rgb8", camera=sc.camera_struct(demo[0]))[0].tobytes()
        for bad in (1, "yes", 1.0):
            with pytest.raises(nif_mock.Badarg):
                beam.call("render", handle, 40, 30, 5, [("camera_rotation", bad)])
    finally:
        dev.close()
        beam.gc(handle)
