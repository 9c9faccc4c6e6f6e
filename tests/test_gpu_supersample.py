"""Supersampled frames (ert_render_params.supersample, DESIGN.md "Supersampling") held bit for bit to their
definition: sample k = j*N + i of pixel (X, Y) is pixel (N*X + i, N*Y + j) of the (N*W) x (N*H) frame of the same
scene, camera, depth and accel, and the pixel is acc / (N*N) with acc summed in sample order.  The reference frame
of every check is that fold of the library's own N x frame, written out as an explicit loop in sample order; the
oracle check folds the C oracle's frame instead."""
import numpy as np
import pytest

from eraytracer_b200 import _lib, raytracer
from eraytracer_b200 import scene as sc
from erl_scenes import stress_scene
from helpers import assert_double_parity, clustered_scene, oracle_frame

ACCELS = ["exact", "linear", "bvh", "bvh_mega", "grid", "auto"]
SCENES = {
    "demo": lambda: sc.flatten(sc.demo_scene()),
    "c3_1200": lambda: sc.synthetic_scene("c3", n_spheres=1200),
    "clustered": lambda: clustered_scene()[0],
    "m3_300": lambda: sc.mesh_scene("m3", n_triangles=300),
    "stress": lambda: sc.flatten(stress_scene()),
}
# counters that depend on which rays are traced, not on how the launches group them
RAY_COUNTS = ("rays", "bounce_path_rays", "bounce_hits")


def fold(big, n):
    """acc = c_0, acc = acc + c_k for k = 1 .. n*n-1 (sample k = j*n + i at rows n*Y + j, columns n*X + i), then
    acc / (n*n): one IEEE operation per channel and step, in sample order."""
    acc = big[0::n, 0::n].copy()
    for k in range(1, n * n):
        j, i = divmod(k, n)
        acc = acc + big[j::n, i::n]
    return acc / float(n * n)


def in_format(v, fmt):
    """The output formats of include/ert_b200.h applied to an F64 frame."""
    if fmt == "f64":
        return v
    if fmt == "f32":
        return v.astype(np.float32)
    q = np.maximum(np.minimum(np.trunc(v * 255.0), 255.0), 0.0)
    return q.astype(np.uint8)


def folded(dev, w, h, depth, n, accel="auto", camera=None):
    big, st = dev.render(n * w, n * h, depth, fmt="f64", accel=accel, camera=camera)
    return fold(big, n), st


@pytest.fixture(scope="module")
def scenes(gpu):
    made = {}

    def get(name):
        if name not in made:
            made[name] = SCENES[name]().upload(0)
        return made[name]
    yield get
    for d in made.values():
        d.close()


def assert_box_filter(dev, w, h, depth, n, accel):
    ref, big_st = folded(dev, w, h, depth, n, accel)
    for fmt in ("f64", "f32", "rgb8"):
        got, st = dev.render(w, h, depth, fmt=fmt, accel=accel, supersample=n)
        want = in_format(ref, fmt)
        assert got.dtype == want.dtype
        assert np.array_equal(got, want), (fmt, depth, n, accel, int((got != want).sum()))
        assert st["accel_used"] == big_st["accel_used"]
        assert st["pixels"] == w * h
        for key in RAY_COUNTS:
            assert st[key] == big_st[key], (key, fmt, depth, n, accel)


@pytest.mark.gpu
@pytest.mark.parametrize("accel", ACCELS)
@pytest.mark.parametrize("scene", list(SCENES))
def test_supersampled_frame_is_the_fold_of_the_larger_frame(scenes, scene, accel):
    dev = scenes(scene)
    for depth in (0, 1, 5):
        for n in (2, 3, 4):
            assert_box_filter(dev, 37, 23, depth, n, accel)           # not whole 8x4 tiles, nor 32x8 blocks
    assert_box_filter(dev, 13, 7, 5, 8, accel)


@pytest.mark.gpu
@pytest.mark.parametrize("accel", ACCELS)
@pytest.mark.parametrize("scene", ["demo", "clustered", "m3_300"])
def test_one_sample_is_todays_frame(scenes, scene, accel):
    dev = scenes(scene)
    for flags in (0, _lib.FLAG_COUNT_TESTS):
        for fmt in ("f64", "rgb8"):
            plain, st0 = dev.render(45, 29, 5, fmt=fmt, accel=accel, flags=flags)
            for n in (0, 1):
                got, st = dev.render(45, 29, 5, fmt=fmt, accel=accel, flags=flags, supersample=n)
                assert got.tobytes() == plain.tobytes()
                for key, v in st0.items():
                    if not key.endswith("_ms"):
                        assert st[key] == v, (key, n, fmt, flags)


@pytest.mark.gpu
def test_counts_sum_over_the_samples(scenes):
    dev = scenes("c3_1200")
    for accel in ("bvh", "grid", "linear"):
        _, big = dev.render(3 * 40, 3 * 24, 5, fmt="rgb8", accel=accel, flags=_lib.FLAG_COUNT_TESTS)
        _, st = dev.render(40, 24, 5, fmt="rgb8", accel=accel, flags=_lib.FLAG_COUNT_TESTS, supersample=3)
        assert st["pixels"] == 40 * 24
        assert st["bounce_path_rays"][0] == st["pixels"] * 9 == big["pixels"]
        for key in RAY_COUNTS + ("bounces_recorded", "accel_used"):
            assert st[key] == big[key], key
        # the passes' launches, each pass's fold and the resolve
        _, one = dev.render(40, 24, 5, fmt="rgb8", accel=accel)
        _, nine = dev.render(40, 24, 5, fmt="rgb8", accel=accel, supersample=3)
        assert nine["gpu_launches"] == 9 * one["gpu_launches"] + 8
        _, timed = dev.render(40, 24, 5, fmt="rgb8", accel=accel, flags=_lib.FLAG_TIME_KERNELS, supersample=3)
        _, timed1 = dev.render(40, 24, 5, fmt="rgb8", accel=accel, flags=_lib.FLAG_TIME_KERNELS)
        assert timed["path_launches"] == 9 * timed1["path_launches"]
        assert timed["shadow_launches"] == 9 * timed1["shadow_launches"]
        assert timed["path_ms"] > 0 and timed["shadow_ms"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["demo", "c3_200"])
def test_oracle_fold_matches_the_supersampled_frame(gpu, scene):
    flat = sc.flatten(sc.demo_scene()) if scene == "demo" else sc.synthetic_scene("c3", n_spheres=200)
    ref, _, _ = oracle_frame(flat, 3 * 48, 3 * 27, 5)
    want = fold(ref, 3)
    dev = flat.upload(0)
    try:
        got, _ = dev.render(48, 27, 5, fmt="f64", supersample=3)
        assert_double_parity(got, want)
        got8, _ = dev.render(48, 27, 5, fmt="rgb8", supersample=3)
        assert np.array_equal(got8, in_format(want, "rgb8"))
    finally:
        dev.close()


@pytest.mark.gpu
def test_parts_assemble_the_supersampled_frame(scenes):
    dev = scenes("c3_1200")
    for fmt in ("rgb8", "f64"):
        whole, _ = dev.render(50, 31, 5, fmt=fmt, supersample=3)
        out = np.zeros_like(whole)
        for part in range(3):
            _, st = dev.render(50, 31, 5, fmt=fmt, supersample=3, band_rows=5, n_parts=3, part=part, out=out)
            rows = [y for y in range(31) if (y // 5) % 3 == part]
            assert st["pixels"] == 50 * len(rows)
        assert np.array_equal(out, whole)


@pytest.mark.gpu
def test_multi_gpu_supersampled_frame_equals_one_gpu(gpu):
    if gpu < 2:
        pytest.skip("needs two devices")
    flat = sc.synthetic_scene("c3", n_spheres=1200)
    one, _ = raytracer.render_frame(96, 54, flat, 5, fmt="f64", supersample=2)
    many, _ = raytracer.render_frame_multi_gpu(96, 54, flat, 5, fmt="f64", supersample=2)
    assert np.array_equal(one, many)


@pytest.mark.gpu
def test_slots_download_and_camera(scenes):
    dev = scenes("clustered")
    w, h = 41, 26
    want_a, _ = dev.render(w, h, 5, fmt="rgb8", supersample=2)
    want_b, _ = dev.render(w, h, 5, fmt="f64", supersample=3)
    pa = _lib.PinnedFrame(w * h * 3)
    pb = _lib.PinnedFrame(w * h * 3 * 8)
    try:
        dev.render_async(w, h, 5, slot=1, fmt="rgb8", supersample=2, host_ptr=pa.ptr, host_bytes=pa.nbytes)
        dev.render_async(w, h, 5, slot=2, fmt="f64", supersample=3, host_ptr=pb.ptr, host_bytes=pb.nbytes)
        dev.wait(1)
        dev.wait(2)
        assert np.array_equal(pa.array(np.uint8, (h, w, 3)), want_a)
        assert np.array_equal(pb.array(np.float64, (h, w, 3)), want_b)
    finally:
        pa.close()
        pb.close()
    # a slot kept on the device, then downloaded
    dev.render_async(w, h, 5, slot=3, fmt="f64", supersample=3)
    out = np.zeros((h, w, 3), dtype=np.float64)
    _lib.check(_lib.load().ert_download(dev.handle, 3, out.ctypes.data, out.nbytes))
    assert np.array_equal(out, want_b)
    # a per-call camera
    cam = sc.pose_camera(5)
    ref, _ = folded(dev, w, h, 5, 2, camera=cam)
    got, _ = dev.render(w, h, 5, fmt="f64", supersample=2, camera=cam)
    assert np.array_equal(got, ref)


@pytest.mark.gpu
def test_bad_sample_counts_are_rejected(scenes):
    dev = scenes("demo")
    for n in (-1, 9):
        with pytest.raises(_lib.BadArg):
            dev.render(16, 8, 2, supersample=n)
    with pytest.raises(_lib.BadArg):
        dev.render_async(2 ** 30, 1, 1, slot=0, supersample=2)          # 2^31 sample columns
    with pytest.raises(_lib.BadArg):
        dev.render_async(1, 2 ** 29, 1, slot=0, supersample=4)          # 2^31 sample rows
    assert_box_filter(dev, 16, 8, 2, 2, "auto")


@pytest.mark.gpu
def test_full_size_c3(gpu):
    dev = sc.synthetic_scene("c3").upload(0)
    try:
        ref, big = folded(dev, 3840, 2160, 5, 2)
        got, st = dev.render(3840, 2160, 5, fmt="f64", accel="auto", supersample=2)
        assert np.array_equal(got, ref)
        assert st["rays"] == big["rays"] and st["accel_used"] == big["accel_used"]
    finally:
        dev.close()


@pytest.mark.gpu
def test_nif_supersample_option(gpu, tmp_path, monkeypatch):
    import nif_mock
    # a copy of the NIF of its own: the mock keeps its resource types per loaded object, and the NIF tests of
    # this session may have loaded the shared one already
    monkeypatch.setattr(nif_mock, "SO", str(tmp_path / "raytracer_gpu_nif.so"))
    beam = nif_mock.MockBeam()
    Badarg = nif_mock.Badarg
    ok, handle = beam.call("scene_upload", sc.demo_scene(), 0)
    assert ok == "ok"
    dev = sc.flatten(sc.demo_scene()).upload(0)
    try:
        want8, _ = dev.render(40, 30, 5, fmt="rgb8", supersample=2)
        want64, _ = dev.render(40, 30, 5, fmt="f64", supersample=2)
        ok, frame = beam.call("render", handle, 40, 30, 5, [("supersample", 2)])
        assert ok == "ok" and frame == want8.tobytes()
        ok, frame = beam.call("render", handle, 40, 30, 5, [("format", "f64"), ("supersample", 2)])
        assert frame == want64.tobytes()
        ok, frame = beam.call("render", handle, 40, 30, 5, [("supersample", 1)])
        assert frame == dev.render(40, 30, 5, fmt="rgb8")[0].tobytes()
        for bad in (0, 9, "two", 2.0):
            with pytest.raises(Badarg):
                beam.call("render", handle, 40, 30, 5, [("supersample", bad)])
    finally:
        dev.close()
        beam.gc(handle)
