"""GPU edge cases and properties: everything the reference's semantics make awkward."""
import json
import os

import numpy as np
import pytest

import eraytracer_b200 as ert
from eraytracer_b200 import _lib, multigpu, raytracer
from eraytracer_b200 import scene as sc
from helpers import (assert_double_parity, assert_image_parity, oracle_frame,
                     oracle_scene_from_flat, quantise)
from oracle import orc

pytestmark = pytest.mark.gpu
ACCELS = ("exact", "linear", "bvh", "bvh_mega")
CAM = ('camera', ('vector', 0, 0, -2), ('vector', 0, 0, 0), 90, ('screen', 4, 3))
L1 = ('point_light', ('colour', 1, 1, 0.5), ('vector', 5, -2, 0), ('colour', 1, 1, 1))
L2 = ('point_light', ('colour', 1, 0, 0.5), ('vector', -10, 0, 7), ('colour', 1, 0, 0.5))


def mat(c=(1, 0.5, 0), sp=4, sh=0.25, refl=0.5):
    return ('material', ('colour',) + tuple(c), sp, sh, refl)


def check_scene(scene, w=64, h=48, depth=4, accels=ACCELS, rays_equal=True):
    flat = sc.flatten(scene)
    dev = flat.upload(0)
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    try:
        for accel in accels:
            frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            assert_double_parity(frame, ref)
            assert np.array_equal(quantise(frame), quantise(ref)), accel
            # a zero-reflectivity hit ends the path on the GPU (0 * child adds nothing), so
            # such scenes trace fewer rays than the reference would
            assert st["rays"] == ref_rays if rays_equal else st["rays"] <= ref_rays, accel
    finally:
        dev.close()
    return ref


@pytest.mark.parametrize("accel", ACCELS)
def test_depth_zero_is_black_without_tracing(gpu, accel):
    dev = sc.flatten(sc.demo_scene()).upload(0)
    frame, st = dev.render(16, 12, 0, fmt="f64", accel=accel)
    assert not frame.any() and st["rays"] == 0
    dev.close()


def test_scene_without_lights_is_black(gpu):
    scene = [e for e in sc.demo_scene() if e[0] != 'point_light']
    ref = check_scene(scene, 16, 12, 5)
    assert not ref.any()


def test_camera_only_scene(gpu):
    ref = check_scene([CAM], 8, 8, 3)
    assert not ref.any()


def test_lights_only_scene(gpu):
    check_scene([CAM, L1, L2], 8, 8, 3)


def test_unknown_elements_keep_their_list_positions(gpu):
    scene = sc.demo_scene()
    scene.insert(3, ('fog', 40))
    scene.insert(1, 'an_atom')
    scene.append(('colour', 1, 1, 1))
    a = check_scene(scene, 32, 24, 3)
    b, _, _ = oracle_frame(sc.flatten(sc.demo_scene()), 32, 24, 3)
    assert np.array_equal(a, b)


@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (31, 9), (65, 7), (257, 3)])
def test_odd_image_sizes(gpu, w, h):
    check_scene(sc.demo_scene(), w, h, 3)


def test_bad_arguments_raise_badarg(gpu):
    dev = sc.flatten(sc.demo_scene()).upload(0)
    for w, h, d in ((0, 4, 1), (4, 0, 1), (-3, 4, 1), (4, 4, -1)):
        with pytest.raises(ert.BadArg):
            dev.render(w, h, d, out=np.zeros((1, 1, 3)))
    with pytest.raises(ert.BadArg):
        dev.render(8, 8, 1, band_rows=4, n_parts=2, part=2)
    with pytest.raises(ert.BadArg):
        dev.render(8, 8, 1, out=np.zeros((4, 8, 3)))          # host frame too small
    order, t = dev.trace_rays(np.zeros((0, 6)))
    assert len(order) == 0
    dev.close()
    lights = np.zeros(2, dtype=_lib.LIGHT_DT)                  # duplicate list positions
    with pytest.raises(ert.BadArg):
        _lib.Scene.create(sc.camera_struct(CAM), lights, np.zeros(0, _lib.SPHERE_DT),
                          np.zeros(0, _lib.TRIANGLE_DT), np.zeros(0, _lib.PLANE_DT))
    sp = np.zeros(1, dtype=_lib.SPHERE_DT)
    sp['radius'] = np.nan
    with pytest.raises(ert.BadArg):
        _lib.Scene.create(sc.camera_struct(CAM), np.zeros(0, _lib.LIGHT_DT), sp,
                          np.zeros(0, _lib.TRIANGLE_DT), np.zeros(0, _lib.PLANE_DT))


def test_equal_distance_goes_to_the_earlier_list_element(gpu):
    """Strict '>' at erl:319: two coincident objects, the first one listed is hit."""
    red = ('plane', ('vector', 0, -1, 0), 5, mat((1, 0, 0), 1, 0, 0.2))
    blue = ('plane', ('vector', 0, -1, 0), 5, mat((0, 0, 1), 1, 0, 0.2))
    s_a = ('sphere', 3, ('vector', 0, 0, 9), mat((1, 0, 0)))
    s_b = ('sphere', 3, ('vector', 0, 0, 9), mat((0, 1, 0)))
    a = check_scene([CAM, L1, red, blue, s_a, s_b], 48, 36, 3)
    b = check_scene([CAM, L1, blue, red, s_b, s_a], 48, 36, 3)
    # a later coincident duplicate never wins a scan (primary or shadow): dropping it changes nothing
    assert np.array_equal(a, check_scene([CAM, L1, red, s_a], 48, 36, 3))
    assert np.array_equal(b, check_scene([CAM, L1, blue, s_b], 48, 36, 3))
    assert not np.array_equal(a, b)
    # the demo triangle's edge lies in the floor plane: exact ties between triangle and plane
    check_scene(sc.demo_scene(), 196, 147, 5)


def test_origin_inside_a_sphere_misses_it(gpu):
    """erl:381 wants both roots >= 0: a camera inside a sphere does not see it."""
    big = ('sphere', 50, ('vector', 0, 0, 0), mat((1, 1, 1)))
    small = ('sphere', 2, ('vector', 0, 0, 10), mat((0, 1, 0), 20, 1, 0.3))
    ref = check_scene([CAM, L1, big, small], 48, 36, 3)
    assert ref.any()


def test_unnormalised_plane_normal_and_non_unit_reflection_rays(gpu):
    """erl:476 returns the stored normal as is, so bounce directions leave the unit sphere and
    the 'divide by 2, not 2A' roots (erl:379-380) matter.  All strategies must follow."""
    floor = ('plane', ('vector', 0, -2, 0), 10, mat((1, 1, 1), 1, 0, 0.6))
    wall = ('plane', ('vector', 0.3, 0, -1.7), 40, mat((0.2, 0.4, 1), 4, 0.5, 0.5))
    spheres = [('sphere', 1.5 + 0.1 * i, ('vector', -6 + 3 * i, 2 - 0.5 * i, 8 + i), mat((0.2 * i, 1, 0.5), 20, 1, 0.4))
               for i in range(5)]
    check_scene([CAM, L1, L2, floor, wall] + spheres, 96, 72, 5)


def test_negative_colours_and_byte_clamp(gpu):
    weird = ('sphere', 4, ('vector', 0, 0, 10), mat((-1, 0.5, 2), 2, 0.5, 0.1))
    flat = sc.flatten([CAM, L1, weird])
    dev = flat.upload(0)
    ref, _, _ = oracle_frame(flat, 32, 24, 2)
    f64, _ = dev.render(32, 24, 2, fmt="f64")
    assert_double_parity(f64, ref)
    assert ref.min() < 0
    rgb8, _ = dev.render(32, 24, 2, fmt="rgb8")
    assert np.array_equal(rgb8.astype(np.int64), np.clip(quantise(ref), 0, 255))
    dev.close()


def test_centres_and_radii_that_are_not_float32_values(gpu):
    rng = np.random.default_rng(3)
    spheres = [('sphere', float(rng.uniform(0.3, 1.7)), ('vector', float(rng.uniform(-8, 8)), float(rng.uniform(-6, 4)),
                float(rng.uniform(6, 30))), mat(tuple(rng.uniform(0, 1, 3)), 20, 0.5, float(rng.uniform(0, 0.7))))
               for _ in range(300)]
    floor = ('plane', ('vector', 0, -1, 0), 5, mat((1, 1, 1), 1, 0, 0.1))
    check_scene([CAM, L1, L2] + spheres + [floor], 96, 72, 4)


def test_far_away_scene_and_camera(gpu):
    """Large coordinates stress the FP32 filters' absolute error terms."""
    rng = np.random.default_rng(5)
    off = np.array([4000.25, -1500.5, 9000.125])
    cam = ('camera', ('vector',) + tuple(off + [0, 0, -2]), ('vector', 0, 0, 0), 90, ('screen', 4, 3))
    light = ('point_light', ('colour', 1, 1, 1), ('vector',) + tuple(off + [5, -20, 0]), ('colour', 1, 1, 1))
    spheres = [('sphere', float(rng.uniform(0.3, 1.5)),
                ('vector',) + tuple(off + [rng.uniform(-10, 10), rng.uniform(-8, 4), rng.uniform(6, 40)]),
                mat(tuple(rng.uniform(0, 1, 3)), 4, 0.5, 0.5)) for _ in range(400)]
    floor = ('plane', ('vector', 0, -1, 0), 5 - 1500.5, mat((1, 1, 1), 1, 0, 0.3))
    check_scene([cam, light] + spheres + [floor], 96, 72, 4)


def test_huge_and_tiny_spheres(gpu):
    spheres = [('sphere', 1000, ('vector', 0, -1010, 50), mat((1, 0.2, 0.2), 4, 0.5, 0.3)),
               ('sphere', 0.01, ('vector', 0.1, 0.1, 1), mat((0, 1, 0), 4, 0.5, 0.3)),
               ('sphere', 300, ('vector', 400, 0, 900), mat((0, 0.3, 1), 50, 1, 0.6))]
    spheres += [('sphere', 0.05, ('vector', -1 + 0.07 * i, 0.5, 2 + 0.01 * i), mat((1, 1, 0), 1, 0, 0)) for i in range(40)]
    floor = ('plane', ('vector', 0, -1, 0), 5, mat((1, 1, 1), 1, 0, 0.2))
    check_scene([CAM, L1, L2] + spheres + [floor], 96, 72, 4, rays_equal=False)


@pytest.mark.parametrize("seed", range(6))
def test_random_mixed_scenes(gpu, seed):
    rng = np.random.default_rng(100 + seed)
    def v(lo, hi):
        return ('vector',) + tuple(float(x) for x in rng.uniform(lo, hi, 3))
    def m():
        return mat(tuple(float(x) for x in rng.uniform(0, 1, 3)), float(rng.choice([1, 2.5, 4, 20])),
                   float(rng.uniform(0, 1)), float(rng.choice([0, 0.3, 0.7, 1.0])))
    elems = [('point_light', ('colour',) + tuple(rng.uniform(0, 1, 3)), v(-20, 20), ('colour',) + tuple(rng.uniform(0, 1, 3)))
             for _ in range(int(rng.integers(1, 5)))]
    n_s = int(rng.choice([5, 60, 700]))
    elems += [('sphere', float(rng.uniform(0.2, 2.5)), ('vector', float(rng.uniform(-12, 12)), float(rng.uniform(-9, 5)),
               float(rng.uniform(2, 40))), m()) for _ in range(n_s)]
    elems += [('triangle', v(-10, 10), v(-10, 10), v(-10, 10), m()) for _ in range(int(rng.integers(0, 12)))]
    elems += [('plane', ('vector', float(rng.uniform(-0.3, 0.3)), -1, float(rng.uniform(-0.3, 0.3))), float(rng.uniform(3, 8)), m())
              for _ in range(int(rng.integers(0, 3)))]
    order = rng.permutation(len(elems))
    scene = [CAM] + [elems[i] for i in order]
    check_scene(scene, 80, 60, 4, rays_equal=False)


def test_band_parts_assemble_the_whole_frame(gpu):
    flat = sc.flatten(sc.demo_scene())
    dev = flat.upload(0)
    w, h, depth = 64, 47, 3
    whole, st = dev.render(w, h, depth, fmt="f64")
    for band_rows, n_parts in ((5, 3), (8, 2), (1, 7), (16, 4)):
        frame = np.full((h, w, 3), np.nan)
        rays = 0
        for part in range(n_parts):
            _, s = dev.render(w, h, depth, fmt="f64", band_rows=band_rows, n_parts=n_parts, part=part, out=frame)
            assert s["pixels"] == len(multigpu.part_rows(h, band_rows, n_parts, part)) * w
            rays += s["rays"]
        assert np.array_equal(frame, whole)
        assert rays == st["rays"]
    dev.close()


def test_async_slots_with_per_frame_cameras(gpu):
    flat = sc.flatten(sc.demo_scene())
    dev = flat.upload(0)
    w, h = 96, 54
    frames = [_lib.PinnedFrame(w * h * 3) for _ in range(_lib.MAX_SLOTS)]
    cams = [sc.pose_camera(k) for k in range(_lib.MAX_SLOTS)]
    for k in range(_lib.MAX_SLOTS):
        dev.render_async(w, h, 1, slot=k, fmt="rgb8", camera=cams[k], host_ptr=frames[k].ptr, host_bytes=w * h * 3)
    for k in range(_lib.MAX_SLOTS):
        dev.wait(k)
        got = frames[k].array(np.uint8, (h, w, 3))
        flat_k = sc.FlatScene(cams[k], flat.lights, flat.spheres, flat.triangles, flat.planes)
        ref, _, _ = oracle_frame(flat_k, w, h, 1)
        assert np.array_equal(got.astype(np.int64), np.clip(quantise(ref), 0, 255))
    for f in frames:
        f.close()
    dev.close()


def test_scene_clone_renders_identically(gpu):
    flat = sc.synthetic_scene("c3", n_spheres=2000)
    a = flat.upload(0)
    b = a.clone(0)
    fa, _ = a.render(160, 90, 3, fmt="f64", accel="bvh")
    fb, _ = b.render(160, 90, 3, fmt="f64", accel="bvh")
    assert np.array_equal(fa, fb)
    a.close()
    b.close()


def test_committed_golden_fixture(gpu):
    """GPU against tests/golden/demo_images.json (no oracle build needed for this one)."""
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "demo_images.json")))
    dev = sc.flatten(sc.demo_scene()).upload(0)
    for key, img in g["images"].items():
        for accel in ACCELS:
            rgb8, st = dev.render(img["width"], img["height"], img["depth"], fmt="rgb8", accel=accel)
            assert rgb8.reshape(-1).tolist() == img["rgb8"], (key, accel)
            assert st["rays"] == img["rays"]
    dev.close()


def test_host_mirror_writes_the_reference_ppm(gpu, tmp_path):
    """raytrace/5 through tracing_function(gpu) (raytracer.erl:723-733) writes the P3 file the
    oracle's pixel list would give."""
    out = tmp_path / "traced.ppm"
    assert raytracer.go(32, 24, str(out), 1, 'gpu') == 'ok'
    flat = sc.flatten(sc.demo_scene())
    ref, _, _ = oracle_frame(flat, 32, 24, 1)
    want = "P3\n32 24\n255\n" + "".join("%d %d %d " % tuple(px) for px in quantise(ref).reshape(-1, 3).tolist())
    assert out.read_text() == want
    pixels = raytracer.raytraced_pixel_list_gpu(4, 3, sc.demo_scene(), 5)
    assert [p[0] for p in pixels] == list(range(12))
    assert quantise(np.array([p[1] for p in pixels])).tolist() == json.load(
        open(os.path.join(os.path.dirname(__file__), "golden", "demo_images.json")))["appendix_a"]["4x3_d5"]
    assert raytracer.standalone(["16", "12", str(out), "1", "gpu"]) == 'ok'
    multi = raytracer.raytraced_pixel_list_gpu_distributed(32, 24, sc.demo_scene(), 1)
    single = raytracer.raytraced_pixel_list_gpu(32, 24, sc.demo_scene(), 1)
    assert multi == single


@pytest.mark.parametrize("workload", ["c1", "c5"])
def test_bench_dumps_the_frame_of_its_last_timed_step(gpu, tmp_path, workload):
    """bench.py --dump-outputs with two timed steps.  C1 (32x24) is written whole and is the RGB8 frame of the demo
    scene.  C5 (7680x4320, camera pose k at step k) is written as a seeded sample of rows under 64 MB, and those rows
    must show pose 1, the last timed step: not pose 0 (the untimed counting run and the first timed step) and not
    pose 2 (the last warm-up frame on the same slot)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", workload, "--steps", "2",
                          "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == 2
    frame, rows = np.load(tmp_path / "frame.npy"), np.load(tmp_path / "frame_rows.npy")
    assert frame.dtype == np.float32 and rows.dtype == np.float64
    w, h, pose = (32, 24, None) if workload == "c1" else (7680, 4320, 1)
    idx = rows.astype(np.int64)
    assert np.array_equal(idx, rows) and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < h
    if workload == "c1":
        assert idx.tolist() == list(range(h))
    else:
        assert len(idx) < h and frame.nbytes + rows.nbytes < 64_000_000
    dev = sc.flatten(sc.demo_scene()).upload(0)
    try:
        def rows_of(k):
            rgb8, _ = dev.render(w, h, 1, fmt="rgb8", camera=None if k is None else sc.pose_camera(k))
            return rgb8[idx].astype(np.float32)
        assert np.array_equal(frame, rows_of(pose))
        if workload == "c5":
            assert not np.array_equal(frame, rows_of(0)) and not np.array_equal(frame, rows_of(2))
    finally:
        dev.close()


# ---- BASELINE.json's full sizes: size-independent properties -------------------------------
def test_c3_full_4k_bvh_equals_linear_on_a_row_subset_and_oracle_on_a_lattice(gpu):
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    w, h, depth = 3840, 2160, 5
    full, st = dev.render(w, h, depth, fmt="f64", accel="bvh")
    assert st["pixels"] == w * h and st["rays"] > 8 * w * h
    sub = np.zeros_like(full)
    dev.render(w, h, depth, fmt="f64", accel="linear", band_rows=1, n_parts=108, part=37, out=sub)
    rows = multigpu.part_rows(h, 1, 108, 37)
    assert np.array_equal(sub[rows], full[rows])
    xs = ((np.arange(48) + 0.5) * w / 48).astype(np.int32)
    ys = ((np.arange(27) + 0.5) * h / 27).astype(np.int32)
    gx, gy = np.meshgrid(xs, ys)
    ref, _, _ = oracle_frame(flat, w, h, depth, pixels=(gx.reshape(-1), gy.reshape(-1)))
    got = full[gy.reshape(-1), gx.reshape(-1)]
    assert_double_parity(got, ref)
    assert np.array_equal(quantise(got), quantise(ref))
    rgb8, _ = dev.render(w, h, depth, fmt="rgb8", accel="bvh")
    assert np.array_equal(rgb8.astype(np.int64), np.clip(quantise(full), 0, 255))
    dev.close()


def test_c4_full_4k_bvh_equals_linear_scan_and_oracle_samples(gpu):
    """Config C4: the BVH must return the linear scan's hits on the 1M-sphere scene."""
    flat = sc.synthetic_scene("c4")
    dev = flat.upload(0)
    w, h, depth = 3840, 2160, 5
    full, st = dev.render(w, h, depth, fmt="f64", accel="bvh")
    assert st["accel_used"] == "bvh" and st["rays"] > 8 * w * h
    # one row in 1080 through the tiled linear scan (1M spheres per ray)
    sub = np.zeros_like(full)
    dev.render(w, h, depth, fmt="f64", accel="linear", band_rows=1, n_parts=1080, part=700, out=sub)
    rows = multigpu.part_rows(h, 1, 1080, 700)
    assert np.array_equal(sub[rows], full[rows])
    # ray batch: BVH == linear scan on (t bits, list position)
    rng = np.random.default_rng(11)
    n = 20000
    o = np.stack([rng.uniform(-210, 210, n), rng.uniform(-160, 5, n), rng.uniform(-5, 410, n)], axis=1)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([o, d], axis=1)
    ob, tb = dev.trace_rays(rays, accel="bvh")
    ol, tl = dev.trace_rays(rays, accel="linear")
    assert np.array_equal(ob, ol) and np.array_equal(tb, tl)
    # shadow rays through the lights' direction grids == shadow rays through the BVH, whole 4K frame
    walk, sw = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_NO_LIGHT_GRID)
    assert np.array_equal(walk, full) and sw["rays"] == st["rays"]
    del walk
    # the CPU oracle on a few pixels (each costs ~16 rays x 1M spheres)
    xs = np.array([400, 1900, 3000, 1200], dtype=np.int32)
    ys = np.array([300, 1500, 900, 2000], dtype=np.int32)
    ref, _, _ = oracle_frame(flat, w, h, depth, pixels=(xs, ys))
    assert_double_parity(full[ys, xs], ref)
    dev.close()


# ---- wavefront form of the BVH path (ERT_ACCEL_BVH) -----------------------------------------
def test_wavefront_binned_queues_render_the_same_frame(gpu):
    """Binning the hit queue by location only reschedules rays: frame and ray count are unchanged."""
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    w, h, depth = 640, 360, 5
    # hits are binned when shadow rays walk the BVH (here: direction grids switched off)
    a, sa = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_NO_LIGHT_GRID)
    b, sb = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_NO_LIGHT_GRID | _lib.FLAG_WF_UNSORTED)
    c, sc_ = dev.render(w, h, depth, fmt="f64", accel="bvh_mega")
    e, se = dev.render(w, h, depth, fmt="f64", accel="bvh")
    assert np.array_equal(a, b) and np.array_equal(a, c) and np.array_equal(a, e)
    assert sa["rays"] == sb["rays"] == sc_["rays"] == se["rays"]
    # binned > arrival order with separate shadow and shade launches > shadow rays and light fold in one launch
    # (every light has a direction grid) > one megakernel
    assert sa["gpu_launches"] > sb["gpu_launches"] > se["gpu_launches"] > sc_["gpu_launches"] == 1
    # instrumented run: same frame, counters filled
    d, sd = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_COUNT_TESTS)
    assert np.array_equal(a, d) and sd["box_tests"] > 0 and sd["sphere_filter_tests"] > 0
    dev.close()


def test_wavefront_deep_recursion_stops_when_the_queue_runs_dry(gpu):
    """Depths past 8 poll the path-queue length between bounces (ert_api.cu launch_wavefront)."""
    scene = [CAM, L1, L2] + [('sphere', 1.0, ('vector', 2.5 * i - 5, 0.3 * i, 8 + i),
                              mat((0.2 + 0.1 * i, 0.5, 0.9 - 0.1 * i), 4, 0.5, 0.6)) for i in range(5)]
    scene.append(('plane', ('vector', 0, -1, 0), 3, mat((1, 1, 1), 1, 0, 0.3)))
    check_scene(scene, 48, 36, 14, accels=("exact", "bvh", "bvh_mega"))


@pytest.mark.parametrize("n_lights", [1, 5])
def test_wavefront_light_counts(gpu, n_lights):
    lights = [('point_light', ('colour', 0.3 + 0.1 * k, 0.5, 0.2 * k), ('vector', 6 * k - 10, -8, -3 + 2 * k),
               ('colour', 1, 1, 1)) for k in range(n_lights)]
    flat = sc.synthetic_scene("c3", n_spheres=3000)
    scene_lights = np.zeros(n_lights, dtype=_lib.LIGHT_DT)
    for k, l in enumerate(lights):
        scene_lights[k]['diffuse_colour'] = l[1][1:]
        scene_lights[k]['location'] = l[2][1:]
        scene_lights[k]['specular_colour'] = l[3][1:]
        scene_lights[k]['order'] = k
    flat.spheres['order'] = np.arange(n_lights, n_lights + len(flat.spheres), dtype=np.int32)
    flat.planes['order'] = n_lights + len(flat.spheres)
    flat.lights = scene_lights
    dev = flat.upload(0)
    w, h, depth = 96, 54, 4
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    for accel in ("bvh", "bvh_mega"):
        frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
        assert_double_parity(frame, ref)
        assert np.array_equal(quantise(frame), quantise(ref))
        assert st["rays"] == ref_rays
    dev.close()


def test_wavefront_row_band_parts_assemble_the_frame(gpu):
    flat = sc.synthetic_scene("c3", n_spheres=5000)
    dev = flat.upload(0)
    w, h, depth = 250, 131, 4                      # ragged: width not a multiple of 8, partial last band
    full, st = dev.render(w, h, depth, fmt="f64", accel="bvh")
    out = np.zeros_like(full)
    rays = 0
    for part in range(3):
        _, sp = dev.render(w, h, depth, fmt="f64", accel="bvh", band_rows=8, n_parts=3, part=part, out=out)
        rays += sp["rays"]
    assert np.array_equal(out, full) and rays == st["rays"]
    dev.close()


def test_light_grids_answer_shadow_queries_like_the_bvh(gpu):
    """Direction grids (light_grid.cpp) vs BVH walks vs the unfiltered FP64 scan: same frame."""
    flat = sc.synthetic_scene("c3")
    dev = flat.upload(0)
    w, h, depth = 480, 270, 5
    a, sa = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_COUNT_TESTS)
    b, sb = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_COUNT_TESTS | _lib.FLAG_NO_LIGHT_GRID)
    c, _ = dev.render(w, h, depth, fmt="f64", accel="exact")
    assert np.array_equal(a, b) and np.array_equal(a, c)
    assert sa["rays"] == sb["rays"]
    assert sa["shadow_box_tests"] == 0 < sb["shadow_box_tests"]        # no walk when the light has a grid
    assert 0 < sa["shadow_filter_tests"] and 0 < sa["path_box_tests"] == sb["path_box_tests"]
    t, st = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_TIME_KERNELS)
    assert np.array_equal(a, t)
    assert st["path_launches"] == depth and st["shadow_launches"] == depth
    assert 0 < st["path_ms"] + st["shadow_ms"] + st["other_ms"] <= st["kernel_ms"] * 1.05
    dev.close()


def test_more_lights_than_direction_grids(gpu):
    """Lights past the first kMaxLightGrids (8) send their shadow rays through the BVH."""
    n_lights = 11
    flat = sc.synthetic_scene("c3", n_spheres=1500)
    lights = np.zeros(n_lights, dtype=_lib.LIGHT_DT)
    for k in range(n_lights):
        lights[k]['diffuse_colour'] = (0.05 * k, 0.3, 0.6 - 0.04 * k)
        lights[k]['location'] = (7.0 * k - 35, -25 + 3 * k, 2.0 * k)
        lights[k]['specular_colour'] = (1, 1, 1)
        lights[k]['order'] = k
    flat.spheres['order'] = np.arange(n_lights, n_lights + len(flat.spheres), dtype=np.int32)
    flat.planes['order'] = n_lights + len(flat.spheres)
    flat.lights = lights
    dev = flat.upload(0)
    w, h, depth = 80, 45, 3
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    frame, st = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_COUNT_TESTS)
    assert_double_parity(frame, ref)
    assert np.array_equal(quantise(frame), quantise(ref)) and st["rays"] == ref_rays
    assert st["shadow_box_tests"] > 0
    dev.close()


def test_light_inside_a_sphere_and_on_a_surface(gpu):
    """The `always` list of a direction grid: a light inside a sphere, and one touching another."""
    spheres = [('sphere', 3.0, ('vector', 0, 0, 12), mat((0.2, 0.6, 1.0), 20, 1, 0.4))]
    rng = np.random.default_rng(3)
    for i in range(80):
        c = rng.uniform(-8, 8, 3) + (0, 0, 14)
        spheres.append(('sphere', float(rng.uniform(0.3, 0.9)), ('vector',) + tuple(c.tolist()),
                        mat(tuple(rng.uniform(0, 1, 3).tolist()), 4, 0.5, 0.3)))
    lights = [('point_light', ('colour', 1, 1, 1), ('vector', 0.5, -0.5, 11), ('colour', 1, 1, 1)),     # inside sphere 0
              ('point_light', ('colour', 1, 0.5, 0.2), ('vector', 0, -3, 12), ('colour', 1, 1, 1)),    # on its surface
              ('point_light', ('colour', 0.3, 1, 0.4), ('vector', -12, -9, 2), ('colour', 1, 1, 1))]
    scene = [CAM] + lights + spheres + [('plane', ('vector', 0, -1, 0), 6, mat((1, 1, 1), 1, 0, 0.2))]
    check_scene(scene, 96, 72, 4, accels=("exact", "bvh", "bvh_mega"))


@pytest.mark.parametrize("n,expect", [(16, "exact"), (17, "linear"), (63, "linear"), (64, "linear"), (192, "linear"),
                                      (193, "bvh")])
def test_auto_strategy_thresholds(gpu, n, expect):
    """AUTO switches strategy at 16/17 and 192/193 spheres; direction grids start at 64.  Same frame on
    both sides of every threshold."""
    rng = np.random.default_rng(n)
    spheres = [('sphere', float(rng.uniform(0.2, 0.9)), ('vector', float(rng.uniform(-7, 7)), float(rng.uniform(-5, 4)),
                float(rng.uniform(4, 22))), mat(tuple(float(x) for x in rng.uniform(0, 1, 3)), 4, 0.5, 0.4))
               for _ in range(n)]
    scene = [CAM, L1, L2] + spheres + [('plane', ('vector', 0, -1, 0), 5, mat((1, 1, 1), 1, 0, 0.2))]
    flat = sc.flatten(scene)
    dev = flat.upload(0)
    w, h, depth = 72, 54, 4
    ref, ref_rays, _ = oracle_frame(flat, w, h, depth)
    frame, st = dev.render(w, h, depth, fmt="f64", accel="auto")
    assert st["accel_used"] == expect
    assert_double_parity(frame, ref)
    assert np.array_equal(quantise(frame), quantise(ref)) and st["rays"] == ref_rays
    wf, sw = dev.render(w, h, depth, fmt="f64", accel="bvh", flags=_lib.FLAG_COUNT_TESTS)
    assert np.array_equal(wf, frame) and sw["rays"] == ref_rays
    assert (sw["shadow_box_tests"] == 0) == (n >= 64)       # direction grids from 64 spheres on
    dev.close()
