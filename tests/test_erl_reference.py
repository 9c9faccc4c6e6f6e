"""Parity pinned to what the reference's SOURCE TEXT computes.

oracle/erlref.py evaluates the reference's raytracer.erl itself (tokeniser, parser, Erlang semantics); the
reference's own test-suite run_tests/0 (erl:736-1133) passed under it.  tests/golden/erl_reference.json holds
what the reference's functions returned under it for the scenes of tests/erl_scenes.py: whole images through
raytraced_pixel_list_simple/4, nearest hits through nearest_object_intersecting_ray/2, and the text
write_pixels_to_ppm/5 wrote; tests/golden/erl_scene.json holds the term its scene/0 returns
(tests/golden/make_golden_erl.py regenerates both from the reference's source).
Here the C oracle, the Python restatement, the product's PPM writer, the Erlang host module and (gpu) the
CUDA path are held to the committed values — all doubles bit for bit on the CPU side; RGB8 equal and
|d| <= 1e-9 relative for the GPU (its shading is the forward form, DESIGN.md "Exactness"), (list position,
Distance bits) for rays.
"""
import json
import os
import sys

import numpy as np
import pytest

from oracle import orc, pyoracle
from erl_scenes import SCENES, scene_records
from helpers import assert_double_parity, assert_image_parity, quantise

HERE = os.path.dirname(os.path.abspath(__file__))

with open(os.path.join(HERE, "golden", "erl_reference.json")) as _fh:
    GOLD = json.load(_fh)
IMAGES = sorted(GOLD["images"])


def _oracle(name, w, h, depth):
    recs = scene_records(name)
    cam = orc.camera_array(recs[0])
    kind, f = orc.flatten(recs[1:])
    rgb, rays, _ = orc.render(cam, kind, f, w, h, depth, retrace=True)
    return rgb


def _gold_pixels(key):
    g = GOLD["images"][key]
    return g, np.array(g["pixels"], dtype=np.float64)


# ------------------------------------------------------------------ both restatements == reference
def test_both_oracles_render_the_references_demo_image():
    """demo_8x6_d2 is what the reference's raytraced_pixel_list_simple/4 returned for its own scene/0; the C oracle
    (on the package's demo scene) and the Python restatement (on its own scene/0) must both return it."""
    gold = np.array(GOLD["ppm"]["demo_8x6_d2"]["pixels"], dtype=np.float64)
    assert np.array_equal(_oracle("demo", 8, 6, 2), gold)
    img = [p[1] for p in pyoracle.raytraced_pixel_list_simple(8, 6, pyoracle.scene(), 2)]
    assert np.array_equal(np.array(img, dtype=np.float64), gold)


def test_scene_function_of_the_source_is_the_demo_scene_of_the_package():
    """tests/golden/erl_scene.json holds the term the reference's scene/0 returns (atoms as strings); every record,
    material and value of the package's demo scene and of the Python restatement's scene/0 must equal it, hit by a
    stored ray or not."""
    from eraytracer_b200 import scene as sc
    def plain(x):
        return [plain(y) for y in x] if isinstance(x, (tuple, list)) else x
    with open(os.path.join(HERE, "golden", "erl_scene.json")) as fh:
        want = json.load(fh)["scene"]
    assert want == plain(sc.demo_scene())
    assert want == plain(pyoracle.scene())


# ------------------------------------------------------------------ oracle == reference (everywhere)
@pytest.mark.parametrize("key", IMAGES)
def test_oracle_equals_the_reference_image_bit_for_bit(key):
    g, gold = _gold_pixels(key)
    rgb = _oracle(g["scene"], g["width"], g["height"], g["depth"])
    assert np.array_equal(rgb, gold), "%d of %d channel values differ" % (int((rgb != gold).sum()), gold.size)


@pytest.mark.parametrize("name", sorted(GOLD["rays"]))
def test_oracle_nearest_hits_equal_the_references(name):
    g = GOLD["rays"][name]
    recs = scene_records(name)
    kind, f = orc.flatten(recs[1:])
    rays = np.array(g["rays"], dtype=np.float64)
    idx, t = orc.nearest_batch(rays, kind, f)
    want_idx = np.array([h[0] for h in g["hits"]])
    want_t = np.array([h[1] for h in g["hits"]], dtype=np.float64)
    assert np.array_equal(idx, want_idx)
    hit = want_idx >= 0
    assert hit.sum() > len(rays) // 4
    assert np.array_equal(t[hit], want_t[hit])


def test_ppm_writer_writes_the_references_text(tmp_path):
    from eraytracer_b200 import ppm
    for key, (w, h) in (("awkward_8x6", (8, 6)), ("demo_8x6_d2", (8, 6))):
        g = GOLD["ppm"][key]
        pixels = [(k, tuple(p)) for k, p in enumerate(g["pixels"])]
        out = tmp_path / (key + ".ppm")
        ppm.write_pixels_to_ppm(w, h, 255, pixels, str(out))
        assert out.read_text() == g["text"], key
    # the quantisation rule the parity metric uses is the writer's (erl:678-680), negative values included
    g = GOLD["ppm"]["awkward_8x6"]
    want = [int(tok) for tok in g["text"].split("\n", 3)[3].split()]
    assert quantise(np.array(g["pixels"])).reshape(-1).tolist() == want


# ------------------------------------------------------------------ CUDA path == reference
GPU_ACCELS = {"demo": ("auto", "exact", "linear", "bvh", "grid"), "pose5": ("auto",), "pose37": ("auto",),
              "stress": ("auto", "exact", "linear", "bvh", "bvh_mega"), "mini_c3": ("auto", "exact", "linear", "bvh", "grid")}


@pytest.mark.gpu
@pytest.mark.parametrize("key", IMAGES)
def test_gpu_equals_the_reference_image(gpu, key):
    from eraytracer_b200 import scene as sc
    g, gold = _gold_pixels(key)
    w, h, depth = g["width"], g["height"], g["depth"]
    dev = sc.flatten(scene_records(g["scene"])).upload(0)
    try:
        for accel in GPU_ACCELS[g["scene"]]:
            frame, st = dev.render(w, h, depth, fmt="f64", accel=accel)
            assert_double_parity(frame.reshape(-1, 3), gold)
            assert np.array_equal(quantise(frame.reshape(-1, 3)), quantise(gold)), (key, accel)
            rgb8, _ = dev.render(w, h, depth, fmt="rgb8", accel=accel)
            assert np.array_equal(rgb8.reshape(-1, 3), np.clip(quantise(gold), 0, 255)), (key, accel)
            assert_image_parity(rgb8.reshape(-1, 3), np.clip(quantise(gold), 0, 255))
    finally:
        dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD["rays"]))
def test_gpu_nearest_hits_equal_the_references(gpu, name):
    from eraytracer_b200 import scene as sc
    g = GOLD["rays"][name]
    dev = sc.flatten(scene_records(name)).upload(0)
    rays = np.array(g["rays"], dtype=np.float64)
    want_idx = np.array([h[0] for h in g["hits"]])
    want_t = np.array([h[1] for h in g["hits"]], dtype=np.float64)
    hit = want_idx >= 0
    try:
        for accel in ("exact", "linear", "bvh", "bvh_mega", "grid"):
            order, t = dev.trace_rays(rays, accel=accel)
            assert np.array_equal(order, want_idx), accel
            assert np.array_equal(t[hit], want_t[hit]), accel
    finally:
        dev.close()


# ------------------------------------------------------------------ the Erlang scene generator of erl/ (SURVEY 8(f2))
def test_erlang_scene_generator_equals_the_python_generator():
    """erl/raytracer_gpu_scenes.erl cannot be compiled here (no OTP); it is EVALUATED by oracle/erlref.py — the
    evaluator the reference's own run_tests/0 passes under — and scene(c3) must equal, value for value, what
    eraytracer_b200/scene.py generates for the tests and the bench (splitmix64 on 64-bit integers, binary32 rounding
    through <<X:32/float>>, list order lights / spheres / plane)."""
    from oracle import erlref
    from eraytracer_b200 import scene as sc
    sys.setrecursionlimit(200000)
    root = os.path.dirname(HERE)
    with open(os.path.join(root, "erl", "raytracer_gpu_scenes.erl")) as fh:
        m = erlref.Module(fh.read(), name="raytracer_gpu_scenes")
    # the generator's primitives
    assert m.call("splitmix64", 0xE7A9C0DE00000003, 1) == 0xFAD5B148BCB3FFF2
    u = sc.splitmix64_uniform(0xE7A9C0DE00000003, 40)
    assert [m.call("uniform", 0xE7A9C0DE00000003, k + 1) for k in range(40)] == [float(x) for x in u]
    scene = erlref.to_py(m.call("scene", erlref.Atom("c3")))
    flat = sc.synthetic_scene("c3")
    assert scene[0] == ["camera", ["vector", 0.0, 0.0, -2.0], ["vector", 0.0, 0.0, 0.0], 90.0, ["screen", 4.0, 2.25]]
    lights, spheres, plane = scene[1:4], scene[4:-1], scene[-1]
    assert len(spheres) == len(flat.spheres) == 10000
    for k, l in enumerate(lights):
        assert l[0] == "point_light"
        assert l[1][1:] == [float(x) for x in flat.lights[k]["diffuse_colour"]]
        assert l[2][1:] == [float(x) for x in flat.lights[k]["location"]]
        assert l[3][1:] == [float(x) for x in flat.lights[k]["specular_colour"]]
    got = np.array([[s[1]] + s[2][1:] + s[3][1][1:] + s[3][2:] for s in spheres], dtype=np.float64)
    want = np.concatenate([flat.spheres["radius"][:, None], flat.spheres["center"], flat.spheres["material"]["colour"],
                           flat.spheres["material"]["specular_power"][:, None], flat.spheres["material"]["shininess"][:, None],
                           flat.spheres["material"]["reflectivity"][:, None]], axis=1)
    assert all(s[0] == "sphere" and s[2][0] == "vector" and s[3][0] == "material" for s in spheres)
    assert np.array_equal(got, want)                                  # every double, bit for bit
    assert plane[0] == "plane" and plane[1][1:] == [float(x) for x in flat.planes[0]["normal"]]
    assert plane[2] == float(flat.planes[0]["distance"])
    pm = flat.planes[0]["material"]
    assert plane[3][1][1:] == [float(x) for x in pm["colour"]]
    assert plane[3][2:] == [float(pm["specular_power"]), float(pm["shininess"]), float(pm["reflectivity"])]


# ------------------------------------------------------------------ the Erlang host module of erl/ (boundary, SURVEY 8(b))
def _host_module():
    from oracle import erlref
    sys.setrecursionlimit(200000)
    root = os.path.dirname(HERE)
    with open(os.path.join(root, "erl", "raytracer_gpu.erl")) as fh:
        return erlref, erlref.Module(fh.read(), name="raytracer_gpu")


def test_erlang_tracing_function_returns_the_references_pixel_list():
    """erl/raytracer_gpu.erl cannot be loaded by a BEAM here; its sequential functions are EVALUATED by oracle/erlref.py
    with the NIFs replaced by stand-ins that answer what the real ones answer (scene_upload -> {ok, Handle},
    render_pixel_list -> the pixel list the reference's raytraced_pixel_list_simple/4 returned for the demo scene at
    8x6, depth 2: {1, Colour} per pixel, erl:86-99, colours from tests/golden/erl_reference.json).  The tracing
    function must then return that list — clause order, guards, ok_or_exit/1 and the case are the module's."""
    from erl_scenes import to_term
    erlref, host = _host_module()
    A = erlref.Atom
    scene = [to_term(None, e) for e in scene_records("demo")]
    want = [(1, tuple(p)) for p in GOLD["ppm"]["demo_8x6_d2"]["pixels"]]
    asked = []
    host.externals[("scene_upload", 2)] = lambda sc_, dev: (A("ok"), ("handle", sc_))
    host.externals[("render_pixel_list", 5)] = lambda h, w, hh, d, opts: asked.append((h, w, hh, d)) or want
    got = host.call("raytraced_pixel_list_gpu", 8, 6, scene, 2)
    assert len(got) == 48 and erlref.exact_eq(got, want)
    assert len(asked) == 1 and erlref.exact_eq(asked[0], (("handle", scene), 8, 6, 2))
    assert host.call("raytraced_pixel_list_gpu", 0, 0, scene, 2) == A("done")          # erl:86-87
    assert host.call("raytraced_pixel_list_gpu_distributed", 0, 0, scene, 2) == A("done")
    with pytest.raises(erlref.ErlError, match="function_clause"):                    # the guards of erl:88-89
        host.call("raytraced_pixel_list_gpu", -1, 6, scene, 2)
    # an error tuple from the NIF becomes exit({raytracer_gpu, Reason})
    reason = (A("no_device"), 100, erlref.ErlString(ord(c) for c in "no CUDA device"))
    host.externals[("scene_upload", 2)] = lambda sc_, dev: (A("error"), reason)
    with pytest.raises(erlref.ErlExit) as ei:
        host.call("raytraced_pixel_list_gpu", 8, 6, scene, 2)
    assert erlref.exact_eq(ei.value.reason, (A("raytracer_gpu"), reason))
    host.externals[("scene_upload", 2)] = lambda sc_, dev: (A("ok"), ("handle", sc_))
    host.externals[("render_pixel_list", 5)] = lambda h, w, hh, d, opts: (A("error"), reason)
    with pytest.raises(erlref.ErlExit) as ei:
        host.call("raytraced_pixel_list_gpu", 8, 6, scene, 2)
    assert erlref.exact_eq(ei.value.reason, (A("raytracer_gpu"), reason))


def test_erlang_frame_helpers():
    """pixel_list_from_f64/3 (native doubles of an F64 frame -> [{Index, {R,G,B}}]), the distributed tracing function on
    top of it (render_binary/5 replaced by a stand-in: it spawns one process per GPU), and write_binary_to_ppm/4, whose
    file must be the text the reference's write_pixels_to_ppm/5 writes for the same image."""
    erlref, host = _host_module()
    A = erlref.Atom
    g = GOLD["ppm"]["demo_8x6_d2"]
    pix = np.array(g["pixels"], dtype=np.float64)
    got = host.call("pixel_list_from_f64", pix.tobytes(), 0, [])
    assert erlref.exact_eq(got, [(k, (float(p[0]), float(p[1]), float(p[2]))) for k, p in enumerate(pix)])
    host.externals[("render_binary", 5)] = lambda w, h, sc_, d, opts: pix.tobytes()
    assert erlref.exact_eq(host.call("raytraced_pixel_list_gpu_distributed", 8, 6, [], 2), got)
    frame = np.clip(quantise(pix), 0, 255).astype(np.uint8).tobytes()
    name = erlref.ErlString(ord(c) for c in "out.ppm")
    assert host.call("write_binary_to_ppm", 8, 6, frame, name) == A("ok")
    assert "".join(host.files["out.ppm"]) == g["text"]


def test_erlang_multi_gpu_driver_deals_the_parts_and_returns_the_shared_frame():
    """render_binary/5 (erl/raytracer_gpu.erl): one upload, clones for the other GPUs, ONE page-locked frame, one linked
    process per GPU rendering its row bands into it, results collected by selective receive.  Evaluated under the
    evaluator's sequential process model (a spawned fun runs to completion at the spawn) with stand-ins for the NIFs
    that record what they are asked and fill the frame the way ert_render places a part's rows."""
    erlref, host = _host_module()
    A = erlref.Atom
    w, h, n_gpus, depth = 8, 40, 4, 3
    calls = {"upload": [], "clone": [], "render": []}
    frame = bytearray(w * h * 3)

    def render_into(handle, fr, d, opts):
        part = next(o[1] for o in opts if isinstance(o, tuple) and o[0] == A("part"))
        band, n, p = part
        calls["render"].append((handle, d, part))
        for y in range(h):
            if (y // band) % n == p:                                 # the row-band rule of ert_render (band b -> part b % n)
                frame[y * w * 3:(y + 1) * w * 3] = bytes([p + 1]) * (w * 3)
        return A("ok")

    host.externals[("device_count", 0)] = lambda: (A("ok"), n_gpus)
    host.externals[("scene_upload", 2)] = lambda sc_, dev: calls["upload"].append(dev) or (A("ok"), ("handle", dev))
    host.externals[("scene_clone", 2)] = lambda hd, dev: calls["clone"].append((hd, dev)) or (A("ok"), ("handle", dev))
    host.externals[("frame_alloc", 3)] = lambda ww, hh, fmt: (A("ok"), ("frame", ww, hh, fmt))
    host.externals[("render_into", 4)] = render_into
    host.externals[("frame_binary", 1)] = lambda fr: bytes(frame)
    out = host.call("render_binary", w, h, [A("scene")], depth, [])
    assert calls["upload"] == [0] and calls["clone"] == [(("handle", 0), d) for d in (1, 2, 3)]   # built once, copied
    assert sorted(c[2][2] for c in calls["render"]) == [0, 1, 2, 3]
    assert all(c[0] == ("handle", c[2][2]) and c[1] == depth and c[2][0] == 8 and c[2][1] == n_gpus for c in calls["render"])
    assert out == bytes(frame) and 0 not in out                       # every row was rendered by exactly one part
    rows = np.frombuffer(out, dtype=np.uint8).reshape(h, w * 3)[:, 0]
    assert rows.tolist() == [(y // 8) % n_gpus + 1 for y in range(h)]
    # a part that fails takes the caller down with exit({raytracer_gpu, Reason})
    reason = (A("cuda"), 700, erlref.ErlString(ord(c) for c in "illegal address"))
    host.externals[("render_into", 4)] = lambda handle, fr, d, opts: (A("error"), reason)
    with pytest.raises(erlref.ErlExit) as ei:
        host.call("render_binary", w, h, [A("scene")], depth, [])
    assert erlref.exact_eq(ei.value.reason, (A("raytracer_gpu"), reason))
