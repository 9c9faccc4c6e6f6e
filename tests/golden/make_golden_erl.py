"""Generates tests/golden/erl_reference.json by RUNNING THE REFERENCE'S SOURCE TEXT.

    python tests/golden/make_golden_erl.py          (needs /root/reference/raytracer.erl; ~3 min)

oracle/erlref.py evaluates /root/reference/raytracer.erl itself (tokeniser + parser + Erlang
semantics; validated by the reference's own run_tests/0, which must return `ok` below).  Every value
in the output file was computed by the reference's functions from the reference's text — no
restatement is involved:

  * images: raytraced_pixel_list_simple/4 (erl:86-99) on scene/0 and on hand-built scenes that reach
    the rows no reference test pins (planes, triangles, shading, shadows, reflection, un-normalised
    plane normals, exact distance ties, several lights, a seeded random-sphere scene);
  * rays: nearest_object_intersecting_ray/2 (erl:300-346) for ray batches -> (list position, Distance);
  * ppm: write_pixels_to_ppm/5 (erl:668-685) run on a pixel list, i.e. the reference's own quantisation;
  * erl_scene.json: the term scene/0 (erl:618-665) returns, atoms as strings.  Its first version was written
    from eraytracer_b200.scene.demo_scene(), which test_scene_function_of_the_source_is_the_demo_scene_of_the_package
    held equal to the evaluated scene/0 from commit 7ea1da3 on (the package's demo scene has not changed since);
    running this script writes it from the source.

The file travels to the GPU box (the reference does not); tests/test_erl_reference.py holds the
oracle, the product's PPM writer and the CUDA path to it.
"""
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.setrecursionlimit(200000)

from oracle import erlref  # noqa: E402
from erl_scenes import SCENES, scene_terms, ray_batch  # noqa: E402


def render(m, scene, w, h, depth):
    px = m.call("raytraced_pixel_list_simple", w, h, scene, depth)
    return [[c for c in p[1]] for p in px]


def main():
    m = erlref.load()
    t0 = time.time()
    ok = m.call("run_tests")
    assert ok == erlref.Atom("ok"), ok
    out = {"source": "/root/reference/raytracer.erl evaluated by oracle/erlref.py",
           "run_tests": erlref.to_py(ok), "images": {}, "rays": {}, "ppm": {}}
    for name, spec in SCENES.items():
        scene = scene_terms(m, name)
        for (w, h, depth) in spec["images"]:
            t1 = time.time()
            out["images"]["%s_%dx%d_d%d" % (name, w, h, depth)] = {
                "scene": name, "width": w, "height": h, "depth": depth,
                "pixels": erlref.to_py(render(m, scene, w, h, depth))}
            print("%s %dx%d depth %d: %.1fs" % (name, w, h, depth, time.time() - t1), flush=True)
        n_rays = spec.get("rays", 0)
        if n_rays:
            rays = ray_batch(name, n_rays)
            res = []
            rest = scene[1:]
            for r in rays:
                ray = (erlref.Atom("ray"), erlref.vec(*r[:3]), erlref.vec(*r[3:]))
                hit = m.call("nearest_object_intersecting_ray", ray, rest)
                if hit == erlref.Atom("none"):
                    res.append([-1, 0.0])
                else:
                    # list position of the object (the reference returns the record itself; the first equal
                    # element is the one its scan kept, erl:319)
                    pos = next(k for k, e in enumerate(rest) if erlref.exact_eq(e, hit[0]))
                    res.append([pos, float(hit[1])])
            out["rays"][name] = {"rays": rays.tolist(), "hits": res}
    # the reference's own writer on a pixel list with the awkward values (erl:668-685)
    awkward = [0, 0.0, 0.5, 1, 1.0, 0.999, 1.5, 254.9 / 255, 255.0 / 255, 256.0 / 255, 3.7, 1e-9, -0.25, -1.5, 0.0039, 0.004]
    pixels = [(k, (awkward[k % len(awkward)], awkward[(k * 5 + 1) % len(awkward)], awkward[(k * 7 + 2) % len(awkward)]))
              for k in range(48)]
    m.call("write_pixels_to_ppm", 8, 6, 255, pixels, erlref.ErlString(ord(c) for c in "mem.ppm"))
    out["ppm"]["awkward_8x6"] = {"pixels": [list(p[1]) for p in pixels], "text": "".join(m.files["mem.ppm"])}
    demo = m.call("raytraced_pixel_list_simple", 8, 6, m.call("scene"), 2)
    m.call("write_pixels_to_ppm", 8, 6, 255, demo, erlref.ErlString(ord(c) for c in "demo.ppm"))
    out["ppm"]["demo_8x6_d2"] = {"pixels": erlref.to_py([list(p[1]) for p in demo]), "text": "".join(m.files["demo.ppm"])}
    with open(os.path.join(HERE, "erl_reference.json"), "w") as fh:
        json.dump(out, fh)
    with open(os.path.join(HERE, "erl_scene.json"), "w") as fh:
        json.dump({"source": "scene/0 of raytracer.erl (erl:618-665) evaluated by oracle/erlref.py",
                   "scene": erlref.to_py(m.call("scene"))}, fh)
    print("wrote erl_reference.json in %.0fs (%d function calls evaluated)" % (time.time() - t0, m.calls))


if __name__ == "__main__":
    main()
