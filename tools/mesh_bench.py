"""Triangle-mesh measurements (DESIGN.md "Triangle BVH"): m4 frames at 3840x2160, depth 1 and 5, through the
triangle BVH; per-ray test counts; the FP64 share of the literal triangle tests; an 8-row band of the walk against
ERT_ACCEL_EXACT (the linear FP64 scan); and small scenes either side of kTriBvhMin.  Prints one JSON line per
measurement, with the card's name, power limit and clocks read in the same run.

usage: python tools/mesh_bench.py [--steps N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import eraytracer_b200 as ert  # noqa: E402
from eraytracer_b200 import _lib, scene as sc  # noqa: E402

# FP64 lane instructions of one literal test that reaches t (triangle_exact, erl:402-455: 24 DADD, 24 DMUL without
# contraction), the division not counted: the share below is an upper bound of what the literal tests ask of the pipe
FP64_INSTR_PER_TRIANGLE_TEST = 48


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"card": "unknown"}
    return dict(zip(["card", "power_limit", "clock_sm", "clock_sm_max", "clock_mem"], [s.strip() for s in out.split(",")]))


def frame_ms(dev, w, h, depth, accel, steps, **kw):
    dev.render(w, h, depth, fmt="rgb8", accel=accel, **kw)                          # warm-up
    ms = []
    for _ in range(steps):
        _, st = dev.render(w, h, depth, fmt="rgb8", accel=accel, **kw)
        ms.append(st["kernel_ms"])
    return float(np.median(ms)), st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ert.load()
    info = card()
    fp64 = _lib.fp64_peak(0)
    rows = []

    def emit(d):
        d.update(info)
        line = json.dumps(d)
        print(line, flush=True)
        rows.append(line)

    t0 = time.time()
    flat = sc.mesh_scene("m4")
    dev = flat.upload(0)
    emit({"what": "m4 scene", "triangles": len(flat.triangles), "spheres": len(flat.spheres),
          "create_s": round(time.time() - t0, 2)})
    W, H = 3840, 2160
    for depth in (1, 5):
        for accel in ("auto", "bvh_mega", "bvh", "grid"):
            ms, st = frame_ms(dev, W, H, depth, accel, a.steps)
            _, cnt = dev.render(W, H, depth, fmt="rgb8", accel=accel, flags=_lib.FLAG_COUNT_TESTS)
            rays = cnt["rays"]
            lit = cnt["exact_other_tests"]
            emit({"what": "m4 frame", "accel": st["accel_used"], "requested": accel, "depth": depth, "ms": round(ms, 3),
                  "rays": rays, "grays_per_s": round(rays / ms / 1e6, 3),
                  "box_tests_per_ray": round(cnt["box_tests"] / rays, 2),
                  "literal_tri_tests_per_ray": round(lit / rays, 2),
                  "fp64_share_of_literal_tests": round(lit * FP64_INSTR_PER_TRIANGLE_TEST / (ms * 1e-3) / fp64, 4),
                  "fp64_peak_lane_instr_per_s": fp64})
    # one band of 8 rows: the walk against the linear FP64 scan of every triangle
    n_parts = H // 8
    for accel in ("auto", "exact"):
        ms, st = frame_ms(dev, W, H, 5, accel, 1 if accel == "exact" else a.steps, band_rows=8, n_parts=n_parts,
                          part=n_parts // 2)
        emit({"what": "m4 band of 8 rows", "accel": st["accel_used"], "depth": 5, "ms": round(ms, 3),
              "rays": st["rays"]})
    dev.close()
    # either side of the triangle-BVH threshold (kTriBvhMin = 64): the linear scan below, the walk from there
    for n_tris in (32, 63, 64, 128, 512):
        small = sc.mesh_scene("m3", n_triangles=n_tris)
        small.spheres = small.spheres[:16]
        small.planes['order'] = 3 + 16 + n_tris
        small.triangles['order'] -= 3000 - 16
        d = small.upload(0)
        for accel in ("auto", "exact"):
            ms, st = frame_ms(d, 1920, 1080, 5, accel, a.steps)
            emit({"what": "threshold", "triangles": n_tris, "spheres": 16, "requested": accel,
                  "accel": st["accel_used"], "ms": round(ms, 3), "rays": st["rays"]})
        d.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
