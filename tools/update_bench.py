"""In-place scene updates (DESIGN.md "Scene updates"): C4 and m4 animated over 64 frames (scene.animated_scene) at
3840x2160, one ert_scene_update per frame, for the default flags (stale grids dropped), ERT_UPDATE_REBUILD_GRIDS and
ERT_UPDATE_REBUILD.  Per step: update wall and device ms, H2D bytes, the trees' area ratios, and the frame at depth
1 and 5 after the update (the accel actually run).  At a few steps the same tables also go through a fresh
ert_scene_create: its seconds and its frames.  Prints one JSON line per measurement, with the card's name, power
limit and clocks read in the same run.

usage: python tools/update_bench.py [--scenes c4,m4] [--modes default,rebuild_grids,rebuild] [--steps 64]
                                    [--fresh-every 16] [--out FILE]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

import eraytracer_b200 as ert  # noqa: E402
from eraytracer_b200 import scene as sc  # noqa: E402
from mesh_bench import card  # noqa: E402

W, H = 3840, 2160
MODES = {"default": {}, "rebuild_grids": {"rebuild_grids": True}, "rebuild": {"rebuild": True}}


def frame(dev, depth, reps=2):
    """median kernel ms of `reps` frames (after one warm-up) and the accel that ran"""
    dev.render(W, H, depth, fmt="rgb8", accel="auto")
    ms = []
    for _ in range(reps):
        _, st = dev.render(W, H, depth, fmt="rgb8", accel="auto")
        ms.append(st["kernel_ms"])
    return round(float(np.median(ms)), 3), st["accel_used"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="c4,m4")
    ap.add_argument("--modes", default="default,rebuild_grids,rebuild")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--fresh-every", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ert.load()
    info = card()
    rows = []

    def emit(d):
        d.update(info)
        line = json.dumps(d)
        print(line, flush=True)
        rows.append(line)

    for name in a.scenes.split(","):
        for mode in a.modes.split(","):
            t0 = time.time()
            dev = sc.animated_scene(name, 0).upload(0)
            create_s = time.time() - t0
            d1, acc1 = frame(dev, 1)
            d5, acc5 = frame(dev, 5)
            emit({"what": "create", "scene": name, "mode": mode, "create_s": round(create_s, 3),
                  "frame_ms_d1": d1, "frame_ms_d5": d5, "accel_d1": acc1, "accel_d5": acc5})
            for k in range(1, a.steps + 1):
                flat = sc.animated_scene(name, k)
                t0 = time.time()
                u = flat.update(dev, **MODES[mode])
                wall = (time.time() - t0) * 1e3
                d1, acc1 = frame(dev, 1)
                d5, acc5 = frame(dev, 5)
                row = {"what": "update", "scene": name, "mode": mode, "step": k, "update_wall_ms": round(wall, 2),
                       "update_host_ms": round(u["host_ms"], 2), "update_device_ms": round(u["device_ms"], 3),
                       "h2d_bytes": u["h2d_bytes"], "sphere_area_ratio": round(u["sphere_area_ratio"], 5),
                       "triangle_area_ratio": round(u["triangle_area_ratio"], 5), "done": u["done"],
                       "has_cell_grid": u["has_cell_grid"], "light_grids": u["light_grids"],
                       "frame_ms_d1": d1, "frame_ms_d5": d5, "accel_d1": acc1, "accel_d5": acc5}
                if mode == "default" and k % a.fresh_every == 0:
                    t0 = time.time()
                    fresh = flat.upload(0)
                    row["fresh_create_s"] = round(time.time() - t0, 3)
                    row["fresh_frame_ms_d1"], row["fresh_accel_d1"] = frame(fresh, 1)
                    row["fresh_frame_ms_d5"], row["fresh_accel_d5"] = frame(fresh, 5)
                    fresh.close()
                emit(row)
            dev.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
