"""Rotated cameras (DESIGN.md "Camera rotation"): C4 at 3840x2160, depth 5, accel=auto, rendered from 16 look_at poses
around the scene (8 azimuths at 2 elevations, the second above the spheres), with the default +z pose and that pose
with ERT_FLAG_CAMERA_ROTATION and a zero rotation as references.  Prints one JSON line per pose with kernel_ms (median
of --steps frames after one warm-up frame, L2 flushed before each), rays, accel_used and has_cell_grid, and the card's
name, power limit and clocks read in the same run.

usage: python tools/orbit_bench.py [--steps 5] [--workload c4] [--out FILE]"""
import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

import eraytracer_b200 as ert  # noqa: E402
from eraytracer_b200 import _lib, scene as sc  # noqa: E402
from mesh_bench import card  # noqa: E402

W, H, DEPTH = 3840, 2160, 5
ELEVATIONS = (("level", 0.0), ("above", -0.6))      # y of the camera above the centre, per unit of orbit radius


def orbit_poses(flat):
    """(label, location, rotation): the centre of the spheres' bounds, an orbit radius of 0.75 of the bounds' larger
    horizontal extent, 8 azimuths from the default camera's side (-z) round, at the centre's height and above."""
    c = flat.spheres['center']
    lo, hi = c.min(axis=0), c.max(axis=0)
    ctr = tuple(float(v) for v in (lo + hi) / 2.0)
    r = 0.75 * float(max(hi[0] - lo[0], hi[2] - lo[2]))
    out = []
    for label, ey in ELEVATIONS:
        for k in range(8):
            a = 2.0 * math.pi * k / 8
            loc = (ctr[0] + r * math.sin(a), ctr[1] + ey * r, ctr[2] - r * math.cos(a))
            if label == "above":
                loc = (loc[0], min(loc[1], float(lo[1]) - 10.0), loc[2])
            out.append(("%s_az%03d" % (label, 45 * k), loc, sc.look_at(loc, ctr)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workload", default="c4", choices=("c3", "c4"))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ert.load()
    info = card()
    rows = []
    flat = sc.synthetic_scene(a.workload)
    t0 = time.time()
    dev = flat.upload(0)
    create_s = time.time() - t0
    pin = _lib.PinnedFrame(W * H * 3)
    out8 = pin.array(np.uint8, (H, W, 3))
    base = flat.camera

    def cam_at(loc, rot):
        cam = _lib.Camera()
        cam.location[:] = loc
        cam.rotation[:] = rot
        cam.fov, cam.screen_width, cam.screen_height = base.fov, base.screen_width, base.screen_height
        return cam

    poses = [("default", tuple(base.location), (0.0, 0.0, 0.0), False),
             ("default_flag_zero", tuple(base.location), (0.0, 0.0, 0.0), True)]
    poses += [(label, loc, rot, True) for label, loc, rot in orbit_poses(flat)]
    for label, loc, rot, flag in poses:
        cam = cam_at(loc, rot)

        def frame():
            return dev.render(W, H, DEPTH, fmt="rgb8", accel="auto", camera=cam, camera_rotation=flag, out=out8)[1]
        frame()                                            # warm-up
        ms = []
        for _ in range(a.steps):
            _lib.l2_flush(0)
            st = frame()
            ms.append(st["kernel_ms"])
        d = {"what": "orbit", "workload": a.workload, "pose": label, "width": W, "height": H, "depth": DEPTH,
             "location": [round(v, 3) for v in loc], "rotation": [round(v, 4) for v in rot], "camera_rotation": flag,
             "kernel_ms": round(float(np.median(ms)), 3), "kernel_ms_min": round(min(ms), 3),
             "kernel_ms_max": round(max(ms), 3), "rays": st["rays"], "grays_per_s": round(st["rays"] / np.median(ms) / 1e6, 3),
             "accel_used": st["accel_used"], "has_cell_grid": st["has_cell_grid"], "steps": a.steps,
             "scene_create_s": round(create_s, 2)}
        d.update(info)
        line = json.dumps(d)
        print(line, flush=True)
        rows.append(line)
    pin.close()
    dev.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
