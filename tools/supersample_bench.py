"""Supersampled frames (DESIGN.md "Supersampling"): kernel time of a supersample=N call against N*N plain frames, the
fold and resolve kernels' share of it, and the end-to-end wall time of an RGB8 frame in pinned host memory against
the host alternative (the N x resolution F64 frame copied to pinned host memory, then box-filtered and quantised in
numpy).  Prints one JSON line per measurement, with the card's name, power limit and clocks read in the same run.
L2 is flushed before every timed frame; every value is the median of --steps frames after one warm-up frame.

usage: python tools/supersample_bench.py [--steps 5] [--only c2,c3,c4,m3] [--out FILE]"""
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
from eraytracer_b200 import _lib, scene as sc  # noqa: E402
from mesh_bench import card  # noqa: E402

WORKLOADS = [
    # name, scene, width, height, depth, sample counts per axis
    ("c2", lambda: sc.flatten(sc.demo_scene()), 1920, 1080, 5, (1, 2, 4)),
    ("c3", lambda: sc.synthetic_scene("c3"), 3840, 2160, 5, (2,)),
    ("c4", lambda: sc.synthetic_scene("c4"), 3840, 2160, 5, (2,)),
    ("m3", lambda: sc.mesh_scene("m3"), 1920, 1080, 5, (2,)),
]


def median_of(steps, fn):
    fn()                                                   # warm-up
    vals = []
    for _ in range(steps):
        _lib.l2_flush(0)
        vals.append(fn())
    return float(np.median(vals))


def host_fold_rgb8(big, n):
    """The box filter of the contract in numpy: acc = c_0, acc + c_k in sample order, / (n*n), then RGB8."""
    acc = big[0::n, 0::n].copy()
    for k in range(1, n * n):
        j, i = divmod(k, n)
        acc += big[j::n, i::n]
    acc /= float(n * n)
    return np.maximum(np.minimum(np.trunc(acc * 255.0), 255.0), 0.0).astype(np.uint8)


def fold_kernel_ms(dev, w, h, depth, n):
    """Device time of the ss_fold launches of one supersampled frame (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.render(w, h, depth, fmt="rgb8", supersample=n)
        torch.cuda.synchronize()
    us, count = 0.0, 0
    for e in prof.key_averages():
        if "ss_fold" in e.key:
            us += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            count += e.count
    return us / 1000.0, count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--only", default="c2,c3,c4,m3")
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

    for name, make, W, H, depth, ns in WORKLOADS:
        if name not in a.only.split(","):
            continue
        t0 = time.time()
        dev = make().upload(0)
        create_s = time.time() - t0
        pin = _lib.PinnedFrame(W * H * 3)
        out8 = pin.array(np.uint8, (H, W, 3))

        def kernel(n):
            return dev.render(W, H, depth, fmt="rgb8", supersample=n, out=out8)[1]["kernel_ms"]
        plain_ms = median_of(a.steps, lambda: kernel(1))
        accel = dev.stats(0)["accel_used"]
        for n in ns:
            ss_ms = median_of(a.steps, lambda: kernel(n))
            st = dev.stats(0)

            def e2e():
                t = time.perf_counter()
                dev.render(W, H, depth, fmt="rgb8", supersample=n, out=out8)
                return (time.perf_counter() - t) * 1e3
            e2e_ms = median_of(a.steps, e2e)
            big_pin = _lib.PinnedFrame(n * W * n * H * 3 * 8)
            big = big_pin.array(np.float64, (n * H, n * W, 3))

            def host_alt():
                t = time.perf_counter()
                dev.render(n * W, n * H, depth, fmt="f64", out=big)
                host_fold_rgb8(big, n)
                return (time.perf_counter() - t) * 1e3
            host_ms = median_of(a.steps, host_alt)
            big_pin.close()
            fold_ms, folds = fold_kernel_ms(dev, W, H, depth, n) if n > 1 else (0.0, 0)
            emit({"what": "supersample", "workload": name, "width": W, "height": H, "depth": depth, "n": n,
                  "accel": accel, "scene_create_s": round(create_s, 2), "kernel_ms": round(ss_ms, 3),
                  "plain_kernel_ms": round(plain_ms, 3), "n2_plain_kernel_ms": round(n * n * plain_ms, 3),
                  "ratio_to_n2_plain": round(ss_ms / (n * n * plain_ms), 4),
                  "fold_resolve_ms": round(fold_ms, 3), "fold_launches": folds,
                  "fold_timing": "torch.profiler CUDA activity, one frame, L2 not flushed" if n > 1 else "none",
                  "rays": st["rays"], "gpu_launches": st["gpu_launches"],
                  "e2e_rgb8_pinned_ms": round(e2e_ms, 3), "host_alternative_ms": round(host_ms, 3),
                  "host_alternative": "N x frame F64 to pinned host, numpy fold + RGB8",
                  "e2e_speedup_vs_host": round(host_ms / e2e_ms, 3), "steps": a.steps})
        pin.close()
        dev.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
