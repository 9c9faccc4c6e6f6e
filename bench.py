#!/usr/bin/env python
"""bench.py — Mrays/s and frame ms of the eraytracer hot path on N B200s.

  python bench.py --gpus N --steps K --warmup W [--workload c4] [--impl reference] [--dump-outputs DIR]

A "step" is one frame of the workload.  The scene is uploaded once before timing
(BASELINE.json north_star: "uploads a flattened SoA scene once"); `value` is timed with the
frame kept on the device, `e2e` through the synchronous C-ABI call ert_render() into a
(pinned / shared) HOST frame with the camera passed in every step.  With N > 1 (torchrun,
one rank per GPU) the SAME frame is split into interleaved row bands, one part per rank
(strong scaling, no collective on the data path); times are CUDA-event times, max over ranks.

--impl reference times the CPU oracle (a C restatement of raytracer.erl; the reference
itself needs Erlang/OTP, which this image does not have) on all host cores over a bounded
lattice of pixels of the same frame.

--dump-outputs DIR writes the RGB8 frame the last step of the timed block rendered (this rank's rows; the values
as float32) to DIR/frame.npy, DIR/frame_rank<R>.npy with N > 1, and the row index of each of its rows to
DIR/frame_rows.npy (frame_rank<R>_rows.npy).  Frames over DUMP_BYTES in float32 keep a fixed, seeded sample of
rows, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (description, scene, width, height, depth)
    "c1": ("C1 demo scene 32x24 depth 1 (run.sh)", "demo", 32, 24, 1),
    "c2": ("C2 demo scene 1920x1080 depth 1 (run-concurrent.sh depth)", "demo", 1920, 1080, 1),
    "c2d5": ("C2 demo scene 1920x1080 depth 5 (raytrace/1 default depth)", "demo", 1920, 1080, 5),
    "c3": ("C3 synthetic 10k-sphere scene 3840x2160, 3 point lights, depth 5", "c3", 3840, 2160, 5),
    "c4": ("C4 synthetic 1M-sphere scene 3840x2160, 3 point lights, depth 5 (accelerated nearest hit == linear scan)", "c4", 3840, 2160, 5),
    "c4d1": ("C4 synthetic 1M-sphere scene 3840x2160, 3 point lights, depth 1 (run-concurrent.sh depth)", "c4", 3840, 2160, 1),
    "c5": ("C5 demo scene 7680x4320 depth 1, camera pose k of 64 per step", "demo", 7680, 4320, 1),
}


DUMP_BYTES = 60 << 20       # float32 frame values written by --dump-outputs, over all ranks
DUMP_SEED = 20260101


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on
# stdout whatever NCCL_DEBUG_FILE says when stderr is a file), so file descriptor 1 is pointed at stderr for
# the whole run and the result line goes to the saved original.
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def build_scene(kind):
    from eraytracer_b200 import scene as sc
    if kind == "demo":
        return sc.flatten(sc.demo_scene())
    return sc.synthetic_scene(kind)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.tmp = None

    def start(self):
        try:
            self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        clocks, maxes, power, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.tmp:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                if int(parts[0]) != self.gpu_index:
                    continue
                clocks.append(float(parts[1]))
                maxes.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.tmp.close()
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass
        if not clocks:
            # the timed region was shorter than the sampling period: one synchronous sample right after it
            try:
                txt = subprocess.run(["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu_index)], capture_output=True, text=True, timeout=20).stdout
                parts = [p.strip() for p in txt.strip().split(",")]
                if len(parts) >= 8:
                    clocks.append(float(parts[1])); maxes.append(float(parts[2])); power.append(float(parts[3]))
                    for nm, val in zip(names, parts[4:8]):
                        if val.lower().startswith("active"):
                            reasons.add(nm)
                    out["note"] = "timed region shorter than the 100 ms sampling period; sampled once right after it"
            except Exception:
                pass
        if clocks:
            out["sm_mhz"] = statistics.median(clocks)
            out["sm_max_mhz"] = max(maxes)
            out["power_w_max"] = max(power)
            out["samples"] = len(clocks)
        out["reasons"] = sorted(reasons)
        return out


# --------------------------------------------------------------------------- CPU arm
def lattice(width, height, nx, ny):
    xs = ((np.arange(nx) + 0.5) * width / nx).astype(np.int32)
    ys = ((np.arange(ny) + 0.5) * height / ny).astype(np.int32)
    gx, gy = np.meshgrid(xs, ys)
    return gx.reshape(-1).astype(np.int32), gy.reshape(-1).astype(np.int32)


class CpuArm:
    """The oracle (oracle/oracle.c) on all host cores over a lattice of pixels."""

    def __init__(self, flat, width, height, depth):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from helpers import oracle_scene_from_flat
        from oracle import orc
        self.orc = orc
        self.cam, self.kind, self.f = oracle_scene_from_flat(flat)
        self.w, self.h, self.depth = width, height, depth
        self.cores = os.cpu_count() or 1

    def run(self, nx, ny):
        px = lattice(self.w, self.h, nx, ny)
        t0 = time.perf_counter()
        _, rays, _ = self.orc.render(self.cam, self.kind, self.f, self.w, self.h, self.depth,
                                     pixels=px, nthreads=self.cores)
        dt = time.perf_counter() - t0
        return rays, dt, len(px[0])

    def sized_sample(self, budget_s):
        """Picks a lattice that costs about budget_s seconds (capped at the full frame)."""
        nx, ny = 8, 4
        rays, dt, npx = self.run(nx, ny)
        per_px = max(dt / npx, 1e-7)
        target = int(min(self.w * self.h, max(32, budget_s / per_px)))
        aspect = self.w / self.h
        ny = max(1, int((target / aspect) ** 0.5))
        nx = max(1, int(ny * aspect))
        return min(nx, self.w), min(ny, self.h)


def reference_arm(args, rank):
    if rank != 0:
        return 0
    desc, kind, w, h, depth = WORKLOADS[args.workload]
    flat = build_scene(kind)
    arm = CpuArm(flat, w, h, depth)
    total_steps = args.steps + args.warmup
    budget = min(10.0, 150.0 / max(total_steps, 1))
    nx, ny = arm.sized_sample(budget)
    for _ in range(args.warmup):
        arm.run(nx, ny)
    rays_total, t_total, npx = 0, 0.0, 0
    for _ in range(args.steps):
        rays, dt, npx = arm.run(nx, ny)
        rays_total += rays
        t_total += dt
    value = rays_total / t_total / 1e6
    sample = "%dx%d pixel lattice (%d px) of the %dx%d frame per step" % (nx, ny, npx, w, h)
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_total / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "width": w, "height": h, "depth": depth,
                   "sample": sample, "rays": "unique rays (one per nearest-object scan)"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": arm.cores, "kind": "port",
                         "sample": sample,
                         "note": "C restatement of raytracer.erl (oracle/oracle.c), not BEAM: "
                                 "Erlang/OTP is not installed in this image"},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)
    return 0


# --------------------------------------------------------------------------- GPU arm
def dump_frame(out_dir, dev, w, h, band_rows, n_parts, rank, world):
    """Writes the RGB8 rows of this rank's part that slot 0 rendered last (ert_download), see --dump-outputs."""
    from eraytracer_b200 import _lib, multigpu
    frame = np.zeros((h, w, 3), dtype=np.uint8)
    _lib.check(_lib.load().ert_download(dev.handle, 0, frame.ctypes.data, frame.nbytes))
    rows = multigpu.part_rows(h, band_rows, n_parts, rank)
    max_rows = DUMP_BYTES // world // (w * 3 * 4)
    if len(rows) > max_rows:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(rows, max_rows, replace=False))
    name = "frame" if world == 1 else "frame_rank%d" % rank
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), frame[rows].astype(np.float32))
    np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
    log("[rank %d] wrote %d of %d rows of the last timed frame to %s" % (rank, len(rows), h, out_dir))


def gpu_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from eraytracer_b200 import _lib, multigpu
    from eraytracer_b200 import scene as sc

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device is visible; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL writes its version banner (levels VERSION and WARN) to stdout; the bench prints exactly one
        # line there, so NCCL's log goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(value, op):
        if world == 1:
            return value
        t = torch.tensor([float(value)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return float(t.item())

    desc, kind, w, h, depth = WORKLOADS[args.workload]
    accel = args.accel
    t0 = time.perf_counter()
    flat = build_scene(kind)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    dev = flat.upload(local_rank)
    t_upload = time.perf_counter() - t0
    log("[rank %d] scene built in %.2fs, flattened+BVH+uploaded in %.2fs" % (rank, t_gen, t_upload))

    n_parts = world
    band_rows = multigpu.default_band_rows(h, world)
    fmt = "rgb8"
    frame_bytes = w * h * 3
    # C5 (a batch of camera poses) keeps two frames in flight, so it needs two host frames
    pipelined = args.workload == "c5"
    n_host = 2 if pipelined else 1
    hosts, shareds = [], []
    for k in range(n_host):
        if world == 1:
            hosts.append(_lib.PinnedFrame(frame_bytes))
            shareds.append(None)
        else:
            name = "ert_b200_frame_%s_%d" % (os.environ.get("MASTER_PORT", "0"), k)
            sh = multigpu.SharedFrame(name, frame_bytes, create=True) if rank == 0 else None
            barrier()
            if rank != 0:
                sh = multigpu.SharedFrame(name, frame_bytes, create=False)
            sh.register()
            hosts.append(sh)
            shareds.append(sh)
    host_ptr = hosts[0].ptr
    shared = shareds[0]

    def camera_for(step):
        return sc.pose_camera(step % 64) if args.workload == "c5" else None

    common = dict(fmt=fmt, accel=accel, band_rows=band_rows, n_parts=n_parts, part=rank)
    peak = _lib.fp32_peak(local_rank)
    peak_rrr = _lib.fp32_peak_rrr(local_rank)
    peak64 = _lib.fp64_peak(local_rank)
    d2h_peak = _lib.d2h_peak(local_rank, max(frame_bytes // max(world, 1), 1 << 20))

    # warm-up through the full end-to-end path
    for i in range(max(args.warmup, 0)):
        k = i % n_host                               # the pipelined loop uses two slots: warm both
        dev.render_async(w, h, depth, slot=k, camera=camera_for(i), host_ptr=hosts[k].ptr,
                         host_bytes=frame_bytes, **common)
        dev.wait(k)

    # instrumented (untimed) run: test counters for the roofline accounting
    dev.render_async(w, h, depth, slot=0, flags=_lib.FLAG_COUNT_TESTS, camera=camera_for(0), **common)
    dev.wait(0)
    counted = dev.stats(0)
    # per-level ray counts of this rank's part (untimed): the reference re-traces the reflection once per
    # light (erl:216-224), so level b of its recursion runs L^b times; frames that did not go through the
    # wavefront are run through it once to get the counts
    levels = counted
    if not counted.get("bounces_recorded"):
        dev.render_async(w, h, depth, slot=0, camera=camera_for(0), **dict(common, accel="bvh"))
        dev.wait(0)
        levels = dev.stats(0)
    n_l = int(len(flat.lights))
    uniq = sum(p_ + n_l * h_ for p_, h_ in zip(levels["bounce_path_rays"], levels["bounce_hits"]))
    refeq = sum((n_l ** b) * (p_ + n_l * h_)
                for b, (p_, h_) in enumerate(zip(levels["bounce_path_rays"], levels["bounce_hits"])))
    refeq_ratio = (refeq / uniq) if uniq else 1.0

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- timed block A: frame stays on the device (inputs resident in HBM) ----
    barrier()
    kernel_ms, rays = 0.0, 0
    launches = 0
    split = {"path_ms": 0.0, "shadow_ms": 0.0, "other_ms": 0.0, "path_launches": 0, "shadow_launches": 0}
    for i in range(args.steps):
        _lib.l2_flush(local_rank)
        dev.render_async(w, h, depth, slot=0, camera=camera_for(i), **common)
        dev.wait(0)
        st = dev.stats(0)
        kernel_ms += st["kernel_ms"]                  # two CUDA events on the launching stream around the frame's launches
        rays += st["rays"]
        launches += st["gpu_launches"]
    barrier()
    if args.dump_outputs:
        dump_frame(args.dump_outputs, dev, w, h, band_rows, n_parts, rank, world)
    # split by kernel class: a separate pass with one event before and after EVERY launch (ERT_FLAG_TIME_KERNELS;
    # the events cost ~3 % on a 2 ms part, so the pass is kept out of `value`)
    split_steps = max(1, min(args.steps, 5))
    split_ms = 0.0
    for i in range(split_steps):
        _lib.l2_flush(local_rank)
        dev.render_async(w, h, depth, slot=0, camera=camera_for(i), flags=_lib.FLAG_TIME_KERNELS, **common)
        dev.wait(0)
        st = dev.stats(0)
        split_ms += st["kernel_ms"]
        for k in split:
            split[k] += st[k]
    for k in ("path_ms", "shadow_ms", "other_ms"):
        split[k] *= args.steps / split_steps          # per-class ms below are divided by args.steps
    split["path_launches"] = split["path_launches"] * args.steps // split_steps
    split["shadow_launches"] = split["shadow_launches"] * args.steps // split_steps
    split_frame_ms = split_ms / split_steps
    barrier()
    kernel_ms_max = reduce(kernel_ms, "max")
    rays_all = reduce(rays, "sum")
    launches_all = int(reduce(launches, "sum"))

    # ---- timed block B: end to end through ert_render() with a host frame ----
    barrier()
    e2e_wall, e2e_dev_ms, d2h = 0.0, 0.0, 0
    lib = _lib.load()
    import ctypes
    if pipelined:
        # sustained frames: pose i renders on slot i % 2 into host frame i % 2 while the previous pose's
        # rows are still on their way to the host (ert_render_async / ert_wait, the same C ABI)
        t1 = time.perf_counter()
        for i in range(args.steps):
            k = i % 2
            dev.wait(k)
            if i >= 2:
                st = dev.stats(k)
                e2e_dev_ms += st["total_ms"]
                d2h += st["d2h_bytes"]
            dev.render_async(w, h, depth, slot=k, camera=camera_for(i), host_ptr=hosts[k].ptr,
                             host_bytes=frame_bytes, **common)
        for k in range(2):
            dev.wait(k)
            st = dev.stats(k)
            if args.steps > k:
                e2e_dev_ms += st["total_ms"]
                d2h += st["d2h_bytes"]
        e2e_wall = time.perf_counter() - t1
    else:
        for i in range(args.steps):
            _lib.l2_flush(local_rank)
            p = dev._params(w, h, depth, fmt, accel, band_rows, n_parts, rank, 0, camera_for(i) or flat.camera)
            t1 = time.perf_counter()
            _lib.check(lib.ert_render(dev.handle, ctypes.byref(p), host_ptr, frame_bytes))
            e2e_wall += time.perf_counter() - t1
            st = dev.stats(0)
            e2e_dev_ms += st["total_ms"]
            d2h += st["d2h_bytes"]
    barrier()
    # ---- the FP32-roofline kernel on this scene: the brute-force scan (the reference's linear scan,
    # erl:300-346) over a 4-row band of the same frame, every ray against every sphere ----
    scan = None
    if rank == 0 and len(flat.spheres) > 192 and not args.no_scan_roofline:
        band = dict(fmt=fmt, accel="linear", band_rows=4, n_parts=max(h // 4, 1), part=max(h // 8, 0))
        for _ in range(2):
            dev.render_async(w, h, depth, slot=0, camera=camera_for(0), **band)
            dev.wait(0)
        dev.render_async(w, h, depth, slot=0, flags=_lib.FLAG_COUNT_TESTS, camera=camera_for(0), **band)
        dev.wait(0)
        sc_counted = dev.stats(0)
        sc_split = {"path_ms": 0.0, "shadow_ms": 0.0, "other_ms": 0.0, "path_launches": 0, "shadow_launches": 0}
        sc_ms, sc_steps = 0.0, 3
        for _ in range(sc_steps):
            _lib.l2_flush(local_rank)
            dev.render_async(w, h, depth, slot=0, flags=_lib.FLAG_TIME_KERNELS, camera=camera_for(0), **band)
            dev.wait(0)
            st = dev.stats(0)
            sc_ms += st["kernel_ms"]
            for k in sc_split:
                sc_split[k] += st[k]
        p_s = sc_split["path_ms"] / sc_steps * 1e-3
        s_s = sc_split["shadow_ms"] / sc_steps * 1e-3
        scan = {
            "kernel": "wf_scan<path> (ert_scan.cuh): FP32 filter of every (path ray, sphere) pair, packed FFMA2, "
                      "TMA-fed shared-memory ring",
            "workload": "rows %d-%d of the %dx%d frame, depth %d, accel=linear: %d rays x %d spheres" % (
                4 * band["part"], 4 * band["part"] + 3, w, h, depth, sc_counted["rays"], len(flat.spheres)),
            "bound": "fp32", "unit": "Glane-instr/s", "peak": peak / 1e9,
            "accounting": "10 FP32-pipe lane-instructions per (ray, sphere) filter test (3 FADD, 1 FMUL, 6 FFMA), "
                          "tests counted by an instrumented run of the same band, divided by the CUDA-event time of "
                          "the scan launches of that class inside %d timed frames" % sc_steps,
            "path_filter_tests": int(sc_counted["path_filter_tests"]),
            "shadow_filter_tests": int(sc_counted["shadow_filter_tests"]),
            "exact_fp64_sphere_tests": int(sc_counted["exact_sphere_tests"]),
            "path_ms": p_s * 1e3, "shadow_ms": s_s * 1e3, "frame_ms": sc_ms / sc_steps,
            "path_launches": sc_split["path_launches"] / sc_steps,
            "achieved": sc_counted["path_filter_tests"] * 10 / max(p_s, 1e-12) / 1e9,
            "frac": sc_counted["path_filter_tests"] * 10 / max(p_s, 1e-12) / peak,
            "shadow_achieved": sc_counted["shadow_filter_tests"] * 10 / max(s_s, 1e-12) / 1e9,
            "shadow_frac": sc_counted["shadow_filter_tests"] * 10 / max(s_s, 1e-12) / peak,
            "shadow_note": "a shadow ray is a full nearest-object scan from the light (erl:256-267 calls "
                           "nearest_object_intersecting_ray/2): every shadow ray meets every sphere, as in the reference",
        }
    e2e_wall_max = reduce(e2e_wall, "max")
    e2e_dev_ms_max = reduce(e2e_dev_ms, "max")
    d2h_all = reduce(d2h, "sum")
    clocks = sampler.stop()

    # the assembled host frame must equal a single-GPU render of the whole frame
    assembled_ok = None
    if world > 1:
        dev.render_async(w, h, depth, slot=0, camera=camera_for(0), host_ptr=hosts[0].ptr, host_bytes=frame_bytes, **common)
        dev.wait(0)
        barrier()
        if rank == 0:
            full, _ = dev.render(w, h, depth, fmt=fmt, accel=accel, camera=camera_for(0))
            assembled_ok = bool(np.array_equal(full, shared.array(np.uint8, (h, w, 3))))

    if rank == 0:
        steps = max(args.steps, 1)
        ms_per_step = kernel_ms_max / steps
        value = rays_all / steps / (ms_per_step * 1e-3) / 1e6
        e2e_ms = 1e3 * e2e_wall_max / steps
        e2e_value = rays_all / steps / (e2e_ms * 1e-3) / 1e6
        # roofline (rank 0's launches).  Wavefront frames: the dominant kernel class is the BVH walk of
        # the path rays (wf_trace_path / wf_trace_path_refill); other accels are one kernel per frame.
        k_s = (kernel_ms / steps) * 1e-3
        # cell steps of the grid walks belong to the path class (shadow rays never use the cell grid)
        cell_instr = counted.get("cell_steps", 0) * 4
        frame_lane_instr = counted["box_tests"] * 6 + counted["sphere_filter_tests"] * 10 + cell_instr
        wavefront = split["path_launches"] > 0
        dom = "path" if split["path_ms"] >= split["shadow_ms"] else "shadow"
        if wavefront:
            lane_instr = counted[dom + "_box_tests"] * 6 + counted[dom + "_filter_tests"] * 10 + (cell_instr if dom == "path" else 0)
            dom_s = (split[dom + "_ms"] / steps) * 1e-3
        else:
            lane_instr, dom_s = frame_lane_instr, k_s
        achieved = lane_instr / dom_s
        exact_kernel = (not wavefront) and counted["accel_used"] == "exact"
        if exact_kernel:
            # small scenes: every (ray, object) is decided in the literal FP64 arithmetic; the kernel is bound by the
            # FP64 pipe (and, at this size, by launch latency), not by FP32 filters
            fp64_instr = counted["exact_sphere_tests"] * 20 + counted["exact_other_tests"] * 30
            roof = {
                "bound": "fp64", "achieved": fp64_instr / k_s / 1e9, "peak": peak64 / 1e9, "unit": "Glane-instr/s",
                "frac": fp64_instr / k_s / peak64, "traffic": None,
                "kernel": "render_free_kernel<EXACT>",
                "accounting": "20 FP64 instructions per ray/sphere literal test on its reject path (erl:364-378: 5 DADD/DSUB "
                              "for O-C and the sums, 15 DMUL/DADD for b, c and the discriminant) + 30 per ray/plane or "
                              "ray/triangle test, counted by an instrumented run of the same frame, divided by the frame's "
                              "CUDA-event time; hits add two square roots and two divisions that are not counted",
                "peak_source": "in-bench register-resident DFMA loop on this GPU",
                "exact_fp64_sphere_tests": int(counted["exact_sphere_tests"]),
                "exact_fp64_other_tests": int(counted["exact_other_tests"]),
                "framebuffer_gbs": (w * h * 3 / world) / k_s / 1e9,
                "note": "SURVEY 8(d) calls C2/C5 framebuffer-bound: that holds end to end (see e2e.roofline, the D2H copy); "
                        "the kernel itself writes 3 B/pixel and is nowhere near HBM",
            }
        else:
            roof = {
                "bound": "fp32", "achieved": achieved / 1e9, "peak": peak / 1e9, "unit": "Glane-instr/s",
                "frac": achieved / peak, "traffic": None,
                "kernel": ({("bvh", "path"): "wf_trace_path + wf_trace_path_refill (BVH walks of the path rays, all bounces)",
                            ("bvh", "shadow"): "wf_trace_shadow (direction grids / BVH walks of the shadow rays)",
                            ("grid", "path"): "wf_trace_path<GRID> + wf_trace_path_refill<GRID> (cell-grid walks of the path rays, all bounces)",
                            ("grid", "shadow"): "wf_trace_shadow (direction grids / BVH walks of the shadow rays)",
                            ("linear", "path"): "wf_scan<path> (brute-force filter scan of the path rays)",
                            ("linear", "shadow"): "wf_scan<shadow> (brute-force filter scan of the shadow rays)"}
                           .get((counted["accel_used"], dom), "?") if wavefront else
                           {"bvh_mega": "render_free_kernel<BVH>", "linear": "render_tiled_kernel"}.get(counted["accel_used"], "?")),
                "accounting": "6 FFMA per ray/AABB slab test + 10 FP32-pipe instr per ray/sphere filter test + 4 per "
                              "cell step (FFMA, FADD, two FMNMX) of the named kernels (counts from an instrumented run of the same frame on rank 0), divided "
                              "by their CUDA-event time in a separate pass of %d frames with one event before and after every "
                              "launch (ERT_FLAG_TIME_KERNELS; `value` is timed without those events)" % split_steps,
                "launches_per_step": (split[dom + "_launches"] / steps) if wavefront else 1,
                "avg_launch_ms": (split[dom + "_ms"] / max(split[dom + "_launches"], 1)) if wavefront else kernel_ms / steps,
                "share_of_step": (split[dom + "_ms"] / steps / split_frame_ms) if wavefront else 1.0,
                "box_tests": int(counted[dom + "_box_tests"] if wavefront else counted["box_tests"]),
                "sphere_filter_tests": int(counted[dom + "_filter_tests"] if wavefront else counted["sphere_filter_tests"]),
                "exact_fp64_sphere_tests": int(counted["exact_sphere_tests"]),
                "cell_steps": int(counted.get("cell_steps", 0)),
                "frame": {"lane_instr": int(frame_lane_instr), "frac": frame_lane_instr / k_s / peak,
                          "box_tests": int(counted["box_tests"]),
                          "sphere_filter_tests": int(counted["sphere_filter_tests"]),
                          "class_frac": {c: ((counted[c + "_box_tests"] * 6 + counted[c + "_filter_tests"] * 10
                                              + (cell_instr if c == "path" else 0))
                                             / max(split[c + "_ms"] / steps * 1e-3, 1e-12) / peak)
                                         for c in ("path", "shadow")} if wavefront else None,
                          "ms": {"path": split["path_ms"] / steps, "shadow": split["shadow_ms"] / steps,
                                 "other": split["other_ms"] / steps, "all_with_per_launch_events": split_frame_ms,
                                 "all": kernel_ms / steps}},
                "peak_source": "in-bench register-resident FFMA loop on this GPU (MEASURED_PEAKS.json has no FP32 entry); "
                               "FFMA with an immediate addend, the fastest form",
                "peak_rrr": peak_rrr / 1e9, "frac_of_peak_rrr": achieved / peak_rrr,
                "peak_rrr_source": "the same loop with three register operands per FFMA, the form the intersection "
                                   "kernels issue",
                "framebuffer_gbs": (w * h * 3 / world) / k_s / 1e9,
                "traffic_note": "dram__bytes of the named kernels are in the ncu summaries under profiles/ (r02_*_full.txt); "
                                "bench.py does not run under ncu and reports no number it did not measure",
            }
        d2h_per_gpu = (d2h_all / max(world, 1) / steps) / max(e2e_ms * 1e-3, 1e-12) / 1e9
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64 decisions+shading, f32 conservative filters", "data": "synthetic",
            "config": {
                "workload": desc, "width": w, "height": h, "depth": depth, "accel": counted["accel_used"],
                "spheres": int(len(flat.spheres)), "lights": int(len(flat.lights)),
                "rays": "unique rays (one per nearest-object scan: primary + reflection + shadow)",
                "rays_per_frame": rays_all / steps,
                "partition": ("row bands of %d rows dealt round-robin to %d GPUs" % (band_rows, world)
                              if world > 1 else "whole frame on one GPU"),
                "l2": "flushed between steps (256 MiB device write outside the timed events)",
                "timing": "value: CUDA events around the frame's launches on the launching stream, no per-launch events; "
                          "max over ranks of the per-rank sums",
                "output": "RGB8 framebuffer (min(trunc(C*255),255) fused)",
                "scene_upload_s": t_upload,
            },
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_ms,
                    "device_ms_per_step": e2e_dev_ms_max / steps,
                    "h2d_bytes_per_step": int(counted["h2d_bytes"]),
                    "d2h_bytes_per_step": int(d2h_all / steps),
                    "what": ("ert_render_async()/ert_wait() per step on two slots (two frames in flight): camera + "
                             "params in, kernel, pinned D2H of the RGB8 rows; L2 not flushed in this loop (the only "
                             "per-step data is the output frame)") if pipelined else
                            "ert_render() per step: camera + params in, kernel, pinned D2H of the RGB8 rows",
                    "frames_per_s": 1e3 / e2e_ms,
                    "d2h_gbs_per_gpu": d2h_per_gpu,
                    "roofline": {"bound": "pcie", "achieved": d2h_per_gpu, "peak": d2h_peak, "unit": "GB/s per GPU",
                                 "frac": d2h_per_gpu / max(d2h_peak, 1e-12),
                                 "peak_source": "in-bench cudaMemcpyAsync device -> pinned host of one part's bytes on this "
                                                "GPU, alone on the box",
                                 "note": "meaningful for the frames whose step is the copy (C2, C5); on C3/C4 the copy is "
                                         "a few percent of the step"}},
            "gpu_launches": launches_all,
            "reference_equivalent": {
                "ratio": refeq_ratio, "rays_per_frame": refeq_ratio * rays_all / steps,
                "Mrays_per_s": refeq_ratio * value,
                "what": "rays the reference would trace for the same frame: its lighting function re-traces the "
                        "reflection once per light (erl:216-224), so level b runs L^b times; from the per-level "
                        "counts of rank 0's part (ert_stats.bounce_path_rays / bounce_hits)"},
            "roofline": roof,
        }
        if scan is not None:
            line["roofline_scan"] = scan
        if assembled_ok is not None:
            line["config"]["assembled_frame_equals_single_gpu"] = assembled_ok
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(flat, w, h, depth)
            nx, ny = arm.sized_sample(args.cpu_budget)
            c_rays, c_dt, c_px = arm.run(nx, ny)
            line["cpu_baseline"] = {
                "value": c_rays / c_dt / 1e6, "unit": "Mrays/s", "cores": arm.cores, "kind": "port",
                "sample": "%dx%d pixel lattice (%d px) of the %dx%d frame, %.1f s" % (nx, ny, c_px, w, h, c_dt),
                "note": "C restatement of raytracer.erl (oracle/oracle.c), not BEAM: Erlang/OTP is not installed"}
        emit_line(line)

    barrier()
    for hst in hosts:
        hst.close()
    dev.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--accel", default="auto", choices=("auto", "exact", "linear", "bvh", "bvh_mega", "grid"))
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU-baseline sample at N=1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scan-roofline", action="store_true", help="skip the brute-force-scan roofline band")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the frame of the last timed step as DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU frame; --impl reference has none")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step")
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        log("bench.py: warm-up raised to 3 steps (timing rule)")
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args, rank)
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000)] + sys.argv
        return subprocess.call(cmd)
    return gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
