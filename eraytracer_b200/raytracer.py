"""Host-side mirror of raytracer.erl's entry points with a GPU tracing function.

Erlang/OTP is not in this image, so the host side above the C ABI is written in
Python with the reference's names, argument meaning and error behaviour; the
Erlang module + NIF a maintainer would add are in erl/ and c_src/ (INTEGRATION.md).

The seam is the 4-arity tracing function (raytracer.erl:714-719, 728-732):
    Fun(Width, Height, Scene, Recursion_depth) -> [{Index, {R, G, B}}]
`raytraced_pixel_list_gpu/4` is that function; everything it does happens in
libert_b200.so on a B200.  There is no CPU fallback here: the reference's
simple/concurrent/distributed drivers stay in the Erlang host.
"""
import time

import numpy as np

from . import _lib
from . import scene as _scene
from .ppm import write_pixels_to_ppm, write_frame_to_ppm  # noqa: F401  (re-exported)


def scene():
    """scene/0, raytracer.erl:618-665."""
    return _scene.demo_scene()


def _function_clause(name, args):
    # what BEAM raises when no clause of a function matches (guards at erl:89)
    raise ValueError("function_clause: no clause of %s matches %r" % (name, args))


def render_frame(width, height, scene_list, recursion_depth, fmt="f64", accel="auto", device=0, supersample=1,
                 camera_rotation=False):
    """Renders one frame on one GPU; returns (frame[H,W,3], stats).  supersample=N box-filters N x N rays per
    pixel: the pixels of the (N*width) x (N*height) frame that fall in it.  camera_rotation=True turns the primary
    rays by the camera's rotation, which the reference ignores (ERT_FLAG_CAMERA_ROTATION)."""
    flat = scene_list if isinstance(scene_list, _scene.FlatScene) else _scene.flatten(scene_list)
    dev_scene = flat.upload(device)
    try:
        return dev_scene.render(width, height, recursion_depth, fmt=fmt, accel=accel, supersample=supersample,
                                camera_rotation=camera_rotation)
    finally:
        dev_scene.close()


def render_frame_multi_gpu(width, height, scene_list, recursion_depth, fmt="f64", accel="auto",
                           devices=None, band_rows=16, supersample=1, camera_rotation=False):
    """One frame split into row bands dealt round-robin to the GPUs of this box
    (the row-band mapping of distribute_work/7, raytracer.erl:139-149).  Every GPU copies
    its bands straight into one pinned host frame; there is no gather step."""
    n_dev = _lib.device_count()
    devices = list(range(n_dev)) if devices is None else list(devices)
    if not devices:
        raise _lib.ErtError(_lib.ERT_ERR_NO_DEVICE, "no CUDA device is visible")
    flat = scene_list if isinstance(scene_list, _scene.FlatScene) else _scene.flatten(scene_list)
    code = _lib.FORMATS[fmt]
    dt = np.dtype(_lib.FORMAT_DTYPES[code])
    nbytes = width * height * 3 * dt.itemsize
    pinned = _lib.PinnedFrame(nbytes)
    scenes = []
    try:
        first = flat.upload(devices[0])
        scenes.append(first)
        for d in devices[1:]:
            scenes.append(first.clone(d))
        for part, sc in enumerate(scenes):
            sc.render_async(width, height, recursion_depth, slot=0, fmt=fmt, accel=accel,
                            band_rows=band_rows, n_parts=len(scenes), part=part,
                            host_ptr=pinned.ptr, host_bytes=nbytes, supersample=supersample,
                            camera_rotation=camera_rotation)
        for sc in scenes:
            sc.wait(0)
        stats = [sc.stats(0) for sc in scenes]
        frame = pinned.array(dt, (height, width, 3)).copy()
        return frame, stats
    finally:
        for sc in scenes:
            sc.close()
        pinned.close()


def _pixel_list(frame):
    h, w, _ = frame.shape
    flat = frame.reshape(-1, 3).tolist()
    # Index as the concurrent/distributed drivers number pixels: X + Y*Width (erl:112, 173);
    # the list is already in that order, which is what the writer needs (erl:667).
    return [(i, (p[0], p[1], p[2])) for i, p in enumerate(flat)]


def raytraced_pixel_list_gpu(width, height, scene_list, recursion_depth):
    """The GPU tracing function: same contract as raytraced_pixel_list_simple/4
    (raytracer.erl:86-99).  Returns unclamped float triples in row-major order."""
    if width == 0 and height == 0:
        return 'done'                                   # erl:86-87
    if not (isinstance(width, int) and isinstance(height, int) and width > 0 and height > 0):
        _function_clause('raytraced_pixel_list_gpu/4', (width, height))
    frame, _ = render_frame(width, height, scene_list, recursion_depth, fmt="f64")
    return _pixel_list(frame)


def raytraced_pixel_list_gpu_distributed(width, height, scene_list, recursion_depth):
    """Row bands over every GPU of the box (the role of raytraced_pixel_list_distributed/4,
    raytracer.erl:121-137)."""
    if width == 0 and height == 0:
        return 'done'
    if not (isinstance(width, int) and isinstance(height, int) and width > 0 and height > 0):
        _function_clause('raytraced_pixel_list_gpu_distributed/4', (width, height))
    frame, _ = render_frame_multi_gpu(width, height, scene_list, recursion_depth, fmt="f64")
    return _pixel_list(frame)


def tracing_function(strategy):
    """tracing_function/1, raytracer.erl:714-719, with the GPU strategies added."""
    if strategy == 'gpu':
        return raytraced_pixel_list_gpu
    if strategy == 'gpu_distributed':
        return raytraced_pixel_list_gpu_distributed
    if strategy in ('simple', 'concurrent', 'distributed'):
        raise NotImplementedError(
            "strategy %r is the reference's CPU driver and stays in the Erlang host "
            "(raytracer.erl:86-178); this package only provides 'gpu' and 'gpu_distributed'"
            % (strategy,))
    _function_clause('tracing_function/1', (strategy,))


def raytrace(*args):
    """raytrace/1 and raytrace/5, raytracer.erl:721-733."""
    if len(args) == 1:
        return raytrace(4, 3, "/tmp/traced.ppm", 5, args[0])
    if len(args) != 5:
        _function_clause('raytrace', args)
    width, height, filename, recursion_depth, function = args
    return write_pixels_to_ppm(width, height, 255,
                               function(width, height, scene(), recursion_depth), filename)


def go(*args):
    """go/1 and go/5, raytracer.erl:707-712."""
    if len(args) == 1:
        return raytrace(tracing_function(args[0]))
    if len(args) != 5:
        _function_clause('go', args)
    width, height, filename, recursion_depth, strategy = args
    return raytrace(width, height, filename, recursion_depth, tracing_function(strategy))


def standalone(*args):
    """standalone/1 (list of strings, as `erl -run` passes them) and standalone/5,
    raytracer.erl:688-705.  Does not halt the interpreter."""
    if len(args) == 1:
        width, height, filename, recursion_depth, strategy = args[0]
        return standalone(int(width), int(height), filename, int(recursion_depth),
                          tracing_function(strategy))
    if len(args) != 5:
        _function_clause('standalone', args)
    width, height, filename, recursion_depth, function = args
    t0 = time.perf_counter()
    raytrace(width, height, filename, recursion_depth, function)
    print("Done in %s seconds" % (time.perf_counter() - t0))
    return 'ok'
