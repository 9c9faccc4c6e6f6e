"""CPU checks of the supersampling interface: the header's field and the Python binding agree, the struct keeps its
size and layout, and every Python entry point renders one sample per pixel unless asked for more."""
import ctypes
import inspect
import os
import subprocess

from eraytracer_b200 import _lib, raytracer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_supersample_field_matches_the_header(tmp_path):
    src = tmp_path / "ss_layout.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "ert_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %d\n", offsetof(ert_render_params, supersample), sizeof(((ert_render_params *)0)->supersample),
         offsetof(ert_render_params, flags), sizeof(ert_render_params), ERT_MAX_SUPERSAMPLE);
  return 0; }''')
    exe = tmp_path / "ss_layout"
    subprocess.check_call(["gcc", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    off, size, flags_off, total, max_ss = map(int, subprocess.check_output([str(exe)], text=True).split())
    assert off == _lib.RenderParams.supersample.offset
    assert size == 4
    # the field took the place of the reserved int32 after `flags`: size and layout of the struct are unchanged
    assert off == flags_off + 4 == 36
    assert total == ctypes.sizeof(_lib.RenderParams) == 48
    assert max_ss == _lib.MAX_SUPERSAMPLE == 8
    assert [n for n, _ in _lib.RenderParams._fields_] == ["width", "height", "depth", "format", "accel", "band_rows",
                                                         "n_parts", "part", "flags", "supersample", "camera"]


def test_python_entry_points_default_to_one_sample():
    for fn in (_lib.Scene.render, _lib.Scene.render_async, raytracer.render_frame, raytracer.render_frame_multi_gpu):
        assert inspect.signature(fn).parameters["supersample"].default == 1, fn.__qualname__
    # the 4-arity tracing functions are the reference's contract: one ray per pixel, no option
    for fn in (raytracer.raytraced_pixel_list_gpu, raytracer.raytraced_pixel_list_gpu_distributed):
        assert list(inspect.signature(fn).parameters) == ["width", "height", "scene_list", "recursion_depth"]


def test_params_carry_the_sample_count():
    s = _lib.Scene(None, 0)
    for n in (0, 1, 2, 8):
        p = s._params(16, 8, 1, "rgb8", "auto", 0, 1, 0, 0, None, n)
        assert p.supersample == n
