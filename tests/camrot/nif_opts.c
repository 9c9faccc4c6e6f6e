/* The NIF (c_src/raytracer_gpu_nif.c, included unchanged) with its Opts decoder exported, so that the decoding of
 * {camera_rotation, Bool} can be checked without a device (tests/test_camera_rotation_host.py). */
#include "../../c_src/raytracer_gpu_nif.c"

/* 1 and the render params' flags, or 0 for badarg */
int camrot_decode_opts(ErlNifEnv *env, ERL_NIF_TERM opts, unsigned *flags)
{
    ert_render_params p;
    ert_camera cam;
    memset(&p, 0, sizeof p);
    if (!decode_opts(env, opts, &p, &cam)) return 0;
    *flags = p.flags;
    return 1;
}
