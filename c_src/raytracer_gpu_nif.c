/*
 * raytracer_gpu_nif.c — Erlang NIF over the C ABI of include/ert_b200.h.
 *
 * Glue only: Erlang term -> ert_scene_desc / ert_render_params -> ert_* call ->
 * Erlang term.  All logic lives behind ert_b200.h.  Every NIF that touches the
 * GPU runs on a dirty scheduler (a 4K frame blocks for milliseconds to seconds).
 * No ports, no CPU fallback: errors come back as {error, {Class, Code, Msg}}
 * and undecodable terms raise badarg.
 *
 * Written against the OTP erl_nif API without an OTP installation in this
 * image (no erl_nif.h here).  tests/mock_erl/ holds a minimal stand-in header
 * and term library so that this file is compiled and its decode/encode paths
 * are executed by the test-suite; building against a real OTP only needs
 *   gcc -shared -fPIC -I$ERL_ROOT/usr/include -Iinclude c_src/raytracer_gpu_nif.c \
 *       -Leraytracer_b200/lib -lert_b200 -o priv/raytracer_gpu.so
 *
 * Scene wire format = the record tuples scene_test pins (raytracer.erl:760-801):
 *   {camera,{vector,X,Y,Z},{vector,..},Fov,{screen,W,H}}
 *   {point_light,{colour,R,G,B},{vector,..},{colour,..}}
 *   {sphere,Radius,{vector,..},{material,{colour,..},SpecPow,Shininess,Reflectivity}}
 *   {triangle,V1,V2,V3,Material}      {plane,{vector,..},Distance,Material}
 * Numbers may be Erlang integers or floats (raytracer.erl:619-664 mixes them).
 * List elements that are none of these are skipped (raytracer.erl:357-358).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "erl_nif.h"
#include "ert_b200.h"

static ErlNifResourceType *scene_rt;
static ErlNifResourceType *frame_rt;

typedef struct {
    ert_scene *scene;
} scene_res;

/* A frame in page-locked host memory (ert_host_alloc): the GPUs copy their rows straight into it, and Erlang
 * sees it as a binary without another copy (enif_make_resource_binary keeps this resource alive). */
typedef struct {
    void *pinned;
    size_t bytes;
    int width, height, format;
} frame_res;

static void scene_dtor(ErlNifEnv *env, void *obj)
{
    scene_res *r = (scene_res *)obj;
    (void)env;
    if (r->scene) ert_scene_destroy(r->scene);
    r->scene = NULL;
}

static void frame_dtor(ErlNifEnv *env, void *obj)
{
    frame_res *r = (frame_res *)obj;
    (void)env;
    if (r->pinned) ert_host_free(r->pinned);
    r->pinned = NULL;
}

static int open_types(ErlNifEnv *env, ErlNifResourceFlags flags)
{
    scene_rt = enif_open_resource_type(env, NULL, "ert_b200_scene", scene_dtor, flags, NULL);
    frame_rt = enif_open_resource_type(env, NULL, "ert_b200_frame", frame_dtor, flags, NULL);
    return scene_rt && frame_rt ? 0 : 1;
}

static int load(ErlNifEnv *env, void **priv, ERL_NIF_TERM info)
{
    (void)priv; (void)info;
    return open_types(env, ERL_NIF_RT_CREATE);
}

/* hot code upgrade: the resource types exist already and are taken over by the new module instance */
static int upgrade(ErlNifEnv *env, void **priv, void **old_priv, ERL_NIF_TERM info)
{
    (void)priv; (void)old_priv; (void)info;
    return open_types(env, (ErlNifResourceFlags)(ERL_NIF_RT_CREATE | ERL_NIF_RT_TAKEOVER));
}

/* ---- term helpers --------------------------------------------------------- */
static int is_atom_named(ErlNifEnv *env, ERL_NIF_TERM t, const char *name)
{
    char buf[32];
    if (!enif_is_atom(env, t)) return 0;
    if (enif_get_atom(env, t, buf, sizeof buf, ERL_NIF_LATIN1) <= 0) return 0;
    return strcmp(buf, name) == 0;
}

/* enif_get_double fails on integers: try both */
static int get_number(ErlNifEnv *env, ERL_NIF_TERM t, double *out)
{
    ErlNifSInt64 i;
    if (enif_get_double(env, t, out)) return 1;
    if (enif_get_int64(env, t, &i)) { *out = (double)i; return 1; }
    return 0;
}

/* {Tag, A, B, C} */
static int get_tagged3(ErlNifEnv *env, ERL_NIF_TERM t, const char *tag, double out[3])
{
    int arity;
    const ERL_NIF_TERM *e;
    if (!enif_get_tuple(env, t, &arity, &e) || arity != 4 || !is_atom_named(env, e[0], tag)) return 0;
    return get_number(env, e[1], &out[0]) && get_number(env, e[2], &out[1]) && get_number(env, e[3], &out[2]);
}

static int get_material(ErlNifEnv *env, ERL_NIF_TERM t, ert_material *m)
{
    int arity;
    const ERL_NIF_TERM *e;
    if (!enif_get_tuple(env, t, &arity, &e) || arity != 5 || !is_atom_named(env, e[0], "material")) return 0;
    return get_tagged3(env, e[1], "colour", m->colour) && get_number(env, e[2], &m->specular_power) &&
           get_number(env, e[3], &m->shininess) && get_number(env, e[4], &m->reflectivity);
}

static int get_camera(ErlNifEnv *env, ERL_NIF_TERM t, ert_camera *c)
{
    int arity, sa;
    const ERL_NIF_TERM *e, *s;
    if (!enif_get_tuple(env, t, &arity, &e) || arity != 5 || !is_atom_named(env, e[0], "camera")) return 0;
    if (!get_tagged3(env, e[1], "vector", c->location) || !get_tagged3(env, e[2], "vector", c->rotation) ||
        !get_number(env, e[3], &c->fov))
        return 0;
    if (!enif_get_tuple(env, e[4], &sa, &s) || sa != 3 || !is_atom_named(env, s[0], "screen")) return 0;
    return get_number(env, s[1], &c->screen_width) && get_number(env, s[2], &c->screen_height);
}

typedef struct {
    ert_scene_desc desc;
    ert_point_light *lights;
    ert_sphere *spheres;
    ert_triangle *triangles;
    ert_plane *planes;
} decoded_scene;

static void decoded_free(decoded_scene *d)
{
    free(d->lights); free(d->spheres); free(d->triangles); free(d->planes);
    memset(d, 0, sizeof *d);
}

/* [Camera | Rest] (raytracer.erl:180) -> tables; returns 1 on success, 0 => badarg */
static int decode_scene(ErlNifEnv *env, ERL_NIF_TERM list, decoded_scene *d)
{
    unsigned len;
    ERL_NIF_TERM head, tail;
    int32_t order = 0;
    memset(d, 0, sizeof *d);
    if (!enif_get_list_length(env, list, &len) || len == 0) return 0;
    if (!enif_get_list_cell(env, list, &head, &tail) || !get_camera(env, head, &d->desc.camera)) return 0;
    {
        /* first pass: how many records of each kind (by tag and arity), so that every table is allocated at its
         * size — a 1 M-sphere list would otherwise pay for four full-length tables */
        size_t nl = 0, ns = 0, nt = 0, np = 0;
        ERL_NIF_TERM h2, t2 = tail;
        while (enif_get_list_cell(env, t2, &h2, &t2)) {
            int arity;
            const ERL_NIF_TERM *e;
            if (!enif_get_tuple(env, h2, &arity, &e) || arity < 1) continue;
            if (arity == 4 && is_atom_named(env, e[0], "point_light")) nl++;
            else if (arity == 4 && is_atom_named(env, e[0], "sphere")) ns++;
            else if (arity == 5 && is_atom_named(env, e[0], "triangle")) nt++;
            else if (arity == 4 && is_atom_named(env, e[0], "plane")) np++;
        }
        d->lights = calloc(nl ? nl : 1, sizeof *d->lights);
        d->spheres = calloc(ns ? ns : 1, sizeof *d->spheres);
        d->triangles = calloc(nt ? nt : 1, sizeof *d->triangles);
        d->planes = calloc(np ? np : 1, sizeof *d->planes);
    }
    if (!d->lights || !d->spheres || !d->triangles || !d->planes) { decoded_free(d); return 0; }
    while (enif_get_list_cell(env, tail, &head, &tail)) {
        int arity;
        const ERL_NIF_TERM *e;
        int32_t pos = order++;
        if (!enif_get_tuple(env, head, &arity, &e) || arity < 1) continue;          /* unknown element */
        if (arity == 4 && is_atom_named(env, e[0], "point_light")) {
            ert_point_light *l = &d->lights[d->desc.n_lights];
            if (!get_tagged3(env, e[1], "colour", l->diffuse_colour) || !get_tagged3(env, e[2], "vector", l->location) ||
                !get_tagged3(env, e[3], "colour", l->specular_colour))
                goto bad;
            l->order = pos;
            d->desc.n_lights++;
        } else if (arity == 4 && is_atom_named(env, e[0], "sphere")) {
            ert_sphere *s = &d->spheres[d->desc.n_spheres];
            if (!get_number(env, e[1], &s->radius) || !get_tagged3(env, e[2], "vector", s->center) ||
                !get_material(env, e[3], &s->material))
                goto bad;
            s->order = pos;
            d->desc.n_spheres++;
        } else if (arity == 5 && is_atom_named(env, e[0], "triangle")) {
            ert_triangle *t = &d->triangles[d->desc.n_triangles];
            if (!get_tagged3(env, e[1], "vector", t->v1) || !get_tagged3(env, e[2], "vector", t->v2) ||
                !get_tagged3(env, e[3], "vector", t->v3) || !get_material(env, e[4], &t->material))
                goto bad;
            t->order = pos;
            d->desc.n_triangles++;
        } else if (arity == 4 && is_atom_named(env, e[0], "plane")) {
            ert_plane *p = &d->planes[d->desc.n_planes];
            if (!get_tagged3(env, e[1], "vector", p->normal) || !get_number(env, e[2], &p->distance) ||
                !get_material(env, e[3], &p->material))
                goto bad;
            p->order = pos;
            d->desc.n_planes++;
        }
        /* any other tuple: neither object nor light, skipped like erl:357-358 / 248-249 */
    }
    d->desc.lights = d->lights;
    d->desc.spheres = d->spheres;
    d->desc.triangles = d->triangles;
    d->desc.planes = d->planes;
    return 1;
bad:
    decoded_free(d);
    return 0;
}

static ERL_NIF_TERM make_error(ErlNifEnv *env, int code)
{
    const char *cls = code == ERT_ERR_NO_DEVICE ? "no_device" : code == ERT_ERR_CUDA ? "cuda" :
                      code == ERT_ERR_NOMEM ? "nomem" : "badarg";
    return enif_make_tuple2(env, enif_make_atom(env, "error"),
                            enif_make_tuple3(env, enif_make_atom(env, cls), enif_make_int(env, code),
                                             enif_make_string(env, ert_last_error(), ERL_NIF_LATIN1)));
}

/* ---- NIFs ------------------------------------------------------------------ */
/* device_count() -> {ok, N} | {error, _} */
static ERL_NIF_TERM nif_device_count(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    int n = 0, rc;
    (void)argc; (void)argv;
    rc = ert_device_count(&n);
    if (rc != ERT_OK) return make_error(env, rc);
    return enif_make_tuple2(env, enif_make_atom(env, "ok"), enif_make_int(env, n));
}

/* scene_info(Scene) -> {NLights, NSpheres, NTriangles, NPlanes}; badarg on malformed scenes.
 * Needs no GPU: lets the host validate a scene term. */
static ERL_NIF_TERM nif_scene_info(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    decoded_scene d;
    ERL_NIF_TERM out;
    (void)argc;
    if (!decode_scene(env, argv[0], &d)) return enif_make_badarg(env);
    out = enif_make_tuple4(env, enif_make_int64(env, d.desc.n_lights), enif_make_int64(env, d.desc.n_spheres),
                           enif_make_int64(env, d.desc.n_triangles), enif_make_int64(env, d.desc.n_planes));
    decoded_free(&d);
    return out;
}

/* scene_upload(Scene, Device) -> {ok, Handle} | {error, _}   (dirty) */
static ERL_NIF_TERM nif_scene_upload(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    decoded_scene d;
    int device, rc;
    ert_scene *scene = NULL;
    scene_res *res;
    ERL_NIF_TERM term;
    (void)argc;
    if (!enif_get_int(env, argv[1], &device)) return enif_make_badarg(env);
    if (!decode_scene(env, argv[0], &d)) return enif_make_badarg(env);
    rc = ert_scene_create(&d.desc, device, &scene);
    decoded_free(&d);
    if (rc == ERT_ERR_BADARG) return enif_make_badarg(env);
    if (rc != ERT_OK) return make_error(env, rc);
    res = enif_alloc_resource(scene_rt, sizeof *res);
    if (!res) { ert_scene_destroy(scene); return make_error(env, ERT_ERR_NOMEM); }
    res->scene = scene;
    term = enif_make_resource(env, res);
    enif_release_resource(res);
    return enif_make_tuple2(env, enif_make_atom(env, "ok"), term);
}

/* scene_clone(Handle, Device) -> {ok, Handle2} | {error, _}   (dirty)
 * The flattened scene and its acceleration structures are copied to another GPU without rebuilding them
 * (ert_scene_clone): one upload + N-1 clones instead of N uploads of the same term. */
static ERL_NIF_TERM nif_scene_clone(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    scene_res *src, *res;
    ert_scene *scene = NULL;
    ERL_NIF_TERM term;
    int device, rc;
    (void)argc;
    if (!enif_get_resource(env, argv[0], scene_rt, (void **)&src) || !src->scene) return enif_make_badarg(env);
    if (!enif_get_int(env, argv[1], &device)) return enif_make_badarg(env);
    rc = ert_scene_clone(src->scene, device, &scene);
    if (rc == ERT_ERR_BADARG) return enif_make_badarg(env);
    if (rc != ERT_OK) return make_error(env, rc);
    res = enif_alloc_resource(scene_rt, sizeof *res);
    if (!res) { ert_scene_destroy(scene); return make_error(env, ERT_ERR_NOMEM); }
    res->scene = scene;
    term = enif_make_resource(env, res);
    enif_release_resource(res);
    return enif_make_tuple2(env, enif_make_atom(env, "ok"), term);
}

/* Opts: proplist of {format, rgb8|f32|f64} | {accel, auto|exact|linear|bvh|bvh_mega|grid} |
 *       {part, {BandRows, NParts, Part}} | {camera, CameraRecord} |
 *       {supersample, N}: N x N rays per pixel, box-filtered, N an integer in 1..ERT_MAX_SUPERSAMPLE (8) |
 *       {camera_rotation, true | false}: turn the primary rays by the camera's rotation (ERT_FLAG_CAMERA_ROTATION) */
static int decode_opts(ErlNifEnv *env, ERL_NIF_TERM opts, ert_render_params *p, ert_camera *cam)
{
    ERL_NIF_TERM head, tail = opts;
    while (enif_get_list_cell(env, tail, &head, &tail)) {
        int arity;
        const ERL_NIF_TERM *e;
        if (!enif_get_tuple(env, head, &arity, &e) || arity != 2) return 0;
        if (is_atom_named(env, e[0], "format")) {
            if (is_atom_named(env, e[1], "rgb8")) p->format = ERT_FMT_RGB8;
            else if (is_atom_named(env, e[1], "f32")) p->format = ERT_FMT_F32;
            else if (is_atom_named(env, e[1], "f64")) p->format = ERT_FMT_F64;
            else return 0;
        } else if (is_atom_named(env, e[0], "accel")) {
            if (is_atom_named(env, e[1], "auto")) p->accel = ERT_ACCEL_AUTO;
            else if (is_atom_named(env, e[1], "exact")) p->accel = ERT_ACCEL_EXACT;
            else if (is_atom_named(env, e[1], "linear")) p->accel = ERT_ACCEL_LINEAR;
            else if (is_atom_named(env, e[1], "bvh")) p->accel = ERT_ACCEL_BVH;
            else if (is_atom_named(env, e[1], "bvh_mega")) p->accel = ERT_ACCEL_BVH_MEGAKERNEL;
            else if (is_atom_named(env, e[1], "grid")) p->accel = ERT_ACCEL_GRID;
            else return 0;
        } else if (is_atom_named(env, e[0], "part")) {
            int a3;
            const ERL_NIF_TERM *q;
            if (!enif_get_tuple(env, e[1], &a3, &q) || a3 != 3) return 0;
            if (!enif_get_int(env, q[0], &p->band_rows) || !enif_get_int(env, q[1], &p->n_parts) ||
                !enif_get_int(env, q[2], &p->part))
                return 0;
        } else if (is_atom_named(env, e[0], "supersample")) {
            if (!enif_get_int(env, e[1], &p->supersample) || p->supersample < 1 || p->supersample > ERT_MAX_SUPERSAMPLE)
                return 0;
        } else if (is_atom_named(env, e[0], "camera_rotation")) {
            if (is_atom_named(env, e[1], "true")) p->flags |= ERT_FLAG_CAMERA_ROTATION;
            else if (is_atom_named(env, e[1], "false")) p->flags &= ~ERT_FLAG_CAMERA_ROTATION;
            else return 0;
        } else if (is_atom_named(env, e[0], "camera")) {
            if (!get_camera(env, e[1], cam)) return 0;
            p->camera = cam;
        } else {
            return 0;
        }
    }
    return enif_is_empty_list(env, tail);
}

static size_t elem_size(int format) { return format == ERT_FMT_RGB8 ? 1 : format == ERT_FMT_F32 ? 4 : 8; }

static int decode_render_args(ErlNifEnv *env, const ERL_NIF_TERM argv[], scene_res **res, ert_render_params *p,
                              ert_camera *cam)
{
    memset(p, 0, sizeof *p);
    if (!enif_get_resource(env, argv[0], scene_rt, (void **)res) || !(*res)->scene) return 0;
    if (!enif_get_int(env, argv[1], &p->width) || !enif_get_int(env, argv[2], &p->height) ||
        !enif_get_int(env, argv[3], &p->depth))
        return 0;
    p->format = ERT_FMT_RGB8;
    p->accel = ERT_ACCEL_AUTO;
    p->n_parts = 1;
    return decode_opts(env, argv[4], p, cam);
}

static frame_res *frame_new(int width, int height, int format)
{
    frame_res *fr = enif_alloc_resource(frame_rt, sizeof *fr);
    if (!fr) return NULL;
    fr->pinned = NULL;
    fr->width = width; fr->height = height; fr->format = format;
    fr->bytes = (size_t)width * (size_t)height * 3 * elem_size(format);
    if (ert_host_alloc(fr->bytes, &fr->pinned) != ERT_OK) {
        enif_release_resource(fr);             /* runs frame_dtor with pinned == NULL */
        return NULL;
    }
    memset(fr->pinned, 0, fr->bytes);
    return fr;
}

/* render(Handle, Width, Height, Depth, Opts) -> {ok, FrameBinary} | {error, _}   (dirty)
 * The binary is the full row-major frame (Y = 0 first), 3 channels per pixel.  It is a resource binary over
 * page-locked memory: the rows arrive by asynchronous D2H copies and Erlang gets them without a further copy. */
static ERL_NIF_TERM nif_render(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    scene_res *res;
    ert_render_params p;
    ert_camera cam;
    frame_res *fr;
    ERL_NIF_TERM bin;
    int rc;
    (void)argc;
    if (!decode_render_args(env, argv, &res, &p, &cam)) return enif_make_badarg(env);
    if (p.width <= 0 || p.height <= 0 || p.depth < 0) return enif_make_badarg(env);   /* guards erl:89 */
    fr = frame_new(p.width, p.height, p.format);
    if (!fr) return make_error(env, ERT_ERR_NOMEM);
    rc = ert_render(res->scene, &p, fr->pinned, fr->bytes);
    if (rc != ERT_OK) {
        enif_release_resource(fr);
        return rc == ERT_ERR_BADARG ? enif_make_badarg(env) : make_error(env, rc);
    }
    bin = enif_make_resource_binary(env, fr, fr->pinned, fr->bytes);
    enif_release_resource(fr);                 /* the binary term holds the remaining reference */
    return enif_make_tuple2(env, enif_make_atom(env, "ok"), bin);
}

/* frame_alloc(Width, Height, Format) -> {ok, Frame} | {error, _}
 * One page-locked frame that several renders (one per GPU, each with its {part, ...} option) fill in place. */
static ERL_NIF_TERM nif_frame_alloc(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    int w, h, format;
    frame_res *fr;
    ERL_NIF_TERM term;
    (void)argc;
    if (!enif_get_int(env, argv[0], &w) || !enif_get_int(env, argv[1], &h) || w <= 0 || h <= 0) return enif_make_badarg(env);
    if (is_atom_named(env, argv[2], "rgb8")) format = ERT_FMT_RGB8;
    else if (is_atom_named(env, argv[2], "f32")) format = ERT_FMT_F32;
    else if (is_atom_named(env, argv[2], "f64")) format = ERT_FMT_F64;
    else return enif_make_badarg(env);
    fr = frame_new(w, h, format);
    if (!fr) return make_error(env, ERT_ERR_NOMEM);
    term = enif_make_resource(env, fr);
    enif_release_resource(fr);
    return enif_make_tuple2(env, enif_make_atom(env, "ok"), term);
}

/* render_into(Handle, Frame, Depth, Opts) -> ok | {error, _}   (dirty)
 * Renders this call's part ({part, {BandRows, NParts, Part}}) of the frame's size and format; its rows land at
 * their place in Frame.  Calls for different parts may run at the same time from different processes. */
static ERL_NIF_TERM nif_render_into(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    scene_res *res;
    frame_res *fr;
    ert_render_params p;
    ert_camera cam;
    int rc;
    (void)argc;
    memset(&p, 0, sizeof p);
    if (!enif_get_resource(env, argv[0], scene_rt, (void **)&res) || !res->scene) return enif_make_badarg(env);
    if (!enif_get_resource(env, argv[1], frame_rt, (void **)&fr) || !fr->pinned) return enif_make_badarg(env);
    if (!enif_get_int(env, argv[2], &p.depth) || p.depth < 0) return enif_make_badarg(env);
    p.width = fr->width; p.height = fr->height;
    p.format = fr->format;
    p.accel = ERT_ACCEL_AUTO;
    p.n_parts = 1;
    if (!decode_opts(env, argv[3], &p, &cam) || p.format != fr->format) return enif_make_badarg(env);
    rc = ert_render(res->scene, &p, fr->pinned, fr->bytes);
    if (rc == ERT_ERR_BADARG) return enif_make_badarg(env);
    if (rc != ERT_OK) return make_error(env, rc);
    return enif_make_atom(env, "ok");
}

/* frame_binary(Frame) -> Binary: the frame's memory as a binary, no copy */
static ERL_NIF_TERM nif_frame_binary(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    frame_res *fr;
    (void)argc;
    if (!enif_get_resource(env, argv[0], frame_rt, (void **)&fr) || !fr->pinned) return enif_make_badarg(env);
    return enif_make_resource_binary(env, fr, fr->pinned, fr->bytes);
}

/* render_pixel_list(Handle, Width, Height, Depth, Opts) -> [{Index, {R,G,B}}] | {error, _}   (dirty)
 * The reference's own return type (raytracer.erl:86-99): unclamped floats, row-major,
 * Index = X + Y*Width as the concurrent driver numbers pixels (erl:112).  For small images:
 * the list costs ~100 bytes of BEAM heap per pixel. */
static ERL_NIF_TERM nif_render_pixel_list(ErlNifEnv *env, int argc, const ERL_NIF_TERM argv[])
{
    scene_res *res;
    ert_render_params p;
    ert_camera cam;
    double *buf;
    size_t n, bytes;
    ERL_NIF_TERM list;
    int rc;
    (void)argc;
    if (!decode_render_args(env, argv, &res, &p, &cam)) return enif_make_badarg(env);
    if (p.width <= 0 || p.height <= 0 || p.depth < 0) return enif_make_badarg(env);
    p.format = ERT_FMT_F64;
    n = (size_t)p.width * (size_t)p.height;
    bytes = n * 3 * sizeof(double);
    buf = malloc(bytes);
    if (!buf) return make_error(env, ERT_ERR_NOMEM);
    rc = ert_render(res->scene, &p, buf, bytes);
    if (rc != ERT_OK) {
        free(buf);
        return rc == ERT_ERR_BADARG ? enif_make_badarg(env) : make_error(env, rc);
    }
    {
        /* BEAM floats are finite (an overflow is badarith in the reference): a non-finite channel cannot be a term */
        size_t k;
        for (k = 0; k < 3 * n; k++) {
            if (!(buf[k] - buf[k] == 0.0)) {
                free(buf);
                return enif_make_tuple2(env, enif_make_atom(env, "error"),
                                        enif_make_tuple2(env, enif_make_atom(env, "badarith"),
                                                         enif_make_int64(env, (ErlNifSInt64)(k / 3))));
            }
        }
    }
    list = enif_make_list(env, 0);
    while (n-- > 0) {
        ERL_NIF_TERM px = enif_make_tuple3(env, enif_make_double(env, buf[3 * n]), enif_make_double(env, buf[3 * n + 1]),
                                           enif_make_double(env, buf[3 * n + 2]));
        list = enif_make_list_cell(env, enif_make_tuple2(env, enif_make_int64(env, (ErlNifSInt64)n), px), list);
    }
    free(buf);
    return list;
}

static ErlNifFunc nif_funcs[] = {
    {"device_count", 0, nif_device_count, 0},
    {"scene_info", 1, nif_scene_info, 0},
    /* scene_upload builds the BVH and the grids on the host: CPU-bound; the others wait for the GPU: IO-bound */
    {"scene_upload", 2, nif_scene_upload, ERL_NIF_DIRTY_JOB_CPU_BOUND},
    {"scene_clone", 2, nif_scene_clone, ERL_NIF_DIRTY_JOB_IO_BOUND},
    {"render", 5, nif_render, ERL_NIF_DIRTY_JOB_IO_BOUND},
    {"render_pixel_list", 5, nif_render_pixel_list, ERL_NIF_DIRTY_JOB_IO_BOUND},
    {"frame_alloc", 3, nif_frame_alloc, ERL_NIF_DIRTY_JOB_IO_BOUND},
    {"render_into", 4, nif_render_into, ERL_NIF_DIRTY_JOB_IO_BOUND},
    {"frame_binary", 1, nif_frame_binary, 0},
};

ERL_NIF_INIT(raytracer_gpu, nif_funcs, load, NULL, upgrade, NULL)
