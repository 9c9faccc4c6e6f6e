/*
 * ert_b200.h — C ABI of the B200-native eraytracer hot path.
 *
 * This is the drop-in boundary for ONE path of plouj/eraytracer: the per-pixel
 * render that raytracer.erl reaches through its 4-arity "tracing function"
 *     Fun(Width, Height, Scene, Recursion_depth) -> [{Index, {R,G,B}}]
 * (selected in tracing_function/1, raytracer.erl:714-719, called from
 * raytrace/5, raytracer.erl:723-733).  Everything below that call —
 * trace_ray_through_pixel/3 (180-184) down to the vector primitives (524-573)
 * — runs in hand-written sm_100a CUDA kernels behind these entry points.
 * Scene construction, the drivers and the PPM writer stay on the host.
 *
 * The shared object (libert_b200.so) has no CPU fallback: every entry point
 * that needs a GPU returns ERT_ERR_NO_DEVICE / ERT_ERR_CUDA when none works.
 *
 * Structs mirror the reference's records (raytracer.erl:72-81) field by field,
 * as doubles (Erlang numbers; integers are promoted by the caller).  `order`
 * is the element's zero-based position in the scene list AFTER the camera
 * (raytracer.erl:180 pops the camera): it carries the two order-dependent
 * rules of the reference through the flattening — the earlier list element
 * wins equal distances (strict '>' at raytracer.erl:319) and lights are folded
 * in list order (raytracer.erl:211-252).
 */
#ifndef ERT_B200_H
#define ERT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ERT_ABI_VERSION 3

#if defined(__GNUC__)
#define ERT_API __attribute__((visibility("default")))
#else
#define ERT_API
#endif

/* ---- status codes (every function returns one) -------------------------- */
#define ERT_OK             0
#define ERT_ERR_BADARG     1   /* malformed scene/params: the NIF raises badarg */
#define ERT_ERR_NO_DEVICE  2   /* no usable CUDA device; there is no CPU fallback */
#define ERT_ERR_CUDA       3   /* a CUDA call failed; see ert_last_error() */
#define ERT_ERR_NOMEM      4

/* ---- records (raytracer.erl:72-81) -------------------------------------- */
typedef struct ert_material {      /* -record(material, ...) erl:77 */
    double colour[3];
    double specular_power;
    double shininess;
    double reflectivity;
} ert_material;

typedef struct ert_camera {        /* -record(camera, ...) erl:76, screen erl:75 */
    double location[3];
    double rotation[3];            /* degrees; ignored like erl:487 unless ERT_FLAG_CAMERA_ROTATION is set */
    double fov;                    /* degrees */
    double screen_width;
    double screen_height;
} ert_camera;

typedef struct ert_point_light {   /* erl:81 */
    double diffuse_colour[3];
    double location[3];
    double specular_colour[3];
    int32_t order;
    int32_t reserved;
} ert_point_light;

typedef struct ert_sphere {        /* erl:78 */
    double radius;
    double center[3];
    ert_material material;
    int32_t order;
    int32_t reserved;
} ert_sphere;

typedef struct ert_triangle {      /* erl:79 */
    double v1[3], v2[3], v3[3];
    ert_material material;
    int32_t order;
    int32_t reserved;
} ert_triangle;

typedef struct ert_plane {         /* erl:80 */
    double normal[3];
    double distance;
    ert_material material;
    int32_t order;
    int32_t reserved;
} ert_plane;

/* The scene list of scene/0 (erl:618-665), camera split off, one table per
 * record kind.  Elements that are none of these kinds (the reference skips
 * them, erl:357-358 and erl:248-249) are simply not listed; their list
 * positions stay unused in `order`. */
typedef struct ert_scene_desc {
    ert_camera camera;
    int64_t n_lights;     const ert_point_light *lights;
    int64_t n_spheres;    const ert_sphere *spheres;
    int64_t n_triangles;  const ert_triangle *triangles;
    int64_t n_planes;     const ert_plane *planes;
} ert_scene_desc;

/* ---- render call --------------------------------------------------------- */
/* Output formats.  All are row-major, Y=0 first (erl:90-99), 3 channels. */
#define ERT_FMT_RGB8  0   /* uint8: min(trunc(C*255),255) fused (erl:678-680); <0 clamps to 0 */
#define ERT_FMT_F32   1   /* float: unclamped colour rounded to binary32 */
#define ERT_FMT_F64   2   /* double: unclamped colour, what colour_to_pixel returns (erl:613) */

/* Nearest-hit strategies.  All return the reference's linear-scan result
 * (erl:300-346): minimum distance, earlier list element on ties. */
#define ERT_ACCEL_AUTO    0
#define ERT_ACCEL_EXACT   1   /* FP64 scan of every object, scene read through the constant/L1 path */
#define ERT_ACCEL_LINEAR  2   /* FP32 conservative filter over shared-memory sphere tiles + FP64 on candidates */
#define ERT_ACCEL_BVH     3   /* sphere BVH (FP32 conservative slabs/filter) + FP64 on candidates;
                               * wavefront form: path / shadow / shade queues in HBM, full warps of one ray kind */
#define ERT_ACCEL_BVH_MEGAKERNEL 4  /* same BVH, one launch, per-pixel state machine (kept as a cross-check) */
#define ERT_ACCEL_GRID    5   /* the wavefront of ERT_ACCEL_BVH whose path rays step through a uniform cell grid
                               * over the spheres (3-D DDA, FP32 conservative) instead of walking the BVH.  Built
                               * for scenes of many small spheres; scenes without one (and rays that start far
                               * outside the scene) use the BVH.  ERT_ACCEL_AUTO prefers it when the scene has one. */
#define ERT_ACCEL_WARP    6   /* ert_trace_rays only: one WARP per ray — the lanes stride over the sphere list (FP32 filter,
                               * FP64 literal test on their survivors) and the nearest hit is the warp-wide lexicographic
                               * minimum of (Distance, list position), three __reduce_min_sync steps.  The optional
                               * warp-wide reduction of the design brief; measured against the thread-per-ray scan in
                               * DESIGN.md (it loses wherever the rays of a warp can share the sphere loop). */

#define ERT_FLAG_COUNT_TESTS  1u  /* instrumented run: fill the test counters in ert_stats (slower) */
#define ERT_FLAG_TIME_KERNELS  8u  /* ERT_ACCEL_BVH: CUDA events around every launch; fills the *_ms split of ert_stats */
#define ERT_FLAG_NO_LIGHT_GRID 4u /* ERT_ACCEL_BVH: shadow rays walk the BVH even for lights that have a
                                   * direction grid (A/B switch; same frame) */
#define ERT_FLAG_WF_UNSORTED  2u  /* ERT_ACCEL_BVH: skip the binning of hits by location (A/B switch; the
                                   * frame is identical, only the schedule of the queues changes) */
/* Turn the primary rays by the camera's `rotation` (the per-call camera, or the scene's).  Without this flag the
 * rotation is not read and every frame is the reference's, which ignores it (erl:487).  With it:
 *   - primary ray: v = point_on_screen - location as today (erl:486-507), O = location, D = vnormalize(d) with
 *     d_i = (M[i][0]*v.x + M[i][1]*v.y) + M[i][2]*v.z in FP64, nothing contracted;
 *   - M = Ry(ry) . (Rx(rx) . Rz(rz)) with (rx, ry, rz) = rotation in degrees, right-handed rotations about the
 *     world axes: Rx = [[1,0,0],[0,c,-s],[0,s,c]], Ry = [[c,0,s],[0,1,0],[-s,0,c]], Rz = [[c,-s,0],[s,c,0],[0,0,1]],
 *     each product entry (A[i][0]*B[0][j] + A[i][1]*B[1][j]) + A[i][2]*B[2][j], computed once per call on the host;
 *   - angle: a = fmod(deg, 360.0) (exact); a in {0, +-90, +-180, +-270} gives the exact (s, c) in {-1, 0, 1} (s = +0
 *     where it is 0), any other a gives s = sin(r), c = cos(r) with r = a * (M_PI / 180.0) (the host libm);
 *   - if M is exactly the identity (e.g. (0,0,0), (360,-720,0), (180,180,180)) the frame is bit-identical to the
 *     same call without the flag.
 * World +y is down (floors at y = 5, lights at negative y), so (0,90,0) looks along +x, (0,180,0) along -z,
 * (90,0,0) along -y (up), and rz rolls the picture about the view axis.  Supersampling (each sub-pixel ray is
 * turned), parts, slots, ert_download and ert_stats behave as without the flag.  A non-finite rotation is
 * ERT_ERR_BADARG with the flag and is accepted without it. */
#define ERT_FLAG_CAMERA_ROTATION 16u

typedef struct ert_render_params {
    int32_t width, height;      /* pixels, both > 0 (guards at erl:89) */
    int32_t depth;              /* Recursion_depth >= 0; 0 renders black (erl:186-187) */
    int32_t format;             /* ERT_FMT_* */
    int32_t accel;              /* ERT_ACCEL_* */
    /* Row-band partition (the distributed driver's chunking, erl:130-149, mapped
     * onto rows): rows are cut into bands of band_rows rows, band b belongs to
     * part (b % n_parts).  band_rows == 0 or n_parts <= 1 => the whole frame. */
    int32_t band_rows;
    int32_t n_parts;
    int32_t part;
    uint32_t flags;
    /* Samples per axis N (box-filtered supersampling; 0 or 1: one ray per pixel, the reference's frame).
     * With 2 <= N <= ERT_MAX_SUPERSAMPLE, sample k = j*N + i (i, j in [0, N)) of pixel (X, Y) is the unclamped
     * FP64 colour of pixel (N*X + i, N*Y + j) of the (N*width) x (N*height) frame of the same scene, camera,
     * depth and accel; the pixel is acc / (double)(N*N) with acc = c_0, then acc = acc + c_k for k = 1 .. N*N-1,
     * stored in `format` by the rules of the formats above.  Parts, depth 0 and `camera` behave as for one
     * sample.  ert_stats: `pixels` counts output pixels; rays, the test counters, bounce_path_rays[] and
     * bounce_hits[] sum over all samples (bounce_path_rays[0] = pixels*N*N); times, gpu_launches and the
     * ERT_FLAG_TIME_KERNELS split span all sample passes.  N < 0, N > ERT_MAX_SUPERSAMPLE, or N*width or
     * N*height above INT32_MAX is ERT_ERR_BADARG. */
    int32_t supersample;
    const ert_camera *camera;   /* NULL => the camera stored with the scene */
} ert_render_params;

#define ERT_MAX_SUPERSAMPLE 8

#define ERT_MAX_BOUNCE_STATS 16

typedef struct ert_stats {
    double kernel_ms;           /* CUDA-event time of the render kernel(s) on the slot's stream */
    double total_ms;            /* kernel(s) + device-to-host copies, CUDA events */
    uint64_t rays;              /* nearest-object scans resolved (primary + reflection + shadow) */
    uint64_t pixels;
    uint64_t gpu_launches;      /* kernels launched by the last call on this slot */
    uint64_t d2h_bytes;
    uint64_t h2d_bytes;
    /* filled only with ERT_FLAG_COUNT_TESTS */
    uint64_t sphere_filter_tests;   /* FP32 ray/sphere filter evaluations */
    uint64_t box_tests;             /* FP32 ray/AABB slab tests */
    uint64_t exact_sphere_tests;    /* FP64 literal ray_sphere_intersect evaluations */
    uint64_t exact_other_tests;     /* FP64 plane/triangle evaluations */
    int32_t accel_used;             /* ERT_ACCEL_* actually run */
    int32_t reserved;
    /* wavefront form (ERT_ACCEL_BVH) only.  Test counters split by kernel class (with
     * ERT_FLAG_COUNT_TESTS) and device time by kernel class (with ERT_FLAG_TIME_KERNELS). */
    uint64_t path_box_tests, path_filter_tests;       /* wf_trace_path*: BVH walks of path rays */
    uint64_t shadow_box_tests, shadow_filter_tests;   /* wf_trace_shadow: direction grids / BVH walks */
    double path_ms, shadow_ms, other_ms;              /* other: hit emission, binning, shading, finalize */
    uint64_t path_launches, shadow_launches;
    /* ABI 3 */
    uint64_t cell_steps;            /* cells visited by the grid walks of path rays (ERT_FLAG_COUNT_TESTS) */
    int32_t has_cell_grid;          /* the scene has a cell grid (ERT_ACCEL_GRID is available) */
    int32_t bounces_recorded;       /* entries of the two arrays below that are filled (wavefront frames only) */
    /* Per reflection level b (0 = primary): path rays traced and hits found.  rays = sum_b (path[b] + L*hits[b]);
     * the reference re-traces the reflection once per light (erl:216-224), so its own ray count for the
     * same frame is sum_b L^b * (path[b] + L*hits[b]) (plus the reflections off surfaces of reflectivity
     * exactly 0, which it traces and multiplies by 0, and this library does not trace). */
    uint64_t bounce_path_rays[ERT_MAX_BOUNCE_STATS];
    uint64_t bounce_hits[ERT_MAX_BOUNCE_STATS];
} ert_stats;

typedef struct ert_scene ert_scene;     /* opaque: device-resident flattened scene */

#define ERT_MAX_SLOTS 4

/* Number of CUDA devices visible to this process. */
ERT_API int ert_device_count(int *count);

/* Flattens `desc` to SoA, builds the sphere BVH on the host and uploads
 * everything to `device` once ("upload once, render many").  Replaces the
 * by-value Scene argument of the tracing function (erl:728-732). */
ERT_API int ert_scene_create(const ert_scene_desc *desc, int device, ert_scene **out);

/* Same scene on another device without rebuilding the BVH. */
ERT_API int ert_scene_clone(const ert_scene *src, int device, ert_scene **out);

ERT_API int ert_scene_destroy(ert_scene *scene);

/* ---- in-place update ------------------------------------------------------ */
#define ERT_UPDATE_REBUILD_GRIDS 1u  /* rebuild stale cell / direction grids on the device */
#define ERT_UPDATE_REBUILD       2u  /* full rebuild of every structure in place (the create path), handle kept */

/* ert_update_info.changed: the tables that differ from the scene's (element for element, by `order`) */
#define ERT_CHANGED_CAMERA         1u
#define ERT_CHANGED_LIGHTS         2u   /* any light field */
#define ERT_CHANGED_LIGHT_POS      4u   /* a light location */
#define ERT_CHANGED_SPHERES        8u   /* sphere centres or radii */
#define ERT_CHANGED_SPHERE_MAT    16u
#define ERT_CHANGED_TRIANGLES     32u   /* triangle vertices */
#define ERT_CHANGED_TRIANGLE_MAT  64u
#define ERT_CHANGED_PLANES       128u   /* plane normals, distances or materials */

/* ert_update_info.done */
#define ERT_DID_REFIT_SPHERES        1u  /* sphere BVH refitted on the device (filters and constants recomputed) */
#define ERT_DID_REFIT_TRIANGLES      2u  /* triangle BVH refitted on the device */
#define ERT_DID_DROP_CELL_GRID       4u  /* the cell grid went stale and was dropped */
#define ERT_DID_DROP_LIGHT_GRIDS     8u  /* direction grids went stale and were dropped */
#define ERT_DID_REBUILD_CELL_GRID   16u  /* ERT_UPDATE_REBUILD_GRIDS: the cell grid was built again on the device */
#define ERT_DID_REBUILD_LIGHT_GRIDS 32u  /* ERT_UPDATE_REBUILD_GRIDS: direction grids were built again on the device */
#define ERT_DID_REBUILD_TRI_BVH     64u  /* a tree triangle broke the builder's admission rule: triangle BVH rebuilt on the host */
#define ERT_DID_REBUILD            128u  /* ERT_UPDATE_REBUILD: every structure built again on the host */

typedef struct ert_update_info {
    uint32_t changed;               /* ERT_CHANGED_* */
    uint32_t done;                  /* ERT_DID_* */
    int32_t has_cell_grid;          /* after the update */
    int32_t light_grids;            /* lights with a direction grid after the update */
    int32_t light_grids_rebuilt;
    int32_t reserved;
    uint64_t h2d_bytes;             /* element tables uploaded (and trees rebuilt on the host, the direction grids' descriptors) */
    double host_ms;                 /* wall time of the call */
    double device_ms;               /* CUDA events around the uploads, the update kernels and the grid builds */
    /* per tree: total child-box surface area now over the area at its last build (1 when unchanged or absent);
     * a refitted tree degrades as this grows, ERT_UPDATE_REBUILD resets it */
    double sphere_area_ratio;
    double triangle_area_ratio;
} ert_update_info;

/* Replaces the scene's values with those of `desc`, keeping the handle.  `desc` must have the list shape of the
 * scene's create: the same element counts per kind and the same set of `order` values per kind, in any table order.
 * Any value may change.  A shape mismatch, a non-finite value or a duplicate `order` returns ERT_ERR_BADARG and
 * leaves the scene untouched (everything is validated before any device write).  The call first finishes every
 * slot, so a frame already queued renders the old scene.  Without ERT_UPDATE_REBUILD the BVHs are refitted on the
 * device, and a cell or direction grid that the change made stale is dropped (ERT_ACCEL_GRID falls back to the BVH
 * wavefront, shadow rays walk the BVH) unless ERT_UPDATE_REBUILD_GRIDS rebuilds it.  Every frame stays the linear
 * scan's.  A CUDA failure during the update leaves the scene unusable (renders return ERT_ERR_CUDA) until a
 * successful update.  `info` may be NULL. */
ERT_API int ert_scene_update(ert_scene *scene, const ert_scene_desc *desc, uint32_t flags, ert_update_info *info);

/* Renders the rows of params->part and copies them into `host_frame`, a buffer
 * for the FULL width*height frame (each part lands at its own rows, so parts
 * rendered on different GPUs assemble one frame without a gather step).
 * host_frame_bytes must be >= width*height*3*sizeof(element).
 * Replaces trace_ray_through_pixel/3 applied to every pixel (erl:90-99, 180-184). */
ERT_API int ert_render(ert_scene *scene, const ert_render_params *params, void *host_frame,
               size_t host_frame_bytes);

/* Asynchronous form on one of ERT_MAX_SLOTS independent (stream, framebuffer)
 * slots; host_frame may be NULL (keep the result on the device).  ert_wait
 * blocks until the slot is idle and reports the first error of the call. */
ERT_API int ert_render_async(ert_scene *scene, const ert_render_params *params, int slot,
                     void *host_frame, size_t host_frame_bytes);
ERT_API int ert_wait(ert_scene *scene, int slot);

/* Copies the part last rendered on `slot` to the host (same placement rule). */
ERT_API int ert_download(ert_scene *scene, int slot, void *host_frame, size_t host_frame_bytes);

ERT_API int ert_get_stats(ert_scene *scene, int slot, ert_stats *out);

/* Nearest object for a batch of rays (origin xyz, direction xyz as doubles):
 * nearest_object_intersecting_ray/2 (erl:300-302).  order_out[i] is the list
 * position of the nearest object or -1 for 'none'; t_out[i] its Distance.
 * The device time of the kernel is left in slot 0's stats (ert_get_stats(scene, 0, ..).kernel_ms). */
ERT_API int ert_trace_rays(ert_scene *scene, int64_t n_rays, const double *rays6, int accel,
                   int32_t *order_out, double *t_out);

/* Pinned host memory for frames, and registration of caller-owned memory
 * (e.g. a shared mapping that several per-GPU processes fill). */
ERT_API int ert_host_alloc(size_t bytes, void **out);
ERT_API int ert_host_free(void *p);
ERT_API int ert_host_register(void *p, size_t bytes);
ERT_API int ert_host_unregister(void *p);

/* Measured FP32 issue peak of `device`: lane-instructions per second of a
 * register-resident FFMA loop (the roofline denominator of the scan kernels). */
ERT_API int ert_fp32_peak(int device, double *lane_instr_per_s);
/* The same loop with three register operands per FFMA, the form the intersection kernels issue. */
ERT_API int ert_fp32_peak_rrr(int device, double *lane_instr_per_s);

/* Measured FP64 issue peak of `device` (register-resident DFMA loop): the roofline denominator of the kernels
 * that decide every object in the literal FP64 arithmetic (small scenes, ERT_ACCEL_EXACT). */
ERT_API int ert_fp64_peak(int device, double *lane_instr_per_s);
/* Measured device -> pinned-host copy rate of `device` in GB/s for copies of `bytes` (the roofline denominator of
 * the frames that are bound by getting the framebuffer to the host: C2, C5). */
ERT_API int ert_d2h_peak(int device, size_t bytes, double *gb_per_s);

/* Writes a buffer larger than L2 on `device` (bench hygiene between timed steps). */
ERT_API int ert_l2_flush(int device);

/* Message of the last failing call on the calling thread. */
ERT_API const char *ert_last_error(void);

ERT_API int ert_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ERT_B200_H */
