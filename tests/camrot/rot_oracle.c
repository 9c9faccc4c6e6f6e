/*
 * rot_oracle.c — the C oracle (oracle/oracle.c, included unchanged) with the camera rotation of
 * ERT_FLAG_CAMERA_ROTATION restated on top of it.  TEST INFRASTRUCTURE ONLY.
 *
 * Written from include/ert_b200.h, not from the library: the angle of each axis is reduced with fmod (exact),
 * quarter turns take their exact sine and cosine, other angles glibc sin/cos of a * (M_PI / 180.0); the matrix is
 * Ry . (Rx . Rz), every entry (A[i][0]*B[0][j] + A[i][1]*B[1][j]) + A[i][2]*B[2][j]; the primary direction is
 * v_normalize of M v, v = point_on_screen - location.  Build like the oracle: -ffp-contract=off -fno-fast-math.
 */
#include "../../oracle/oracle.c"

typedef double mat3[3][3];

static void rot_sin_cos(double deg, double *s, double *c)
{
    double a = fmod(deg, 360.0);
    if (a == 0.0) { *s = 0.0; *c = 1.0; return; }
    if (a == 90.0 || a == -270.0) { *s = 1.0; *c = 0.0; return; }
    if (a == 180.0 || a == -180.0) { *s = 0.0; *c = -1.0; return; }
    if (a == -90.0 || a == 270.0) { *s = -1.0; *c = 0.0; return; }
    double r = a * (M_PI / 180.0);
    *s = sin(r);
    *c = cos(r);
}

static void rot_mul(mat3 a, mat3 b, mat3 out)
{
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double t = a[i][0] * b[0][j];
            t = t + a[i][1] * b[1][j];
            out[i][j] = t + a[i][2] * b[2][j];
        }
}

/* returns 1 when the matrix is exactly the identity */
static int rot_matrix(const double *rot, mat3 m)
{
    double sx, cx, sy, cy, sz, cz;
    rot_sin_cos(rot[0], &sx, &cx);
    rot_sin_cos(rot[1], &sy, &cy);
    rot_sin_cos(rot[2], &sz, &cz);
    mat3 rx = {{1, 0, 0}, {0, cx, -sx}, {0, sx, cx}};
    mat3 ry = {{cy, 0, sy}, {0, 1, 0}, {-sy, 0, cy}};
    mat3 rz = {{cz, -sz, 0}, {sz, cz, 0}, {0, 0, 1}};
    mat3 xz;
    rot_mul(rx, rz, xz);
    rot_mul(ry, xz, m);
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++)
            if (m[i][j] != (i == j ? 1.0 : 0.0)) return 0;
    return 1;
}

EXPORT int orc_camera_matrix(const double *rot3, double *m9)
{
    mat3 m;
    int id = rot_matrix(rot3, m);
    for (int i = 0; i < 9; i++) m9[i] = m[i / 3][i % 3];
    return id;
}

/* the primary ray of pixel coordinates (x, y) = (X/W, Y/H); rotate == 0 is ray_through_pixel itself */
static ray rot_ray_through_pixel(double x, double y, const double *cam, int rotate, mat3 m)
{
    if (!rotate) return ray_through_pixel(x, y, cam);
    vec from = v3(cam[0], cam[1], cam[2]);
    vec v = v_sub(point_on_screen(x, y, cam), from);
    vec d = v3(m[0][0] * v.x + m[0][1] * v.y + m[0][2] * v.z,
               m[1][0] * v.x + m[1][1] * v.y + m[1][2] * v.z,
               m[2][0] * v.x + m[2][1] * v.y + m[2][2] * v.z);
    ray r;
    r.o = from;
    r.d = v_normalize(d);
    return r;
}

EXPORT void orc_ray_through_pixel_rot(double x, double y, const double *cam, int rotate, double *o6)
{
    mat3 m;
    rot_matrix(cam + 3, m);
    ray r = rot_ray_through_pixel(x, y, cam, rotate, m);
    o6[0] = r.o.x; o6[1] = r.o.y; o6[2] = r.o.z; o6[3] = r.d.x; o6[4] = r.d.y; o6[5] = r.d.z;
}

typedef struct {
    job_t j;
    int rotate;
    mat3 m;
} rjob_t;

static void *rot_worker(void *arg)
{
    rjob_t *rj = (rjob_t *)arg;
    job_t *j = &rj->j;
    counters_t c = {0, 0};
    int64_t chunk = j->npix / ((int64_t)j->nthreads * 16);
    if (chunk < 1) chunk = 1;
    if (chunk > 64) chunk = 64;
    for (;;) {
        int64_t lo, hi;
        pthread_mutex_lock(&j->mu);
        lo = j->next;
        j->next += chunk;
        pthread_mutex_unlock(&j->mu);
        if (lo >= j->npix) break;
        hi = lo + chunk < j->npix ? lo + chunk : j->npix;
        for (int64_t k = lo; k < hi; k++) {
            int x = j->xs ? j->xs[k] : (int)(k % j->width);
            int y = j->ys ? j->ys[k] : (int)(k / j->width);
            ray r = rot_ray_through_pixel((double)x / (double)j->width, (double)y / (double)j->height, j->cam,
                                          rj->rotate, rj->m);
            vec col = pixel_colour_from_ray(r, &j->sc, j->depth, j->retrace, &c);
            j->out[3 * k] = col.x; j->out[3 * k + 1] = col.y; j->out[3 * k + 2] = col.z;
        }
    }
    pthread_mutex_lock(&j->mu);
    j->total.rays += c.rays;
    j->total.tests += c.tests;
    pthread_mutex_unlock(&j->mu);
    return NULL;
}

/* orc_render with a rotate switch: 0 renders exactly what orc_render renders (the rotation is not read), 1 turns
 * the primary rays by the matrix of cam[3..5], even when that matrix is the identity */
EXPORT int orc_render_rot(const double *cam, int n, const int32_t *kind, const double *f, int width, int height,
                          int depth, int rotate, int64_t npix, const int32_t *xs, const int32_t *ys, double *out,
                          int nthreads, uint64_t *counters2)
{
    rjob_t rj;
    pthread_t th[256];
    if (width <= 0 || height <= 0 || depth < 0) return -1;
    memset(&rj, 0, sizeof rj);
    job_t *j = &rj.j;
    j->cam = cam;
    j->sc.n = n; j->sc.kind = kind; j->sc.f = f;
    j->width = width; j->height = height; j->depth = depth;
    j->xs = xs; j->ys = ys;
    j->npix = (xs && ys) ? npix : (int64_t)width * height;
    j->out = out;
    rj.rotate = rotate;
    if (rotate) rot_matrix(cam + 3, rj.m);
    pthread_mutex_init(&j->mu, NULL);
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    j->nthreads = nthreads;
    for (int t = 1; t < nthreads; t++) pthread_create(&th[t], NULL, rot_worker, &rj);
    rot_worker(&rj);
    for (int t = 1; t < nthreads; t++) pthread_join(th[t], NULL);
    pthread_mutex_destroy(&j->mu);
    if (counters2) { counters2[0] = j->total.rays; counters2[1] = j->total.tests; }
    return 0;
}
