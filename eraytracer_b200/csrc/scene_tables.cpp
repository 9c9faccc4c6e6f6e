#include "scene_tables.h"

#include <algorithm>
#include <cmath>
#include <utility>

namespace ert {

namespace {

bool finite3(const double *v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); }
bool finite_mat(const ert_material &m)
{
    return finite3(m.colour) && std::isfinite(m.specular_power) && std::isfinite(m.shininess) &&
           std::isfinite(m.reflectivity);
}
void put_mat(double *o, const ert_material &m)
{
    for (int a = 0; a < 3; a++) o[a] = m.colour[a];
    o[3] = m.specular_power; o[4] = m.shininess; o[5] = m.reflectivity;
}

std::string check_header(const ert_scene_desc &d)
{
    if (d.n_lights < 0 || d.n_spheres < 0 || d.n_triangles < 0 || d.n_planes < 0) return "negative element count";
    if ((d.n_lights && !d.lights) || (d.n_spheres && !d.spheres) || (d.n_triangles && !d.triangles) ||
        (d.n_planes && !d.planes))
        return "element table pointer is NULL";
    if (d.n_spheres >= (1 << 28) || d.n_planes >= (1 << 28) || d.n_triangles >= (1 << 28) || d.n_lights >= (1 << 20))
        return "too many elements";
    return check_camera(d.camera);
}

// the indices of tab by list position; empty when it is in that order already
template <typename E>
std::vector<int64_t> by_order(const E *tab, int64_t n)
{
    if (std::is_sorted(tab, tab + n, [](const E &a, const E &b) { return a.order < b.order; })) return {};
    std::vector<int64_t> idx((size_t)n);
    for (int64_t k = 0; k < n; k++) idx[(size_t)k] = k;
    std::sort(idx.begin(), idx.end(), [&](int64_t a, int64_t b) { return tab[a].order < tab[b].order; });
    return idx;
}

// Scene element i (list position want[i]) is element map[i] of the new table; an empty map is the identity (the
// caller lists the elements as the scene does, the animation case: one linear pass).
template <typename E>
std::string map_by_order(const E *tab, int64_t n, const std::vector<int> &want, const char *kind,
                         std::vector<int64_t> &map)
{
    map.clear();
    bool same = true;
    for (int64_t i = 0; i < n && same; i++) same = tab[i].order == want[(size_t)i];
    if (same) return {};
    std::vector<std::pair<int32_t, int64_t>> got((size_t)n), had((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        got[(size_t)i] = {tab[i].order, i};
        had[(size_t)i] = {want[(size_t)i], i};
    }
    std::sort(got.begin(), got.end());
    std::sort(had.begin(), had.end());
    for (size_t i = 1; i < got.size(); i++)
        if (got[i].first == got[i - 1].first)
            return std::string("duplicate list position in `order` among the ") + kind;
    map.assign((size_t)n, 0);
    for (size_t i = 0; i < got.size(); i++) {
        if (got[i].first != had[i].first)
            return std::string("the ") + kind + " do not have the list positions of the scene's create";
        map[(size_t)had[i].second] = got[i].second;
    }
    return {};
}

}  // namespace

std::string check_camera(const ert_camera &c)
{
    if (finite3(c.location) && std::isfinite(c.fov) && std::isfinite(c.screen_width) && std::isfinite(c.screen_height))
        return {};
    return "camera has a non-finite field";
}

std::string check_create(const ert_scene_desc *d, SourceOrder &src, std::vector<int> order[K_COUNT])
{
    if (!d) return "scene descriptor is NULL";
    if (std::string e = check_header(*d); !e.empty()) return e;
    src = SourceOrder{by_order(d->lights, d->n_lights), {}, {}, by_order(d->spheres, d->n_spheres)};
    std::vector<int32_t> all;
    auto gather = [&](int k, const auto *tab, int64_t n) {
        order[k].resize((size_t)n);
        for (int64_t i = 0; i < n; i++) order[k][(size_t)i] = tab[src[k].empty() ? i : src[k][(size_t)i]].order;
        all.insert(all.end(), order[k].begin(), order[k].end());
    };
    gather(K_LIGHTS, d->lights, d->n_lights);
    gather(K_PLANES, d->planes, d->n_planes);
    gather(K_TRIS, d->triangles, d->n_triangles);
    gather(K_SPHERES, d->spheres, d->n_spheres);
    // list positions must be distinct: they decide ties (erl:319) and the light fold order (erl:211)
    std::sort(all.begin(), all.end());
    for (size_t i = 0; i < all.size(); i++) {
        if (all[i] < 0) return "negative list position in `order`";
        if (i && all[i] == all[i - 1]) return "duplicate list position in `order`";
    }
    return {};
}

std::string check_update(const ert_scene_desc *d, const std::vector<int> order[K_COUNT], SourceOrder &src)
{
    if (!d) return "scene descriptor is NULL";
    if (d->n_lights != (int64_t)order[K_LIGHTS].size() || d->n_planes != (int64_t)order[K_PLANES].size() ||
        d->n_triangles != (int64_t)order[K_TRIS].size() || d->n_spheres != (int64_t)order[K_SPHERES].size())
        return "element counts differ from the scene's (a new list shape needs ert_scene_create)";
    std::string e = check_header(*d);      // whose count checks the scene's counts passed at create
    if (e.empty()) e = map_by_order(d->lights, d->n_lights, order[K_LIGHTS], "lights", src[K_LIGHTS]);
    if (e.empty()) e = map_by_order(d->spheres, d->n_spheres, order[K_SPHERES], "spheres", src[K_SPHERES]);
    if (e.empty()) e = map_by_order(d->triangles, d->n_triangles, order[K_TRIS], "triangles", src[K_TRIS]);
    if (e.empty()) e = map_by_order(d->planes, d->n_planes, order[K_PLANES], "planes", src[K_PLANES]);
    return e;
}

std::string pack_tables(const ert_scene_desc &d, const SourceOrder &src, double *const tab[T_COUNT])
{
    auto at = [&](int k, int64_t i) { return src[k].empty() ? i : src[k][(size_t)i]; };
    for (int64_t i = 0; i < d.n_lights; i++) {
        const ert_point_light &l = d.lights[at(K_LIGHTS, i)];
        if (!finite3(l.diffuse_colour) || !finite3(l.location) || !finite3(l.specular_colour))
            return "point_light has a non-finite field";
        double *o = tab[T_LIGHTS] + 9 * i;
        for (int a = 0; a < 3; a++) { o[a] = l.diffuse_colour[a]; o[3 + a] = l.location[a]; o[6 + a] = l.specular_colour[a]; }
    }
    for (int64_t i = 0; i < d.n_planes; i++) {
        const ert_plane &q = d.planes[at(K_PLANES, i)];
        if (!finite3(q.normal) || !std::isfinite(q.distance) || !finite_mat(q.material))
            return "plane has a non-finite field";
        double *o = tab[T_PLANES] + 4 * i;
        o[0] = q.normal[0]; o[1] = q.normal[1]; o[2] = q.normal[2]; o[3] = q.distance;
        put_mat(tab[T_PLANE_MAT] + 6 * i, q.material);
    }
    for (int64_t i = 0; i < d.n_triangles; i++) {
        const ert_triangle &q = d.triangles[at(K_TRIS, i)];
        if (!finite3(q.v1) || !finite3(q.v2) || !finite3(q.v3) || !finite_mat(q.material))
            return "triangle has a non-finite field";
        double *o = tab[T_TRIS] + 9 * i;
        for (int a = 0; a < 3; a++) { o[a] = q.v1[a]; o[3 + a] = q.v2[a]; o[6 + a] = q.v3[a]; }
        put_mat(tab[T_TRI_MAT] + 6 * i, q.material);
    }
    for (int64_t i = 0; i < d.n_spheres; i++) {
        const ert_sphere &q = d.spheres[at(K_SPHERES, i)];
        if (!finite3(q.center) || !std::isfinite(q.radius) || !finite_mat(q.material))
            return "sphere has a non-finite field";
        double *o = tab[T_SPH_EXACT] + 4 * i;
        o[0] = q.center[0]; o[1] = q.center[1]; o[2] = q.center[2]; o[3] = q.radius;
        put_mat(tab[T_SPH_MAT] + 6 * i, q.material);
        tab[T_SPH_REFL][i] = q.material.reflectivity;
    }
    return {};
}

}  // namespace ert
