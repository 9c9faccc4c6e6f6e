// The FP64 element tables of a scene, and the checks and the packer that read an ert_scene_desc into them for both
// ert_scene_create and ert_scene_update, so that a moved scene equals a fresh create.  Plain C++ (no CUDA).
#pragma once
#include <array>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/ert_b200.h"

namespace ert {

enum ElemKind { K_LIGHTS, K_PLANES, K_TRIS, K_SPHERES, K_COUNT };   // the order the packer checks them in
// DevScene's arrays of the same names, in the order of an update's staging buffer
enum TableId { T_LIGHTS, T_PLANES, T_PLANE_MAT, T_TRIS, T_TRI_MAT, T_SPH_EXACT, T_SPH_MAT, T_SPH_REFL, T_COUNT };
// per: doubles per element; changed: the ert_update_info.changed bit of a change to the table
struct TableInfo { const char *name; ElemKind kind; int per; uint32_t changed; };
// a light is diffuse rgb, location xyz, specular rgb; a plane normal xyz, distance; a triangle v1 v2 v3; a sphere
// centre xyz, radius; a material colour rgb, specular_power, shininess, reflectivity; sph_refl the reflectivity again
inline constexpr TableInfo kTables[T_COUNT] = {
    {"lights", K_LIGHTS, 9, ERT_CHANGED_LIGHTS},       {"planes", K_PLANES, 4, ERT_CHANGED_PLANES},
    {"plane_mat", K_PLANES, 6, ERT_CHANGED_PLANES},    {"tris", K_TRIS, 9, ERT_CHANGED_TRIANGLES},
    {"tri_mat", K_TRIS, 6, ERT_CHANGED_TRIANGLE_MAT},  {"sph_exact", K_SPHERES, 4, ERT_CHANGED_SPHERES},
    {"sph_mat", K_SPHERES, 6, ERT_CHANGED_SPHERE_MAT}, {"sph_refl", K_SPHERES, 1, ERT_CHANGED_SPHERE_MAT},
};

// scene element i of kind k is element src[k][i] of the descriptor's table; an empty src[k] is the identity
using SourceOrder = std::array<std::vector<int64_t>, K_COUNT>;

// The checks return the message of the first defect (an ERT_ERR_BADARG), or an empty string.
std::string check_camera(const ert_camera &c);
// ert_scene_create: the header, then list positions >= 0 and distinct across all kinds.  src: lights and spheres in
// list order, planes and triangles as listed; order[k]: the list positions of kind k in that order.
std::string check_create(const ert_scene_desc *d, SourceOrder &src, std::vector<int> order[K_COUNT]);
// ert_scene_update of a scene with the list positions order[k]: the same counts, the header, then per kind the same
// list positions; src maps each scene element to the descriptor's.
std::string check_update(const ert_scene_desc *d, const std::vector<int> order[K_COUNT], SourceOrder &src);
// Checks every element (lights, planes, triangles, spheres, each in scene element order) and writes the tables; tab[t]
// has room for the kind's count times kTables[t].per doubles.
std::string pack_tables(const ert_scene_desc &d, const SourceOrder &src, double *const tab[T_COUNT]);

}  // namespace ert
