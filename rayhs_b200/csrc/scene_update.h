// scene_update.h — what rh_scene_update has to rebuild: the class of an update, which lights' lit-triangle bits change,
// and which (light, occluder mesh) cube maps are rasterised anew or carried over from the previous tables.  Pure host
// logic with no CUDA header, so that it can be compiled and tested on its own.
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/rayhs_b200.h"

namespace rh {

enum UpdateClass : int {
  kUpdateNone = 0,      // no byte of a named field changed
  kUpdateColours = 1,   // light color / radius (not a sphere light's) and material color1 / color2 / size only: upload the tables
  kUpdateEmitters = 2,  // some object became or stopped being an emitter: occluder tables and all light tables anew
  kUpdateTables = 3,    // same occluders, other lights or material kinds: rebuild only the light tables that changed
};

template <class T>
inline bool same_bytes(const T& a, const T& b) { return memcmp(&a, &b, sizeof a) == 0; }

// What a light's cube maps and lit-triangle bits depend on, and, for a sphere light, its ball: a sphere light's radius is
// geometry (its light points, and whether it has those tables at all follows from its kind).
inline bool same_light_geometry(const rh_light& a, const rh_light& b) {
  return a.kind == b.kind && same_bytes(a.vec, b.vec) && (a.kind != RH_LIGHT_SPHERE || same_bytes(a.radius, b.radius));
}

inline UpdateClass classify_update(const rh_material* old_m, const rh_material* new_m, uint32_t n_materials, const rh_light* old_l,
                                   uint32_t n_old_lights, const rh_light* new_l, uint32_t n_new_lights,
                                   const std::vector<int32_t>& object_material) {
  bool any = n_old_lights != n_new_lights, colours_only = n_old_lights == n_new_lights;
  for (uint32_t i = 0; i < n_materials; i++) {
    const rh_material &a = old_m[i], &b = new_m[i];
    const bool shape = a.kind == b.kind && a.cmap_kind == b.cmap_kind && same_bytes(a.ior, b.ior) && a.texture == b.texture;
    colours_only &= shape;
    any |= !shape || !same_bytes(a.color1, b.color1) || !same_bytes(a.color2, b.color2) || !same_bytes(a.size, b.size);
  }
  for (uint32_t i = 0; i < n_old_lights && i < n_new_lights; i++) {
    const bool geometry = same_light_geometry(old_l[i], new_l[i]);
    colours_only &= geometry;
    any |= !geometry || !same_bytes(old_l[i].color, new_l[i].color) || !same_bytes(old_l[i].radius, new_l[i].radius);
  }
  if (!any) return kUpdateNone;
  if (colours_only) return kUpdateColours;
  for (int32_t m : object_material)
    if ((old_m[m].kind == RH_MAT_EMMIT) != (new_m[m].kind == RH_MAT_EMMIT)) return kUpdateEmitters;
  return kUpdateTables;
}

// Light indices below 12 (the lit-triangle bits) whose bits must be cleared and, where a light has the index now,
// recomputed: a new light, another kind or position / direction at the same index, or an index no light has any more.
inline uint32_t lit_changed_mask(const rh_light* old_l, uint32_t n_old_lights, const rh_light* new_l, uint32_t n_new_lights) {
  uint32_t mask = 0;
  for (uint32_t i = 0; i < 12 && (i < n_old_lights || i < n_new_lights); i++)
    if (i >= n_old_lights || i >= n_new_lights || !same_light_geometry(old_l[i], new_l[i])) mask |= 1u << i;
  return mask;
}

// For each new light: the old point light with the same position whose cube maps it can take over (each old light at
// most once, the first unclaimed one in index order), or -1 (a new light: its maps are rasterised).
inline std::vector<int32_t> match_point_lights(const rh_light* old_l, uint32_t n_old_lights, const rh_light* new_l,
                                               uint32_t n_new_lights) {
  std::vector<int32_t> match(n_new_lights, -1);
  std::vector<bool> taken(n_old_lights, false);
  for (uint32_t i = 0; i < n_new_lights; i++) {
    if (new_l[i].kind != RH_LIGHT_POINT) continue;
    for (uint32_t j = 0; j < n_old_lights; j++)
      if (!taken[j] && same_light_geometry(old_l[j], new_l[i])) {
        match[i] = (int32_t)j;
        taken[j] = true;
        break;
      }
  }
  return match;
}

// One (point light, occluder mesh) pair of the new tables, in the order the builder numbers the maps: mesh-major, then
// light index.  raster: build the map anew.  Else the pair takes over the old map old_map (kEmpty: the old pair's map was
// not worth having, and the same triangles and light give the same verdict).
struct MapStep {
  uint32_t mesh, light;
  bool raster;
  uint32_t old_map;
};

// old_index: the old tables' light_map_index (n_old_lights * kOccMeshes entries, kOccMeshes = 8), or empty when none
// can be reused (no old tables, another resolution, another occluder set): then every pair is rasterised.
inline std::vector<MapStep> plan_maps(const std::vector<uint32_t>& old_index, const std::vector<int32_t>& match,
                                      const rh_light* new_l, uint32_t n_new_lights, uint32_t n_meshes) {
  constexpr uint32_t kMeshes = 8, kNone = 0xFFFFFFFFu;
  std::vector<MapStep> steps;
  for (uint32_t m = 0; m < n_meshes; m++)
    for (uint32_t li = 0; li < n_new_lights; li++) {
      if (new_l[li].kind != RH_LIGHT_POINT) continue;
      const bool keep = !old_index.empty() && match[li] >= 0;
      steps.push_back({m, li, !keep, keep ? old_index[(size_t)match[li] * kMeshes + m] : kNone});
    }
  return steps;
}

}  // namespace rh
