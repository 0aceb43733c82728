// C entry points of rayhs_b200/csrc/scene_update.h for tests/test_scene_update_cpu.py.  TEST INFRASTRUCTURE ONLY.
#include "../rayhs_b200/csrc/scene_update.h"

extern "C" int su_classify(const rh_material* old_m, const rh_material* new_m, uint32_t n_materials, const rh_light* old_l,
                           uint32_t n_old, const rh_light* new_l, uint32_t n_new, const int32_t* object_material, uint32_t n_objects) {
  return rh::classify_update(old_m, new_m, n_materials, old_l, n_old, new_l, n_new,
                             std::vector<int32_t>(object_material, object_material + n_objects));
}

extern "C" uint32_t su_lit_mask(const rh_light* old_l, uint32_t n_old, const rh_light* new_l, uint32_t n_new) {
  return rh::lit_changed_mask(old_l, n_old, new_l, n_new);
}

// Plans the maps of n_meshes occluder meshes; old_index: n_old * 8 words or null (nothing reusable).  Returns the number
// of steps; when it is at most cap, fills steps[k] = {mesh, light, raster, old_map}.
extern "C" int su_plan(const uint32_t* old_index, const rh_light* old_l, uint32_t n_old, const rh_light* new_l, uint32_t n_new,
                       uint32_t n_meshes, int cap, uint32_t* steps) {
  const std::vector<uint32_t> idx = old_index ? std::vector<uint32_t>(old_index, old_index + (size_t)n_old * 8) : std::vector<uint32_t>();
  const std::vector<rh::MapStep> p = rh::plan_maps(idx, rh::match_point_lights(old_l, n_old, new_l, n_new), new_l, n_new, n_meshes);
  if ((int)p.size() > cap) return (int)p.size();
  for (size_t k = 0; k < p.size(); k++) {
    steps[4 * k] = p[k].mesh;
    steps[4 * k + 1] = p[k].light;
    steps[4 * k + 2] = p[k].raster ? 1u : 0u;
    steps[4 * k + 3] = p[k].old_map;
  }
  return (int)p.size();
}
