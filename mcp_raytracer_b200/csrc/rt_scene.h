// rt_scene.h — host-side scene compiler: rt_scene_desc -> flat device-ready arrays.
#pragma once
#include <string>
#include <vector>

#include "../../include/rt_b200.h"
#include "rt_types.h"

namespace rt {

struct HostScene {
  DevCamera cam{};
  float cam_u[3], cam_v[3], cam_w[3];
  double focus_distance = 0;
  int image_width = 0, image_height = 0;
  int n_objects = 0;
  int bvh_kind = 0;
  int n_unbounded = 0;
  int planar_any = 0;
  int list_n[6] = {0, 0, 0, 0, 0, 0}; // LIST: slots per kind (spheres, aa-quads x/y/z, quads, planes)
  float sph_cmax = 0, sph_r2max = 0;  // LIST: max |centre component| and max r^2 over the spheres
  int max_depth = 0; // deepest leaf below node 0
  std::vector<Node> nodes;
  std::vector<F4> p0, p1, p2, p3;
  std::vector<I2> slot_info;
  std::vector<ExactPrim> exact;
  std::vector<F4> matA, matE, matF;
  std::vector<I4> matB;
  std::vector<DevLight> lights;
};

// Validates the description (same failure conditions as src/scenes/scenes.ts:109-199) and
// compiles it.  Never throws; on failure returns a status and fills `err`.
rt_status compile_scene(const rt_scene_desc* scene, const rt_render_opts* opts, HostScene& out, std::string& err);

} // namespace rt
