// feature_oracle.cpp — per-sample first-hit features from the oracle, for the feature-buffer tests.
// TEST INFRASTRUCTURE ONLY (tests/feature_oracle.py compiles it into a library of its own).
//
// This file compiles oracle/oracle.cpp as it stands (its functions are reachable here because it is part of this
// translation unit) and adds two entry points:
//   orc_camera_rays:   rayFromPixel (Projection.hs:22-39) at n pixel coordinates xy[n][2]: rays_out[n][6] = origin, direction
//                      (what orc_ray_from_pixel returns, one call for all of them);
//   orc_feature_batch: closestIntersection (RayHs.hs:67-71) of rays double[n][6] on n_threads host threads (<= 0: all),
//                      and per ray t_out[n] (+inf on a miss), n_out[n][3] (the Hit's normal; 0 on a miss),
//                      albedo_out[n][3] (colorAt of a Diffuse / Plastic material at the hit's uv, color1 of Emmit, the
//                      normal of ShowNormal, (u, v, 0) of ShowUV, (1, 1, 1) of Mirror / Transparent; 0 on a miss) and
//                      ids_out[n][2] (object, tri; -1, -1 on a miss) and uv_out[n][2] (the Hit's uv; 0 on a miss).
#include "../oracle/oracle.cpp"

extern "C" {

void orc_camera_rays(const rh_camera* cam, double w, double h, const double* xy, uint64_t n, double* rays_out) {
  for (uint64_t i = 0; i < n; i++) orc_ray_from_pixel(cam, w, h, xy[2 * i], xy[2 * i + 1], rays_out + 6 * i);
}

int orc_feature_batch(void* s, const double* rays, uint64_t n, double* t_out, double* n_out, double* albedo_out, int32_t* ids_out,
                      double* uv_out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  n_threads = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)std::max(n_threads, 1), (n + 1023) / 1024));
  std::atomic<uint64_t> next{0};
  auto worker = [&]() {
    for (;;) {
      const uint64_t b = next.fetch_add(1024);
      if (b >= n) break;
      for (uint64_t i = b; i < std::min<uint64_t>(n, b + 1024); i++) {
        const double* q = rays + 6 * i;
        Counters c;
        MatHit h;
        double* nn = n_out + 3 * i;
        double* a = albedo_out + 3 * i;
        if (!closestIntersection(sc, Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, &h, c, 0)) {
          t_out[i] = inf;
          nn[0] = nn[1] = nn[2] = a[0] = a[1] = a[2] = 0;
          ids_out[2 * i] = ids_out[2 * i + 1] = -1;
          uv_out[2 * i] = uv_out[2 * i + 1] = 0;
          continue;
        }
        const rh_material& m = sc.materials[h.material];
        Color al{1, 1, 1};
        if (m.kind == RH_MAT_DIFFUSE || m.kind == RH_MAT_PLASTIC) al = colorAt(sc, m, h.uv);
        else if (m.kind == RH_MAT_EMMIT) al = Color{m.color1[0], m.color1[1], m.color1[2]};
        else if (m.kind == RH_MAT_SHOWNORMAL) al = Color{h.n.x, h.n.y, h.n.z};
        else if (m.kind == RH_MAT_SHOWUV) al = Color{h.uv.u, h.uv.v, 0};
        t_out[i] = h.t;
        nn[0] = h.n.x; nn[1] = h.n.y; nn[2] = h.n.z;
        a[0] = al.r; a[1] = al.g; a[2] = al.b;
        ids_out[2 * i] = h.object;
        ids_out[2 * i + 1] = h.tri;
        uv_out[2 * i] = h.uv.u;
        uv_out[2 * i + 1] = h.uv.v;
      }
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; t++) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
  return 0;
}

}  // extern "C"
