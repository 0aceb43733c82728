// batch.cpp — the oracle library liborc.so: oracle.cpp (the restatement and its C interface) and, after it, the batch
// entry points the tests query it through.  TEST INFRASTRUCTURE ONLY, like oracle.cpp.
//
// rayhs_b200/build.py compiles this file, with oracle.cpp's flags, into oracle/_build/liborc.so.  The batch functions
// live here rather than in oracle.cpp so that oracle.cpp stays a self-contained translation unit that other sources can
// #include to reach its internals (closestIntersection, traceRay, ...) and add entry points of their own, including ones
// of these names.
#include "oracle.cpp"

// The parity tests compare the GPU with the oracle over up to millions of caller-built rays, double[n][6] = origin,
// direction; one ctypes call per ray through orc_closest would be far too slow for that.  Each ray's result depends on
// that ray alone and the ray counts are integer sums, so neither the block size nor the thread count changes an output.

// body(c, i) for every i in [0, n) on n_threads host threads (<= 0: all), in blocks of 256 claimed from a counter; c is
// the calling thread's own Counters.  Returns the rays of every class the threads counted, summed.
template <class Body>
static Counters parallel_rays(uint64_t n, int n_threads, const Body& body) {
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  n_threads = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)std::max(n_threads, 1), (n + 255) / 256));
  std::vector<Counters> tc(n_threads);
  std::atomic<uint64_t> next{0};
  auto worker = [&](int tid) {
    Counters c;  // on the thread's own stack, sharing no cache line with another thread
    for (uint64_t b; (b = next.fetch_add(256)) < n;)
      for (uint64_t i = b; i < std::min<uint64_t>(n, b + 256); i++) body(c, i);
    tc[tid] = c;
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; t++) th.emplace_back(worker, t);
  worker(0);
  for (auto& t : th) t.join();
  Counters sum;
  for (const Counters& c : tc)
    for (int k = 0; k < 5; k++) sum.rays[k] += c.rays[k];
  return sum;
}

static Ray ray_at(const double* rays, uint64_t i) {
  const double* q = rays + 6 * i;
  return Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}};
}

extern "C" {

// rayFromPixel (Projection.hs:22-39) at n pixel coordinates xy[n][2]: rays_out[n][6] (orc_ray_from_pixel's, in one call)
void orc_camera_rays(const rh_camera* cam, double w, double h, const double* xy, uint64_t n, double* rays_out) {
  for (uint64_t i = 0; i < n; i++) orc_ray_from_pixel(cam, w, h, xy[2 * i], xy[2 * i + 1], rays_out + 6 * i);
}

// closestIntersection (RayHs.hs:67-71) per ray: one rh_hit record (a miss: t = +inf, p = n = uv = 0, object = tri = -1)
int orc_closest_batch(void* s, const double* rays, uint64_t n, rh_hit* out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  parallel_rays(n, n_threads, [&](Counters& c, uint64_t i) {
    MatHit h;
    rh_hit& o = out[i];
    memset(&o, 0, sizeof o);
    if (!closestIntersection(sc, ray_at(rays, i), &h, c, 0)) {
      o.t = inf;
      o.object = o.tri = -1;
      return;
    }
    o.t = h.t;
    o.p[0] = h.p.x; o.p[1] = h.p.y; o.p[2] = h.p.z;
    o.n[0] = h.n.x; o.n[1] = h.n.y; o.n[2] = h.n.z;
    o.uv[0] = h.uv.u; o.uv[1] = h.uv.v;
    o.object = h.object;
    o.tri = h.tri;
  });
  return 0;
}

// shadowIntersection (RayHs.hs:74-87) towards light `light` per ray: out[i] = 1 where shadowed, else 0.  -1: no such light
int orc_shadow_batch(void* s, uint32_t light, const double* rays, uint64_t n, uint8_t* out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  if (light >= sc.lights.size()) return -1;
  parallel_rays(n, n_threads, [&](Counters& c, uint64_t i) {
    out[i] = shadowIntersection(sc, sc.lights[light], ray_at(rays, i), c) ? 1 : 0;
  });
  return 0;
}

// traceRay sc 0 max_depth r (RayHs.hs:149-154) per ray: colors_out double[n][3], ids_out int32[n][2] (object, tri of the
// ray's closest hit; -1, -1 on a miss; may be null) and counts_out[5] (may be null): the rays of every class the batch
// cast, summed: primary, reflect, probe, exit, shadow.
int orc_trace_batch(void* s, const double* rays, uint64_t n, int max_depth, double* colors_out, int32_t* ids_out,
                    uint64_t* counts_out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  const Counters sum = parallel_rays(n, n_threads, [&](Counters& c, uint64_t i) {
    int obj, tri;
    const Color col = traceRay(sc, 0, max_depth, ray_at(rays, i), c, 0, &obj, &tri);
    colors_out[3 * i] = col.r;
    colors_out[3 * i + 1] = col.g;
    colors_out[3 * i + 2] = col.b;
    if (ids_out) {
      ids_out[2 * i] = obj;
      ids_out[2 * i + 1] = tri;
    }
  });
  if (counts_out)
    for (int k = 0; k < 5; k++) counts_out[k] = sum.rays[k];
  return 0;
}

// closestIntersection per ray and the first-hit features of the feature buffers: t_out[n] (+inf on a miss), n_out[n][3]
// (the Hit's normal), albedo_out[n][3] (colorAt of a Diffuse / Plastic material at the hit's uv, color1 of Emmit, the
// normal of ShowNormal, (u, v, 0) of ShowUV, (1, 1, 1) of Mirror / Transparent), ids_out[n][2] (object, tri; -1, -1 on a
// miss) and uv_out[n][2] (the Hit's uv); normal, albedo and uv are 0 on a miss.
int orc_feature_batch(void* s, const double* rays, uint64_t n, double* t_out, double* n_out, double* albedo_out, int32_t* ids_out,
                      double* uv_out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  parallel_rays(n, n_threads, [&](Counters& c, uint64_t i) {
    MatHit h;
    double* nn = n_out + 3 * i;
    double* a = albedo_out + 3 * i;
    if (!closestIntersection(sc, ray_at(rays, i), &h, c, 0)) {
      t_out[i] = inf;
      nn[0] = nn[1] = nn[2] = a[0] = a[1] = a[2] = 0;
      ids_out[2 * i] = ids_out[2 * i + 1] = -1;
      uv_out[2 * i] = uv_out[2 * i + 1] = 0;
      return;
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
  });
  return 0;
}

}  // extern "C"
