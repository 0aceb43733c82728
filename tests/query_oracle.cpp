// query_oracle.cpp — batches of the oracle's closestIntersection / shadowIntersection for the ray-query tests.
// TEST INFRASTRUCTURE ONLY (tests/query_oracle.py compiles it into a library of its own).
//
// The ray-query tests compare millions of rays with the oracle; one ctypes call per ray through orc_closest is far too
// slow for that.  This file compiles oracle/oracle.cpp as it stands (its functions are reachable here because it is
// part of this translation unit) and adds two entry points over rays double[n][6] = origin, direction, run on
// n_threads host threads (<= 0: all):
//   orc_closest_batch: one rh_hit record per ray (a miss: t = +inf, p = n = uv = 0, object = tri = -1);
//   orc_shadow_batch:  1 where the ray towards light `light` is shadowed, else 0.
#include "../oracle/oracle.cpp"

#include <functional>

namespace {

void parallel_rays(uint64_t n, int n_threads, const std::function<void(uint64_t)>& body) {
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  n_threads = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)std::max(n_threads, 1), (n + 1023) / 1024));
  std::atomic<uint64_t> next{0};
  auto worker = [&]() {
    for (;;) {
      const uint64_t b = next.fetch_add(1024);
      if (b >= n) break;
      for (uint64_t i = b; i < std::min<uint64_t>(n, b + 1024); i++) body(i);
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; t++) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
}

}  // namespace

extern "C" {

int orc_closest_batch(void* s, const double* rays, uint64_t n, rh_hit* out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  parallel_rays(n, n_threads, [&](uint64_t i) {
    const double* q = rays + 6 * i;
    Counters c;
    MatHit h;
    rh_hit& o = out[i];
    memset(&o, 0, sizeof o);
    if (!closestIntersection(sc, Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, &h, c, 0)) {
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

int orc_shadow_batch(void* s, uint32_t light, const double* rays, uint64_t n, uint8_t* out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  if (light >= sc.lights.size()) return -1;
  parallel_rays(n, n_threads, [&](uint64_t i) {
    const double* q = rays + 6 * i;
    Counters c;
    out[i] = shadowIntersection(sc, sc.lights[light], Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, c) ? 1 : 0;
  });
  return 0;
}

}  // extern "C"
