// trace_oracle.cpp — batches of the oracle's traceRay for the radiance-query tests.
// TEST INFRASTRUCTURE ONLY (tests/trace_oracle.py compiles it into a library of its own).
//
// The rh_trace_rays tests compare hundreds of thousands of rays with the oracle ray by ray.  This file compiles
// oracle/oracle.cpp as it stands (its functions are reachable here because it is part of this translation unit) and
// adds one entry point over rays double[n][6] = origin, direction, run on n_threads host threads (<= 0: all):
//   orc_trace_batch: traceRay sc 0 max_depth r (RayHs.hs:149-154) per ray: colors_out double[n][3], ids_out int32[n][2]
//   (object, tri of the ray's closest hit; -1, -1 on a miss; may be null) and counts_out[5] (may be null): the rays of
//   every class the batch cast, summed: primary, reflect, probe, exit, shadow.
#include "../oracle/oracle.cpp"

extern "C" {

int orc_trace_batch(void* s, const double* rays, uint64_t n, int max_depth, double* colors_out, int32_t* ids_out,
                    uint64_t* counts_out, int n_threads) {
  const Scene& sc = ((OracleScene*)s)->sc;
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  n_threads = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)std::max(n_threads, 1), (n + 255) / 256));
  std::vector<Counters> tc(n_threads);
  std::atomic<uint64_t> next{0};
  auto worker = [&](int tid) {
    for (;;) {
      const uint64_t b = next.fetch_add(256);
      if (b >= n) break;
      for (uint64_t i = b; i < std::min<uint64_t>(n, b + 256); i++) {
        const double* q = rays + 6 * i;
        int obj, tri;
        const Color c = traceRay(sc, 0, max_depth, Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, tc[tid], 0, &obj, &tri);
        colors_out[3 * i] = c.r;
        colors_out[3 * i + 1] = c.g;
        colors_out[3 * i + 2] = c.b;
        if (ids_out) {
          ids_out[2 * i] = obj;
          ids_out[2 * i + 1] = tri;
        }
      }
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; t++) th.emplace_back(worker, t);
  worker(0);
  for (auto& t : th) t.join();
  if (counts_out)
    for (int k = 0; k < 5; k++) {
      counts_out[k] = 0;
      for (const Counters& c : tc) counts_out[k] += c.rays[k];
    }
  return 0;
}

}  // extern "C"
