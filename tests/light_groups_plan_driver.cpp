// C entry point of rayhs_b200/csrc/render_plan.h's per-sample byte count for tests/test_light_groups_cpu.py.
// TEST INFRASTRUCTURE ONLY.
#include "../rayhs_b200/csrc/render_plan.h"

// As tests/render_plan_driver.cpp's rp_plan, with the device bytes per sample of a chunk (0: plan_chunks' default).
// Returns the number of chunks; when it is at most cap, fills rows (cap entries).
extern "C" int lg_plan(int rows_local, unsigned long long row_samples, int chunk_samples, unsigned long long device_mem,
                       int host_offsets, unsigned long long bytes_per_sample, int cap, int* rows) {
  const rh::ChunkPlan p = bytes_per_sample
      ? rh::plan_chunks(rows_local, (size_t)row_samples, chunk_samples, (size_t)device_mem, host_offsets != 0, nullptr, false,
                        (size_t)bytes_per_sample)
      : rh::plan_chunks(rows_local, (size_t)row_samples, chunk_samples, (size_t)device_mem, host_offsets != 0, nullptr, false);
  const int n = (int)p.rows.size();
  if (n <= cap) std::copy(p.rows.begin(), p.rows.end(), rows);
  return n;
}

extern "C" unsigned long long lg_default_bytes_per_sample(void) { return rh::kBytesPerSample; }
