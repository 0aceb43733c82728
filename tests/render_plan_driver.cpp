// C entry point of rayhs_b200/csrc/render_plan.h for tests/test_render_plan_cpu.py.  TEST INFRASTRUCTURE ONLY.
#include "../rayhs_b200/csrc/render_plan.h"

// Returns the number of chunks; when it is at most cap, fills rows, first_row and order (cap entries each) and
// info2 = {n_tail, ramped}.  row_cost: rows_local entries, or null.
extern "C" int rp_plan(int rows_local, unsigned long long row_samples, int chunk_samples, unsigned long long device_mem,
                       int host_offsets, const float* row_cost, int compute_bound, int cap, int* rows, int* first_row,
                       int* order, int* info2) {
  const rh::ChunkPlan p = rh::plan_chunks(rows_local, (size_t)row_samples, chunk_samples, (size_t)device_mem,
                                          host_offsets != 0, row_cost, compute_bound != 0);
  const int n = (int)p.rows.size();
  if (n > cap) return n;
  std::copy(p.rows.begin(), p.rows.end(), rows);
  std::copy(p.first_row.begin(), p.first_row.end(), first_row);
  std::copy(p.order.begin(), p.order.end(), order);
  info2[0] = p.n_tail;
  info2[1] = p.ramped ? 1 : 0;
  return n;
}
