// render_plan.h — the chunk plan of a frame: which local rows each wavefront chunk holds and in which order the chunks
// are processed.  Pure host arithmetic with no CUDA header, so that it can be compiled and tested on its own.
#pragma once
#include <algorithm>
#include <cstddef>
#include <vector>

namespace rh {

constexpr int kLanes = 2;                          // chunks in flight, each with its own stream and queues
constexpr size_t kStreamChunk = (size_t)16 << 20;  // chunk size (samples) when the sample offsets stream in from the host
constexpr size_t kStreamFirst = (size_t)4 << 20;   // ... and of the first chunk, whose upload nothing overlaps
// Device bytes per sample of a chunk: accumulators + (two ray queues + hit queue + half a walk queue) at 2 entries per
// sample, in 16-byte double2 words.
constexpr size_t kBytesPerSample = 3 * 8 + 2 * (2 * 4 * 16 + (5 * 16 + 8) + (5 * 16 + 12) / 2);

struct ChunkPlan {
  std::vector<int> rows;       // rows per chunk, in row order
  std::vector<int> first_row;  // first local row of each chunk
  std::vector<int> order;      // processing order of the chunks (rows are independent, Image.hs:34-36)
  int n_tail = 0;              // chunks at the end of `rows` that stay last in `order` (streamed offsets)
  bool ramped = false;         // the compute-bound plan of a streamed frame whose row costs are known
};

// The largest chunk (samples) the library plans on its own: as many samples as 45 % of the device memory holds.
inline size_t max_chunk_samples(size_t device_mem, size_t bytes_per_sample = kBytesPerSample) {
  return std::min<size_t>((size_t)(0.45 * (double)device_mem) / bytes_per_sample, (size_t)0x3ffffff0u);
}

// Mean cost per row of rows [row0, row0 + n).
inline double cost_density(const float* row_cost, int row0, int n) {
  double c = 0;
  for (int r = row0; r < row0 + n; r++) c += row_cost[r];
  return c / std::max(1, n);
}

// The chunk plan (whole rows) of a frame of rows_local rows of row_samples samples.  chunk_samples > 0 is the caller's
// chunk size, else the library picks it from device_mem.  host_offsets: the pass-0 items stream in from the host.
// row_cost: kernel time per row measured by the last streamed frame of the same shape (rows_local entries), or null;
// compute_bound: in that frame the kernels, not the upload, finished last.
//
// The secondary passes of a chunk are short launches whose cost is set by their slowest warp, so the fewer and larger
// the chunks the better (measured on the bench frame with the offsets already in HBM: 16 chunks 65.5 ms, 8 chunks
// 59.1 ms, 4 chunks 57.0 ms, 1 chunk 55.0 ms).  Default: as large as 45 % of the device memory allows.  When the
// offsets stream in from the host, chunk k+1's upload overlaps chunk k's kernels, so the chunks stay moderate and the
// first one, whose upload nothing can overlap, is small.  bytes_per_sample: the device scratch a sample of a chunk needs
// (a frame with more per-sample state than the render's passes its own count).
inline ChunkPlan plan_chunks(int rows_local, size_t row_samples, int chunk_samples, size_t device_mem, bool host_offsets,
                             const float* row_cost, bool compute_bound, size_t bytes_per_sample = kBytesPerSample) {
  ChunkPlan p;
  std::vector<int>& plan = p.rows;
  size_t want = (size_t)chunk_samples, first = want;
  if (chunk_samples <= 0) {
    want = max_chunk_samples(device_mem, bytes_per_sample);
    // a frame that needs several chunks has two of them in flight, each with its own scratch: half the budget each
    if ((size_t)rows_local * row_samples > want) want /= kLanes;
    if (host_offsets) want = std::min<size_t>(want, kStreamChunk);
    first = host_offsets ? std::min<size_t>(want, kStreamFirst) : want;
  }
  const bool know_cost = row_cost && host_offsets && chunk_samples <= 0;
  int ramp_first = 0, ramp_pieces = 1;  // the ramp plan's most expensive chunk starts at plan[ramp_first], in ramp_pieces pieces
  if (know_cost && compute_bound && (size_t)rows_local * row_samples > 2 * want) {
    // Compute-bound streaming (the kernels finish after the last byte has arrived): what counts is that the GPU never
    // waits for data once the first bytes are there.  Equal chunks, the expensive rows first (their kernels keep the GPU
    // busy while the cheap rows arrive), and the very first chunk processed — the most expensive one — cut into
    // 1/8, 1/8, 1/4, 1/2 so that its first piece is uploaded quickly and each piece's kernels cover the next piece's
    // upload.  No small pieces at the end: they only help when the upload finishes last.
    const int rows_per = (int)std::max<size_t>(1, want / row_samples);
    for (int row = 0; row < rows_local; row += rows_per) plan.push_back(std::min(rows_per, rows_local - row));
    if (plan.size() >= 2 && plan.back() * 4 < rows_per) {
      plan[plan.size() - 2] += plan.back();
      plan.pop_back();
    }
    size_t best = 0;
    double best_d = -1;
    for (size_t k = 0, row = 0; k < plan.size(); row += plan[k], k++) {
      const double dk = cost_density(row_cost, (int)row, plan[k]);
      if (dk > best_d) { best_d = dk; best = k; }
    }
    const int n = plan[best];
    ramp_first = (int)best;
    if (n >= 16) {
      const int e = n / 8;
      plan[best] = e;
      plan.insert(plan.begin() + best + 1, {e, 2 * e, n - 4 * e});
      ramp_pieces = 4;
    }
    p.ramped = true;
  } else {
    int row = 0;
    while (row < rows_local) {
      const size_t w = plan.empty() ? first : want;
      const int n = (int)std::max<size_t>(1, std::min<size_t>(w / row_samples, (size_t)(rows_local - row)));
      plan.push_back(n);
      row += n;
    }
    // Streamed offsets: the frame ends with the kernels of the chunk whose upload finishes last, so the frame's last
    // chunk is cut into halves of halves (down to ~1 Mi samples): what is left to do after the last byte has arrived is
    // a small chunk's work.
    if (host_offsets && chunk_samples <= 0 && plan.size() >= 4) {
      int last = plan.back();
      plan.pop_back();
      const int min_rows = (int)std::max<size_t>(1, ((size_t)1 << 20) / row_samples);
      while (last > 2 * min_rows && p.n_tail < 4) {
        plan.push_back(last - last / 2);
        last /= 2;
        p.n_tail++;
      }
      plan.push_back(last);
      p.n_tail++;
    }
  }

  const int n_chunks = (int)plan.size();
  p.first_row.resize(n_chunks);
  p.order.resize(n_chunks);
  for (int ck = 0, row = 0; ck < n_chunks; row += plan[ck], ck++) { p.first_row[ck] = row; p.order[ck] = ck; }
  if (know_cost && n_chunks > 2) {
    // the compute-bound plan: the pieces of the most expensive chunk first, in row order, then everything in descending
    // cost per row; else the small first chunk stays first and the tail pieces last
    std::vector<double> dens(n_chunks);
    for (int ck = 0; ck < n_chunks; ck++) dens[ck] = cost_density(row_cost, p.first_row[ck], plan[ck]);
    if (p.ramped) {
      p.order.clear();
      for (int k = 0; k < ramp_pieces; k++) p.order.push_back(ramp_first + k);
      for (int ck = 0; ck < n_chunks; ck++)
        if (ck < ramp_first || ck >= ramp_first + ramp_pieces) p.order.push_back(ck);
    }
    std::stable_sort(p.order.begin() + (p.ramped ? ramp_pieces : 1), p.order.end() - p.n_tail,
                     [&](int x, int y) { return dens[x] > dens[y]; });
  }
  return p;
}

}  // namespace rh
