// setup_kernels.cu — the light-space tables of rh_scene_create, built on the GPU.
//
// Both tables are embarrassingly parallel over triangles and the records they need are already in HBM when
// rh_scene_create gets to them (triangle records, the cull tree): one thread per (triangle, cube face) rasterises the
// "nearest possible occluder" cube maps with atomicMin on the cells (positive floats order like their bit patterns),
// one thread per (triangle, light) answers the lit-triangle query by walking the mesh's cull tree.  The geometry is
// light_geom.h, the very code the host builder (light_maps.cpp) runs — plain double arithmetic, compiled without
// fused multiply-add on both sides — so the device tables equal the host tables bit for bit
// (tests/test_round2_gpu.py compares them).  Why the tables are conservative: light_maps.cpp.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "device_types.cuh"
#include "light_geom.h"

namespace rhd {
namespace {

using rh::lg::P3;

constexpr uint32_t kInfBits = 0x7f800000u;

struct MarkAtomic {
  int* face;  // float bits
  int R;
  int val;
  __device__ __forceinline__ void operator()(int row, int c0, int c1) const {
    int* r = face + (size_t)row * R;
    for (int c = c0; c <= c1; c++)
      if (r[c] > val) atomicMin(r + c, val);  // (a stale read only costs a redundant atomic: cells only decrease)
  }
};

// Triangles sequence[begin .. end) of the mesh (strided order, see build_light_map) onto the six faces.
__global__ void light_map_raster_kernel(const rh_tri* __restrict__ tris, const uint32_t* __restrict__ slots, unsigned long long n,
                                        unsigned long long begin, unsigned long long end, unsigned long long stride, int permute,
                                        double lx, double ly, double lz, double scale_abs, int R, int* __restrict__ out,
                                        uint32_t* __restrict__ unsafe) {
  const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long i = begin + idx / 6;
  const int face = (int)(idx % 6);
  if (i >= end) return;
  const unsigned long long at = permute ? (i * stride) % n : i;
  const rh_tri& t = tris[slots[at]];
  const P3 lp = rh::lg::mk(lx, ly, lz);
  const P3 p0 = rh::lg::mk(t.p0[0], t.p0[1], t.p0[2]);
  const P3 a = rh::lg::sub(p0, lp);
  const P3 b = rh::lg::sub(rh::lg::add(p0, rh::lg::mk(t.e1[0], t.e1[1], t.e1[2])), lp);
  const P3 c = rh::lg::sub(rh::lg::add(p0, rh::lg::mk(t.e2[0], t.e2[1], t.e2[2])), lp);
  float val;
  if (!rh::lg::light_map_value(a, b, c, scale_abs, &val)) {
    *unsafe = 1u;
    return;
  }
  const P3 tri[3] = {a, b, c};
  MarkAtomic mark{out + (size_t)face * R * R, R, __float_as_int(val)};
  rh::lg::raster_face(R, tri, face / 2, (face & 1) ? -1.0 : 1.0, mark);
}

__global__ void fill_u32_kernel(uint32_t* p, size_t n, uint32_t v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

__global__ void count_empty_kernel(const uint32_t* __restrict__ cells, size_t n, unsigned long long* __restrict__ out) {
  unsigned long long mine = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) mine += cells[i] == kInfBits;
  for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, mine);
}

// Lit flags of one mesh for the lights in `mask`: lit[slot] gets the mesh in bits 12-15 and loses the mask's light bits
// first (the other lights' bits stay), then one thread per (triangle of the mesh, light of the mask) clears nothing and
// sets bit `light` when no other triangle of the mesh meets the triangle's query region K.
__global__ void lit_init_kernel(const uint32_t* __restrict__ slots, uint32_t n_slots, uint32_t mesh, uint32_t mask,
                                uint16_t* __restrict__ lit) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_slots) lit[slots[i]] = (uint16_t)((lit[slots[i]] & 0x0fffu & ~mask) | (mesh << 12));
}

__global__ void __launch_bounds__(128) lit_query_kernel(const rh_tri* __restrict__ tris, const WideNode32* __restrict__ nodes,
                                                        double cx, double cy, double cz, uint32_t root,
                                                        const uint32_t* __restrict__ slots, uint32_t n_slots,
                                                        const rh_light* __restrict__ lights, uint32_t mask, uint32_t n_mask,
                                                        uint32_t* __restrict__ lit_words) {
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t at = idx / n_mask;
  if (at >= n_slots) return;
  uint32_t rest = mask;  // the light: set bit number (idx - at * n_mask) of the mask
  for (uint32_t k = idx - at * n_mask; k; k--) rest &= rest - 1;
  const uint32_t li = (uint32_t)__ffs(rest) - 1;
  const uint32_t s0 = slots[at];
  rh::LitQuery q;
  const rh_light L = lights[li];
  if (!rh::lg::lit_query_make(tris[s0], L.vec, L.kind == RH_LIGHT_DIRECTIONAL, &q)) return;
  // The cull tree's float boxes (rounded outward by more than a float ulp, relative to the scene centre) contain the
  // double boxes the host builder tests, so the walk visits a superset of its leaves: what is "blocked" is decided by
  // the exact triangle test alone and comes out the same.
  uint32_t stack[kStack];
  int sp = 0;
  stack[sp++] = root;
  bool blocked = false;
  const double ctr[3] = {cx, cy, cz};
  while (sp > 0 && !blocked) {
    const WideNode32 w = nodes[stack[--sp]];
    for (int c = 0; c < 2 && !blocked; c++) {
      const uint32_t ch = w.child[c];
      if (ch == kEmpty) continue;
      double lo[3], hi[3];
      for (int k = 0; k < 3; k++) {
        lo[k] = (double)w.box[6 * c + k] + ctr[k];
        hi[k] = (double)w.box[6 * c + 3 + k] + ctr[k];
      }
      if (rh::lg::lit_query_box_outside(q, lo, hi)) continue;
      if (ch & kLeafBit) {
        const uint32_t first = ch & kLeafFirstMask, count = ((ch >> kLeafCountShift) & 7u) + 1u;
        for (uint32_t k = 0; k < count && !blocked; k++) blocked = (first + k != s0) && rh::lg::lit_query_tri_meets(q, tris[first + k]);
      } else if (sp < kStack) {
        stack[sp++] = ch;
      } else {
        blocked = true;  // (deeper than any tree rh_scene_create accepts: no flag)
      }
    }
  }
  if (!blocked) atomicOr(lit_words + (s0 >> 1), (1u << li) << (16 * (s0 & 1u)));
}

__global__ void lit_count_kernel(const uint32_t* __restrict__ slots, uint32_t n_slots, const uint16_t* __restrict__ lit,
                                 unsigned long long* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long mine = (i < n_slots && (lit[slots[i]] & 0x0fffu)) ? 1 : 0;
  for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, mine);
}

}  // namespace

// rh_init: loads this file's kernels (CUDA loads a kernel's code on first use) so that rh_scene_create does not pay for it.
int preload_setup_kernels() {
  cudaFuncAttributes a;
  cudaError_t e = cudaFuncGetAttributes(&a, light_map_raster_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, fill_u32_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, count_empty_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, lit_init_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, lit_query_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, lit_count_kernel);
  return (int)e;
}

// Device version of rh::build_light_map (light_maps.cpp) — same sequence of triangle batches, same early-outs.
// words: two 8-byte device words of scratch.  *useful = 0 when the map would be useless or unsafe.
int device_light_map(const double L[3], const rh_tri* d_tris, const uint32_t* d_slots, size_t n, int R, float* d_out,
                     double min_empty, unsigned long long* d_words, int* useful, double* empty_fraction, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const size_t cells = (size_t)6 * R * R;
  *useful = 0;
  fill_u32_kernel<<<592, 256, 0, st>>>((uint32_t*)d_out, cells, kInfBits);
  cudaMemsetAsync(d_words, 0, 16, st);
  double scale_abs = 1.0;
  for (int k = 0; k < 3; k++) scale_abs = scale_abs < (L[k] < 0 ? -L[k] : L[k]) ? (L[k] < 0 ? -L[k] : L[k]) : scale_abs;
  const size_t stride = n > 4096 ? 4093 : 1;
  const int permute = (stride > 1 && n % stride != 0) ? 1 : 0;
  size_t done = 0, next_check = 16384, prev_empty = 0;
  unsigned long long host_words[2];
  auto count_empty = [&](size_t* empty) -> int {
    cudaMemsetAsync(d_words + 1, 0, 8, st);
    count_empty_kernel<<<592, 256, 0, st>>>((const uint32_t*)d_out, cells, d_words + 1);
    cudaError_t e = cudaMemcpyAsync(host_words, d_words, 16, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    *empty = (size_t)host_words[1];
    return (int)e;
  };
  while (done < n) {
    const size_t end = n < next_check ? n : next_check;
    const size_t threads = (end - done) * 6;
    light_map_raster_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(d_tris, d_slots, n, done, end, stride, permute, L[0], L[1],
                                                                               L[2], scale_abs, R, (int*)d_out, (uint32_t*)d_words);
    done = end;
    if (done == next_check && done < n) {
      next_check *= 2;
      size_t empty = 0;
      if (int e = count_empty(&empty)) return e;
      if (host_words[0] & 0xffffffffull) return 0;  // unsafe
      if ((double)empty < min_empty * (double)cells) return 0;
      if (prev_empty > 0 && empty < prev_empty) {  // a soup shows early (see build_light_map)
        const double r = (double)(prev_empty - empty) / (double)prev_empty;
        const double blocks = (double)(n - done) / (0.5 * (double)done);
        if ((double)empty / (double)cells * pow(1.0 - r, blocks) < 1e-3 * min_empty) return 0;
      }
      prev_empty = empty;
    }
  }
  size_t empty = 0;
  if (int e = count_empty(&empty)) return e;
  if (host_words[0] & 0xffffffffull) return 0;
  if (empty_fraction) *empty_fraction = (double)empty / (double)cells;
  *useful = (double)empty >= min_empty * (double)cells ? 1 : 0;
  return 0;
}

// Device version of the lit-triangle queries of one mesh (runtime.cu's host loop) for the light indices in `mask` (bits
// below 12): clears those bits on the mesh's slots, writes the mesh into bits 12-15 and queries those of the lights
// 0 .. n_lights-1 that are not in `no_query` (sphere lights) only; the other bits stay.  mask 0 only counts.  Enqueues only; the flags of the mesh's slots are
// complete when the stream has run.  d_flagged: device counter, incremented by the number of triangles of this mesh with
// at least one flag.
int device_lit_flags(const rh_tri* d_tris, const WideNode32* d_nodes, const double center[3], uint32_t root, const uint32_t* d_slots,
                     uint32_t n_slots, const rh_light* d_lights, uint32_t n_lights, uint32_t mask, uint32_t no_query, uint32_t mesh,
                     uint16_t* d_lit, unsigned long long* d_flagged, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (!n_slots) return 0;
  mask &= 0x0fffu;
  const uint32_t query = mask & ~no_query & (n_lights >= 12 ? 0x0fffu : (1u << n_lights) - 1), n_query = (uint32_t)__builtin_popcount(query);
  if (mask) lit_init_kernel<<<(n_slots + 255) / 256, 256, 0, st>>>(d_slots, n_slots, mesh, mask, d_lit);
  if (n_query) {
    const unsigned long long threads = (unsigned long long)n_slots * n_query;
    lit_query_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(d_tris, d_nodes, center[0], center[1], center[2], root, d_slots,
                                                                        n_slots, d_lights, query, n_query, (uint32_t*)d_lit);
  }
  lit_count_kernel<<<(n_slots + 255) / 256, 256, 0, st>>>(d_slots, n_slots, d_lit, d_flagged);
  return (int)cudaGetLastError();
}

}  // namespace rhd
