// kernels.cu — sm_100a kernels of the RayHs ray-casting path (SURVEY.md §8a, K1-K7).
//
//   trace_kernel          K1/K2/K4/K5: camera-ray generation (pass 0) or queued secondary rays (pass >= 1), closest hit
//                         through the object list + wide-BVH traversal, shading.  A Diffuse / Plastic hit folds its
//                         lights on the spot (accumDiffuse, RayHs.hs:89-97) unless some light's shadow ray has to walk
//                         a tree: only those hits are queued, with the lights to walk and the lights already settled.
//   shadow_pooled_kernel  K3 for coherent rays: the queued hits of a slab, their tree walks pooled per light into
//                         warp-local rounds of 32, then the fold.
//   shadow_refill_kernel  K3 for incoherent rays (triangle soups): one queued hit per lane, a lane whose ray has ended
//                         takes its next light or the next hit while its neighbours keep walking.
//   shadow_simple_kernel  K3 for scenes with more than 32 lights.
//   resolve_kernel        K6: average the samples of a pixel, toIntC, coalesced RGB8 store (or peer stores).
//   store_colors_kernel   K6 of rh_trace_rays: the linear colours of caller-built rays (trace_kernel<.., RAYS = true>).
//   deinterleave          K7: band re-assembly after the all-gather.
//
// All arithmetic is IEEE double in the reference's operation order and this file is compiled with -fmad=false (GHC
// emits no fused multiply-adds), so every value the reference defines (t, u, v, hit point, normal, colour) is computed
// bit-identically; only atan/acos (sphere uv, Geometry.hs:96) go through CUDA's libm instead of the host's.  No tensor
// cores: the path is branchy gather-bound traversal.  Each device function cites the reference lines it restates;
// nothing here is shared with oracle/.
//
// B200 specifics: persistent warps (one block per SM); the traversal stack is a per-thread column of SHARED memory
// (8-byte entries), never local memory; queues are arrays of 128-entry slabs that a warp reserves or claims with one
// atomic; the trace kernel's next batch of queue entries / sample offsets arrives by bulk async copy
// (cp.async.bulk.shared::cluster.global + mbarrier, SASS: UBLKCP / SYNCS) while the current batch is traced.
#include <cuda_runtime.h>

#include <cstdint>

#include "device_types.cuh"

namespace rhd {
namespace {

constexpr double kEps = 0.000001;              // Geometry.hs:31-32
constexpr double kPiInv = 0.3183098861837907;  // Math.hs:11-12 (1 / pi in double)
constexpr double kPruneSlack = 1.0000001;      // boxes are skipped only when tmin exceeds the best t by > 1e-7 relative
constexpr unsigned kFull = 0xffffffffu;

// ------------------------------------------------------------------ GHC Ord Double (SURVEY App. A-N1)
__device__ __forceinline__ double hs_max(double x, double y) { return (x <= y) ? y : x; }
__device__ __forceinline__ double hs_min(double x, double y) { return (x <= y) ? x : y; }

// ------------------------------------------------------------------ Vec.hs
struct V3 {
  double x, y, z;
};
__device__ __forceinline__ V3 mk(double x, double y, double z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }  // Vec.hs:36
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }  // Vec.hs:40
__device__ __forceinline__ V3 neg(V3 a) { return mk(-a.x, -a.y, -a.z); }                              // Vec.hs:42
__device__ __forceinline__ V3 mul(double l, V3 a) { return mk(l * a.x, l * a.y, l * a.z); }            // Vec.hs:69
__device__ __forceinline__ V3 cmul(V3 a, V3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }        // Color.hs:23
__device__ __forceinline__ double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }        // Vec.hs:105
__device__ __forceinline__ V3 cross(V3 a, V3 b) {                                                       // Vec.hs:108-110
  return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ double sqrLen(V3 v) { return dot(v, v); }                           // Vec.hs:114
__device__ __forceinline__ double sqrDist(V3 v, V3 w) { return sqrLen(v - w); }                // Vec.hs:118
__device__ __forceinline__ V3 normalize(V3 v) { return mul(1 / sqrt(sqrLen(v)), v); }          // Vec.hs:126
__device__ __forceinline__ V3 reflect(V3 v, V3 n) { return v - mul(2 * dot(v, n), n); }        // Vec.hs:130
// Vec.hs:132-140
__device__ __forceinline__ bool refract(V3 i, V3 n, double n1, double n2, V3& out) {
  double n1n2 = n1 / n2;
  double cos0 = -(dot(i, n));
  double sin20 = n1n2 * n1n2 * (1 - cos0 * cos0);
  if (sin20 > 1) return false;
  double coeff = n1n2 * cos0 - sqrt(1.0 - sin20);
  out = mul(n1n2, i) + mul(coeff, n);
  return true;
}
__device__ __forceinline__ V3 ld3(const double* p) { return mk(p[0], p[1], p[2]); }

struct Ray {
  V3 o, d;
};
__device__ __forceinline__ V3 rayAt(const Ray& r, double t) { return r.o + mul(t, r.d); }  // Geometry.hs:29
__device__ __forceinline__ Ray rayEps(V3 p, V3 n) { return Ray{p + mul(kEps, n), n}; }      // Geometry.hs:36


// ------------------------------------------------------------------ shared-memory staging
// Top tree levels, object / material / light tables, and the occluder tables of shadowIntersection with what the
// light fold needs per (light, tree root): which outer side of the root box the light lies on and the light's cube map.
struct SmemTables {
  WideNode32 nodes[kSmemNodes];
  DObject objects[kSmemObjects];
  rh_material materials[kSmemObjects];
  rh_light lights[kSmemLights];
  OccPlane planes[kOccPlanes];
  OccSphere spheres[kOccSpheres];
  // Root boxes (the float cull boxes of the mesh super-roots and of the sphere tree, padded by 2e-6 + 1e-12 |x|) and,
  // per (light, root), on which outer side of each slab the light lies: bit a = below lo[a], bit 3 + a = above hi[a].
  double rootbox[kOccMeshes + 1][6];
  uint32_t mesh_roots[kOccMeshes + 1];  // the sphere tree's super-root follows the meshes'
  uint32_t light_map[kFastLights][kOccMeshes + 1];  // number of the pair's cube map in SceneView::light_maps, or kEmpty
  uint8_t light_side[kFastLights][kOccMeshes + 1];
  uint8_t pad_[4];
  // Plane sides (see fold_lights): per plane the margin terms m0 + m1 * |p|_1 a point needs to count as strictly on one
  // side, and per point light the planes it lies strictly in front of (pn.(L - pp) > margin) / behind.
  double plane_margin[kOccPlanes][2];
  uint32_t light_front[kFastLights], light_behind[kFastLights];
  uint8_t pad2_[32];
};
static_assert(sizeof(rh_material) == 96 && sizeof(rh_light) == 64, "table record sizes");
static_assert(sizeof(SmemTables) % 16 == 0, "per-warp regions follow the tables in dynamic shared memory");
// What the shadow kernels stage: top tree levels, lights, tree roots.
struct WalkTables {
  WideNode32 nodes[kSmemNodes];
  rh_light lights[kSmemLights];
  uint32_t mesh_roots[kOccMeshes + 4];
};
static_assert(sizeof(WalkTables) % 16 == 0, "per-warp regions follow the tables in dynamic shared memory");
extern __shared__ __align__(128) unsigned char rh_smem[];

__device__ __forceinline__ void copy16(void* dst, const void* src, uint32_t bytes) {
  uint4* d = (uint4*)dst;
  const uint4* s = (const uint4*)src;
  for (uint32_t i = threadIdx.x; i < bytes / 16; i += blockDim.x) d[i] = __ldg(s + i);
}

// Traversal stack of one thread: entry k < kShortStack in the thread's column of shared memory, deeper entries in its
// column of the global scratch area (ChunkParams::deep_stack).  Entry = (subtree reference, float entry distance).
struct Stack {
  uint2* col;    // &short_stack[0][threadIdx.x]; entry k at col[k * stride]
  uint2* deep;   // &deep_stack[0][global thread]; entry k at deep[(k - kShortStack) * deep_stride]
  uint32_t stride, deep_stride;
  __device__ __forceinline__ void push(int& sp, uint32_t ref, float tmin) {
    const uint2 e = make_uint2(ref, __float_as_uint(tmin));
    if (sp < kShortStack) col[sp * stride] = e;
    else deep[(size_t)(sp - kShortStack) * deep_stride] = e;
    sp++;
  }
  __device__ __forceinline__ uint2 pop(int& sp) {
    --sp;
    return sp < kShortStack ? col[sp * stride] : deep[(size_t)(sp - kShortStack) * deep_stride];
  }
  // the exact walk keeps its whole stack in the global column ((reference, first slot) pairs)
  __device__ __forceinline__ void push_deep(int& sp, uint32_t ref, uint32_t first) { deep[(size_t)(sp++) * deep_stride] = make_uint2(ref, first); }
  __device__ __forceinline__ uint2 pop_deep(int& sp) { return deep[(size_t)(--sp) * deep_stride]; }
};
__device__ __forceinline__ Stack make_stack(void* smem_columns, uint32_t block_threads, const ChunkParams& P) {
  Stack s;
  s.col = reinterpret_cast<uint2*>(smem_columns) + threadIdx.x;
  s.stride = block_threads;
  s.deep = P.deep_stack + (size_t)blockIdx.x * block_threads + threadIdx.x;
  s.deep_stride = P.deep_stride;
  return s;
}

struct Ctx {
  const SceneView* S;
  const WideNode32* sm_nodes;  // the first S->n_smem_nodes records of S->wide32, staged in shared memory
  const DObject* objects;
  const rh_material* materials;
  const rh_light* lights;
};

// Root boxes and light sides of the staged occluder tables (threads 0 .. n_roots * n_lights of the block).
__device__ __forceinline__ void stage_roots(SmemTables& sm, const SceneView& S) {
  const uint32_t n_meshes = S.n_occ_meshes, n_lights = S.n_lights;
  const uint32_t n_roots = n_meshes + (S.sphere_root != kEmpty ? 1u : 0u);
  if (threadIdx.x < n_roots) {
    const uint32_t root = threadIdx.x < n_meshes ? S.occ_meshes[threadIdx.x] : S.sphere_root;
    sm.mesh_roots[threadIdx.x] = root;
    const float* fb = S.wide32[root].box;  // slot 0 of a super-root = the tree's own box
    for (int a = 0; a < 3; a++) {
      const double lo = (double)fb[a] + S.center[a], hi = (double)fb[3 + a] + S.center[a];  // world coordinates
      sm.rootbox[threadIdx.x][a] = lo - (2e-6 + 1e-12 * fabs(lo));
      sm.rootbox[threadIdx.x][3 + a] = hi + (2e-6 + 1e-12 * fabs(hi));
    }
  }
  __syncthreads();
  if (threadIdx.x < n_roots * n_lights) {
    const uint32_t li = threadIdx.x / n_roots, m = threadIdx.x % n_roots;
    uint32_t side = 0;
    if (sm.lights[li].kind != RH_LIGHT_DIRECTIONAL)
      for (int a = 0; a < 3; a++) {
        if (sm.lights[li].vec[a] < sm.rootbox[m][a]) side |= 1u << a;
        if (sm.lights[li].vec[a] > sm.rootbox[m][3 + a]) side |= 8u << a;
      }
    sm.light_side[li][m] = (uint8_t)side;
    sm.light_map[li][m] = (S.light_map_index && m < n_meshes) ? S.light_map_index[li * kOccMeshes + m] : kEmpty;
  }
  // plane sides: |pn.v| <= |pn|_1 |v|_1 bounds both the 1e-6 step from a hit to its shadow-ray origin and every rounding
  if (threadIdx.x < S.n_occ_planes) {
    const OccPlane& pl = sm.planes[threadIdx.x];
    const double n1 = fabs(pl.n[0]) + fabs(pl.n[1]) + fabs(pl.n[2]), p1 = fabs(pl.p[0]) + fabs(pl.p[1]) + fabs(pl.p[2]);
    sm.plane_margin[threadIdx.x][0] = n1 * (1e-5 + 1e-12 * p1);
    sm.plane_margin[threadIdx.x][1] = n1 * 1e-12;
  }
  __syncthreads();
  if (threadIdx.x < n_lights) {
    const rh_light& L = sm.lights[threadIdx.x];
    uint32_t front = 0, behind = 0;
    if (L.kind != RH_LIGHT_DIRECTIONAL) {
      const V3 lp = ld3(L.vec);
      const double l1 = fabs(lp.x) + fabs(lp.y) + fabs(lp.z);
      for (uint32_t k = 0; k < S.n_occ_planes; k++) {
        const double f = dot(ld3(sm.planes[k].n), lp - ld3(sm.planes[k].p));
        const double m = sm.plane_margin[k][0] + sm.plane_margin[k][1] * l1;
        if (f > m) front |= 1u << k;
        if (f < -m) behind |= 1u << k;
      }
    }
    sm.light_front[threadIdx.x] = front;
    sm.light_behind[threadIdx.x] = behind;
  }
}

__device__ __forceinline__ void stage_tables(SmemTables& sm, const SceneView& S, Ctx& cx) {
  copy16(sm.nodes, S.wide32, S.n_smem_nodes * (uint32_t)sizeof(WideNode32));
  if (S.tables_in_smem) {
    copy16(sm.objects, S.objects, S.n_objects * (uint32_t)sizeof(DObject));
    copy16(sm.materials, S.materials, S.n_materials * (uint32_t)sizeof(rh_material));
    copy16(sm.lights, S.lights, S.n_lights * (uint32_t)sizeof(rh_light));
  }
  if (S.shadow_fast) {
    copy16(sm.planes, S.occ_planes, S.n_occ_planes * (uint32_t)sizeof(OccPlane));
    copy16(sm.spheres, S.occ_spheres, S.n_occ_spheres * (uint32_t)sizeof(OccSphere));
    if (!S.tables_in_smem) copy16(sm.lights, S.lights, S.n_lights * (uint32_t)sizeof(rh_light));
  }
  __syncthreads();
  if (S.shadow_fast) stage_roots(sm, S);
  __syncthreads();
  cx.S = &S;
  cx.sm_nodes = sm.nodes;
  cx.objects = S.tables_in_smem ? sm.objects : S.objects;
  cx.materials = S.tables_in_smem ? sm.materials : S.materials;
  cx.lights = (S.tables_in_smem || S.shadow_fast) ? sm.lights : S.lights;
}

// Shadow kernels: top tree levels, lights (when they fit) and the roots of the occluding trees.
__device__ __forceinline__ void stage_walk_tables(WalkTables& sm, const SceneView& S, Ctx& cx) {
  copy16(sm.nodes, S.wide32, S.n_smem_nodes * (uint32_t)sizeof(WideNode32));
  const bool lights_fit = S.n_lights <= (uint32_t)kSmemLights;
  if (lights_fit) copy16(sm.lights, S.lights, S.n_lights * (uint32_t)sizeof(rh_light));
  if (S.n_occ_meshes <= (uint32_t)kOccMeshes && threadIdx.x < S.n_occ_meshes) sm.mesh_roots[threadIdx.x] = S.occ_meshes[threadIdx.x];
  __syncthreads();
  cx.S = &S;
  cx.sm_nodes = sm.nodes;
  cx.objects = S.objects;  // sphere-tree leaves only
  cx.materials = S.materials;
  cx.lights = lights_fit ? sm.lights : S.lights;
}

// ------------------------------------------------------------------ counters
template <bool COUNT>
struct Cnt {
  unsigned long long box, tri, prim, nodes, gnodes, wtri, shade, texel, deep;
  __device__ __forceinline__ void zero() { box = tri = prim = nodes = gnodes = wtri = shade = texel = deep = 0; }
};
template <>
struct Cnt<false> {
#ifdef RH_WARP_TIMES
  unsigned dn, dt;  // diagnostic build: node steps and triangle tests of this lane
  __device__ __forceinline__ void zero() { dn = dt = 0; }
#else
  __device__ __forceinline__ void zero() {}
#endif
};
#define RH_CNT(field, n) \
  if constexpr (COUNT) cnt.field += (n)
#ifdef RH_WARP_TIMES
#define RH_DBG(field) \
  if constexpr (!COUNT) cnt.field += 1
#else
#define RH_DBG(field)
#endif

template <bool COUNT>
__device__ __forceinline__ void flush_counters(Cnt<COUNT>& cnt, FrameCounters* fc, int which) {
  if constexpr (COUNT) {
    KernelCounters* kc = &fc->k[which];
    unsigned long long* src[8] = {&cnt.box, &cnt.tri, &cnt.prim, &cnt.nodes, &cnt.shade, &cnt.texel, &cnt.gnodes, &cnt.wtri};
    unsigned long long* dst[8] = {&kc->box_tests, &kc->tri_tests, &kc->prim_tests, &kc->node_visits, &kc->shade_fetches,
                                  &kc->texel_fetches, &kc->global_node_visits, &kc->tri_records};
    for (int k = 0; k < 8; k++) {
      unsigned long long v = *src[k];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
      if ((threadIdx.x & 31) == 0 && v) atomicAdd(dst[k], v);
    }
    unsigned long long v = cnt.deep;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&fc->deep_pushes, v);
  }
}

// ------------------------------------------------------------------ KDTree.hs:39-56 rayInterBox
// `inv` holds 1/dx, 1/dy, 1/dz, which the reference recomputes at every box (same values).
__device__ __forceinline__ bool slab(const Ray& r, const V3& inv, double lx, double ly, double lz, double hx, double hy,
                                     double hz, double& tmin) {
  double t1 = inv.x * (lx - r.o.x);
  double t2 = inv.x * (hx - r.o.x);
  double t3 = inv.y * (ly - r.o.y);
  double t4 = inv.y * (hy - r.o.y);
  double t5 = inv.z * (lz - r.o.z);
  double t6 = inv.z * (hz - r.o.z);
  tmin = hs_max(hs_max(hs_min(t1, t2), hs_min(t3, t4)), hs_min(t5, t6));
  double tmax = hs_min(hs_min(hs_max(t1, t2), hs_max(t3, t4)), hs_max(t5, t6));
  return !(tmax < 0 || tmin > tmax);
}

// Conservative float version of the same test, used only to CULL.  The boxes are the double boxes
// rounded outward; the ray origin is widened to [o - e, o + e] with
//   e = 2^-21 * (max|o_k| + largest |box coordinate| in the scene),
// which covers the float roundings of the origin, of o +- e, of d, of 1/d, of origin*(1/d) and of
// the fused multiply-add (seven roundings, each <= 2^-24 relative to |o| + |plane|; e allows eight).  `lo` always pairs with o+e and `hi` with o-e: for
// either sign of d that moves the entry distance down and the exit distance up.  So whenever the
// exact test passes, this one passes; the converse errors only make the traversal look at a few
// more triangles, each of which then gets the exact double test.  Rays with a zero (or denormal)
// direction component never come here (the reference's inf/NaN arithmetic decides those exactly).
struct RayF {
  float ix, iy, iz;     // 1 / d
  float pix, piy, piz;  // (o + e) * (1/d)
  float mix, miy, miz;  // (o - e) * (1/d)
};

// Which rays take the exact double walk instead of the conservative float cull:
//  * a direction component outside [2^-100, 2^100) in magnitude: zero components are the reference's inf/NaN case
//    (SURVEY App. A-N1), and the range keeps 1/d and the products of the float test finite and normal;
//  * an origin farther from the coordinate origin than 4096 x the largest box coordinate (a reflection that left the
//    scene along an unbounded plane and looks back at it): float cannot resolve the boxes from there — the widened
//    test would pass every box and the ray would visit the whole tree (measured: 331 k nodes for one shadow ray of the
//    1 M-triangle synthetic scene, a one-second tail) — while the double test culls as usual.
// Decided on the exponent bits with integer compares.
__device__ __forceinline__ bool needs_exact_walk(const Ray& r, const SceneView& S) {
  const uint32_t lo = 0x39B00000u, span = 0x46300000u - 0x39B00000u;  // biased exponents 923 (2^-100) and 1123 (2^100)
  const uint32_t hx = (uint32_t)__double2hiint(r.d.x) & 0x7fffffffu, hy = (uint32_t)__double2hiint(r.d.y) & 0x7fffffffu,
                 hz = (uint32_t)__double2hiint(r.d.z) & 0x7fffffffu;
  const uint32_t lim = (uint32_t)__double2hiint(4096.0 * (double)S.abs_max);
  // distances are taken from the centre of the scene's boxes, like the float boxes themselves
  const uint32_t ox = (uint32_t)__double2hiint(r.o.x - S.center[0]) & 0x7fffffffu,
                 oy = (uint32_t)__double2hiint(r.o.y - S.center[1]) & 0x7fffffffu,
                 oz = (uint32_t)__double2hiint(r.o.z - S.center[2]) & 0x7fffffffu;
  return !((hx - lo < span) & (hy - lo < span) & (hz - lo < span) & (ox < lim) & (oy < lim) & (oz < lim));
}

// The float boxes are stored relative to S.center (the middle of all tree boxes), so that a scene far from the
// coordinate origin keeps float's full resolution; the ray origin is moved the same way (one correctly rounded double
// subtraction: relative error 2^-53 of the result, far inside e's budget).
__device__ __forceinline__ RayF make_rayf(const Ray& r, const SceneView& S) {
  RayF f;
  const float abs_max = S.abs_max;
  const float ox = (float)(r.o.x - S.center[0]), oy = (float)(r.o.y - S.center[1]), oz = (float)(r.o.z - S.center[2]);
  // (float)max|o_k| == max|(float)o_k|: rounding is monotonic
  const float e = 4.76837158203125e-07f * (fmaxf(fmaxf(fabsf(ox), fabsf(oy)), fabsf(oz)) * 1.0000002f + abs_max);
  f.ix = __frcp_rn((float)r.d.x);  // two roundings (d -> float, reciprocal): still inside e's budget of eight
  f.iy = __frcp_rn((float)r.d.y);
  f.iz = __frcp_rn((float)r.d.z);
  f.pix = (ox + e) * f.ix;
  f.piy = (oy + e) * f.iy;
  f.piz = (oz + e) * f.iz;
  f.mix = (ox - e) * f.ix;
  f.miy = (oy - e) * f.iy;
  f.miz = (oz - e) * f.iz;
  return f;
}

// t = plane * (1/d) - origin * (1/d) as one fused multiply-add per plane (an explicit intrinsic:
// -fmad=false only stops the compiler from fusing the reference's double arithmetic).
__device__ __forceinline__ bool slab32(const RayF& f, float lx, float ly, float lz, float hx, float hy, float hz, float& tmin) {
  const float t1 = __fmaf_rn(lx, f.ix, -f.pix), t2 = __fmaf_rn(hx, f.ix, -f.mix);
  const float t3 = __fmaf_rn(ly, f.iy, -f.piy), t4 = __fmaf_rn(hy, f.iy, -f.miy);
  const float t5 = __fmaf_rn(lz, f.iz, -f.piz), t6 = __fmaf_rn(hz, f.iz, -f.miz);
  tmin = fmaxf(fmaxf(fminf(t1, t2), fminf(t3, t4)), fminf(t5, t6));
  const float tmax = fminf(fminf(fmaxf(t1, t2), fmaxf(t3, t4)), fmaxf(t5, t6));
  return !(tmax < 0.0f || tmin > tmax);
}

// Cell of the cube maps around a point light (light_maps.cpp) for the direction of p - L, in float: the maps are
// marked one cell beyond every triangle, far more than the ~1e-6 of a face these roundings can move a direction.
// Face 2k + (v[k] < 0) for the largest |v[k]|, coordinates (v[a], v[b]) / |v[k]| with (a, b) = (1,2), (0,2), (0,1).
// kEmpty when p is (nearly) the light itself or not finite: no cull then.
__device__ __forceinline__ uint32_t light_map_cell(const V3& p, const V3& lp, uint32_t R) {
  const float vx = (float)(p.x - lp.x), vy = (float)(p.y - lp.y), vz = (float)(p.z - lp.z);
  const float ax = fabsf(vx), ay = fabsf(vy), az = fabsf(vz);
  uint32_t face;
  float w, s, t;
  if (ax >= ay && ax >= az) {
    face = vx < 0 ? 1u : 0u;
    w = ax, s = vy, t = vz;
  } else if (ay >= az) {
    face = vy < 0 ? 3u : 2u;
    w = ay, s = vx, t = vz;
  } else {
    face = vz < 0 ? 5u : 4u;
    w = az, s = vx, t = vy;
  }
  if (!(w > 1e-30f && w < 1e30f)) return kEmpty;
  const float iw = __frcp_rn(w), half = 0.5f * (float)R;
  const int top = (int)R - 1;
  const int ci = min(max((int)floorf((s * iw + 1.0f) * half), 0), top);
  const int cj = min(max((int)floorf((t * iw + 1.0f) * half), 0), top);
  return (face * R + (uint32_t)cj) * R + (uint32_t)ci;
}

// True when no triangle of the mesh behind cube map `mi` can lie between p and the light: every triangle that covers
// the direction of p - L is farther from the light than p is (the map holds a lower bound of that distance per cell,
// +inf where nothing covers it).  inFrontOfLight (RayHs.hs:84-87) would discard whatever the walk found.
__device__ __forceinline__ bool light_map_clears(const SceneView& S, uint32_t mi, uint32_t cell, float dist_up) {
  const size_t cells = (size_t)6 * S.light_map_res * S.light_map_res;
  return dist_up < __ldg(S.light_maps + (size_t)mi * cells + cell);
}

// Closest-hit candidate: key (t asc, leaf desc, position-in-leaf asc) inside one mesh
// (KDTree.hs:109-115 right child wins ties; Geometry.hs:54-57 first minimum inside a leaf),
// strict `<` across objects (RayHs.hs:67-71 first object wins ties).  The device triangle record
// carries both order keys: `pad_` = first slot of the reference leaf (leaves are numbered left to
// right by it), `tri_id` = index in `triangles mesh`, which is also the order inside a leaf because
// the build's list comprehensions keep the list order (KDTree.hs:85-88).  They are only read on an
// exact tie in t.
struct Closest {
  double t, u, v;
  uint32_t slot;
  int obj, cur_obj;
  const rh_tri* tris;
  __device__ __forceinline__ bool wins_tie(uint32_t s) const {
    const uint2 mine = *(const uint2*)&tris[s].tri_id, held = *(const uint2*)&tris[slot].tri_id;  // (tri_id, leaf key)
    return mine.y > held.y || (mine.y == held.y && mine.x < held.x);
  }
  __device__ __forceinline__ bool offer(const Ray&, double tt, double uu, double vv, uint32_t s, double& bound) {
    // (cur_obj < obj only happens when objects are not visited in scene order — the sphere tree is walked after the
    // linear list: the first object of the scene list wins a tie, RayHs.hs:67-71)
    if (tt < t || (tt == t && (cur_obj < obj || (obj == cur_obj && wins_tie(s))))) {
      t = tt;
      u = uu;
      v = vv;
      slot = s;
      obj = cur_obj;
      bound = tt * kPruneSlack;
    }
    return false;
  }
  // A top-level sphere met while walking the sphere tree (any order): the reference's scan keeps the first
  // object of the list among equal times (RayHs.hs:67-71), i.e. the lowest object index.
  __device__ __forceinline__ bool offer_object(const Ray&, double tt, int o, double& bound) {
    if (tt < t || (tt == t && o < obj)) {
      t = tt;
      obj = o;
      bound = tt * kPruneSlack;
    }
    return false;
  }
};

// Shadow candidate (RayHs.hs:74-87): any hit in front of the light ends the query.
struct AnyHit {
  V3 lpos;
  double dl2;  // sqrDist origin lightPos
  bool directional;
  __device__ __forceinline__ bool in_front(const Ray& r, double tt) const {
    if (directional) return true;
    return dl2 > sqrDist(r.o, rayAt(r, tt));
  }
  __device__ __forceinline__ bool offer(const Ray& r, double tt, double, double, uint32_t, double&) const {
    return in_front(r, tt);
  }
  __device__ __forceinline__ bool offer_object(const Ray& r, double tt, int, double&) const { return in_front(r, tt); }
};

// Prefetches (RH_PREFETCH bit 0: the lines of a leaf's triangle records beyond the first when the leaf is entered; bit 1:
// the node record of a child that is stacked for later).  A lone warp walks at the latency of its loads — an L2 hit is
// ~250 cycles, an L1 hit ~32 — and the records a walk will need next are known one step ahead.
#ifndef RH_PREFETCH
#define RH_PREFETCH 0
#endif
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// Mesh.hs:59-82 triangleIntersection over the `count` triangles of one leaf (Geometry.hs:54-57).
// The accept/reject decision is the reference's expression evaluated on the reference's values
// of det, u, v, t.  Before the division, a triangle is dropped early only when that expression is
// certain to reject it: with s = sign(det), u = idet*un and |idet*|det| - 1| <= 2^-52,
//   s*un < -1e-100            =>  u < 0        s*un > |det|(1+1e-12)        =>  u > 1
//   s*vn < -1e-100            =>  v < 0        s*(un+vn) > |det|(1+1e-12)   =>  u+v > 1
//   s*tn < |det|*eps(1-1e-12) =>  t < eps      s*tn > |det|*bound           =>  t > best t (or beyond the light)
// (the 1e-100 guard keeps idet*un away from underflow to -0, which `u < 0` would not reject).
template <bool COUNT, class Sink>
__device__ __forceinline__ bool test_leaf(const rh_tri* __restrict__ tris, uint32_t first, uint32_t count, const Ray& r,
                                          Sink& sink, double& bound, Cnt<COUNT>& cnt, const uint32_t* __restrict__ index = nullptr) {
#if RH_PREFETCH & 1
  if (!index && count > 1) {  // the records are consecutive: first .. first + count - 1, 80 bytes each
    const char* base = (const char*)(tris + first);
    for (uint32_t off = 128; off < count * (uint32_t)sizeof(rh_tri) + 127u; off += 128) prefetch_l1(base + off);
  }
#endif
  for (uint32_t k = 0; k < count; k++) {
    const uint32_t slot = index ? __ldg(index + first + k) : first + k;  // (exact walk over the reference tree's leaves)
    const double2* tp = (const double2*)(tris + slot);
    const double2 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2), d = __ldg(tp + 3);
    const double e2z = __ldg((const double*)(tp + 4));
    RH_CNT(tri, 1);
    RH_DBG(dt);
    if constexpr (COUNT) {
      const unsigned peers = __match_any_sync(__activemask(), slot);
      if ((threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) cnt.wtri += 1;  // triangle records fetched (once per warp instruction)
    }
    const V3 p0 = mk(a.x, a.y, b.x), e1 = mk(b.y, c.x, c.y), e2 = mk(d.x, d.y, e2z);
    const V3 p = cross(r.d, e2);
    const double det = dot(e1, p);
    const double adet = fabs(det);
    if (adet < kEps) continue;
    const bool safe = adet < 1e100;
    const V3 t0 = r.o - p0;
    const double un = dot(t0, p);
    const double sun = det < 0 ? -un : un;
    const double over = adet * 1.000000000001;
    if (safe && (sun < -1e-100 || sun > over)) continue;
    const V3 q = cross(t0, e1);
    const double vn = dot(r.d, q);
    const double svn = det < 0 ? -vn : vn;
    if (safe && (svn < -1e-100 || sun + svn > over)) continue;
    const double tn = dot(e2, q);
    const double stn = det < 0 ? -tn : tn;
    if (safe && (stn < adet * (kEps * 0.999999999999) || stn > adet * bound)) continue;
    const double idet = 1 / det;
    const double u = idet * un;
    const double v = idet * vn;
    const double t = idet * tn;
    if (u < 0 || u > 1 || v < 0 || (u + v) > 1 || t < kEps) continue;
    if (sink.offer(r, t, u, v, slot, bound)) return true;
  }
  return false;
}

__device__ __forceinline__ bool sphere_time(const Ray& r, const DObject& ob, double& time);

// Leaf of the sphere tree: `count` object indices at refs[first..]; each gets the reference's sphere test
// (Geometry.hs:81-95).  Shadow queries skip emitters (isOccluder, RayHs.hs:81-82).
template <bool COUNT, class Sink>
__device__ __forceinline__ bool test_sphere_leaf(const Ctx& cx, uint32_t first, uint32_t count, const Ray& r, Sink& sink,
                                                 double& bound, bool skip_emitters, Cnt<COUNT>& cnt) {
  for (uint32_t k = 0; k < count; k++) {
    const uint32_t oi = __ldg(cx.S->sphere_refs + first + k);
    const DObject& ob = cx.objects[oi];
    if (skip_emitters && ob.is_emitter) continue;
    RH_CNT(prim, 1);
    double time;
    if (sphere_time(r, ob, time) && sink.offer_object(r, time, (int)oi, bound)) return true;
  }
  return false;
}

// One inner node of the cull tree: both child boxes against the float ray; the nearer surviving child becomes `ref`,
// the farther one is stacked with its entry distance.  False when neither survives (the caller pops).
template <bool COUNT>
__device__ __forceinline__ bool node_step(const Ctx& cx, uint32_t& ref, const RayF& f, float fb, Stack& st, int& sp,
                                          Cnt<COUNT>& cnt) {
  const float4* np = ref < cx.S->n_smem_nodes ? (const float4*)&cx.sm_nodes[ref] : (const float4*)&cx.S->wide32[ref];
  const float4 b0 = np[0], b1 = np[1], b2 = np[2];
  const uint2 cw = *(const uint2*)(np + 3);  // child0, child1
  RH_CNT(nodes, 1);
  RH_DBG(dn);
  if constexpr (COUNT) {
    // records read from global memory (not the staged top levels), counted once per warp instruction: lanes that
    // visit the same node share one fetch
    if (ref >= cx.S->n_smem_nodes) {
      const unsigned peers = __match_any_sync(__activemask(), ref);
      if ((threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) cnt.gnodes += 1;
    }
  }
  bool h0 = false, h1 = false;
  float tm0 = 0, tm1 = 0;
  if (cw.x != kEmpty) {
    RH_CNT(box, 1);
    h0 = slab32(f, b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, tm0) && !(tm0 > fb);
  }
  if (cw.y != kEmpty) {
    RH_CNT(box, 1);
    h1 = slab32(f, b1.z, b1.w, b2.x, b2.y, b2.z, b2.w, tm1) && !(tm1 > fb);
  }
  if (h0 && h1) {
    if constexpr (COUNT) {
      if (sp >= kShortStack) cnt.deep += 1;
    }
    if (tm1 < tm0) {
      st.push(sp, cw.x, tm0);
      ref = cw.y;
    } else {
      st.push(sp, cw.y, tm1);
      ref = cw.x;
    }
#if RH_PREFETCH & 2
    {
      const uint32_t far = (tm1 < tm0) ? cw.x : cw.y;  // popped later: its record (or its first triangle) can be on its way
      if (far & kLeafBit) {
        if (!(far & kSphereLeafBit)) prefetch_l1(cx.S->tris + (far & kLeafFirstMask));
      } else if (far >= cx.S->n_smem_nodes) {
        prefetch_l1(&cx.S->wide32[far]);
      }
    }
#endif
    return true;
  }
  if (h0) {
    ref = cw.x;
    return true;
  }
  if (h1) {
    ref = cw.y;
    return true;
  }
  return false;
}

// KDTree.hs:96-107 rayInter, ordered and pruned, culling with the conservative float boxes.
// Subtrees are skipped only when their entry distance exceeds `bound` (the best t so far times
// 1 + 1e-7, or the light distance), both when they are first met and again when they are popped.
// "while-while" form: a lane that reaches a leaf waits at the end of the inner loop until the
// other lanes of its warp hold a leaf too (or are done), so the long triangle loop runs with as
// many lanes as possible.  Returns true when the sink asked to stop (any-hit).
// SPHERES: the tree is the top-level sphere tree (leaves hold object indices) instead of a mesh tree.
template <bool COUNT, class Sink, bool SPHERES = false>
__device__ __forceinline__ bool traverse(const Ctx& cx, uint32_t root, const Ray& r, const RayF& f, double& bound, Sink& sink,
                                         Stack& st, Cnt<COUNT>& cnt, bool skip_emitters = false) {
  int sp = 0;
  uint32_t ref = root;
  const rh_tri* tris = cx.S->tris;
  for (;;) {
    while (!(ref & kLeafBit)) {
      const float fb = __double2float_ru(bound);
      if (node_step<COUNT>(cx, ref, f, fb, st, sp, cnt)) continue;
      uint2 e;
      do {
        if (sp == 0) return false;
        e = st.pop(sp);
      } while (__uint_as_float(e.y) > fb);
      ref = e.x;
    }
    const uint32_t first = ref & kLeafFirstMask, count = ((ref >> kLeafCountShift) & (kLeafMaxCount - 1)) + 1;
    if constexpr (SPHERES) {
      if (test_sphere_leaf<COUNT>(cx, first, count, r, sink, bound, skip_emitters, cnt)) return true;
    } else {
      if (test_leaf<COUNT>(tris, first, count, r, sink, bound, cnt)) return true;
    }
    const float fb = __double2float_ru(bound);
    uint2 e;
    do {
      if (sp == 0) return false;
      e = st.pop(sp);
    } while (__uint_as_float(e.y) > fb);
    ref = e.x;
  }
}

// The same walk over the reference's own tree with the reference's own double slab test (GHC min/max NaN semantics
// included): rays with a zero direction component (centre row/column of the image, SURVEY App. A-N1), far origins, and
// RH_FLAG_EXACT_BOXES validation runs.  Cold path: kept out of line; its stack is the thread's global column.
template <bool COUNT, class Sink, bool SPHERES = false>
__device__ __noinline__ bool traverse_exact_impl(const Ctx& cx, uint32_t root, const Ray& r, double& bound, Sink& sink, Stack& st,
                                                 Cnt<COUNT>& cnt, bool skip_emitters) {
  const V3 inv = mk(1 / r.d.x, 1 / r.d.y, 1 / r.d.z);
  int sp = 0;
  uint32_t ref = root, first = 0;
  const rh_tri* tris = cx.S->tris;
  for (;;) {
    if (!(ref & kLeafBit)) {
      const double2* np = (const double2*)&cx.S->wide[ref];
      const double2 b0 = np[0], b1 = np[1], b2 = np[2], b3 = np[3], b4 = np[4], b5 = np[5];
      const uint4 cw = *(const uint4*)(np + 6);
      const uint32_t refine = *(const uint32_t*)(np + 7);  // bit c: child c's box is not a box the reference tests
                                                           // (sphere tree): it always passes here
      RH_CNT(nodes, 2);  // a 128-byte record = two 64-byte units
      RH_CNT(gnodes, 2);
      bool h0 = false, h1 = false;
      double tm0 = 0, tm1 = 0;
      // A box that passes with tmin = +inf is not behind the bound: a zero direction component with the origin on one
      // of the box's planes makes the reference's slab terms inf * 0 = NaN, and GHC's min / max then let the box pass
      // with tmin = +inf whatever its real entry distance (the ray runs in the box's face).  Only a finite tmin prunes.
      if (cw.x != kEmpty) {
        RH_CNT(box, 1);
        h0 = (refine & 1u) || (slab(r, inv, b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, tm0) && !(tm0 > bound && !isinf(tm0)));
      }
      if (cw.y != kEmpty) {
        RH_CNT(box, 1);
        h1 = (refine & 2u) || (slab(r, inv, b3.x, b3.y, b4.x, b4.y, b5.x, b5.y, tm1) && !(tm1 > bound && !isinf(tm1)));
      }
      if (h0 && h1) {
        if (tm1 < tm0) {
          st.push_deep(sp, cw.x, cw.z);
          ref = cw.y;
          first = cw.w;
        } else {
          st.push_deep(sp, cw.y, cw.w);
          ref = cw.x;
          first = cw.z;
        }
        continue;
      }
      if (h0) {
        ref = cw.x;
        first = cw.z;
        continue;
      }
      if (h1) {
        ref = cw.y;
        first = cw.w;
        continue;
      }
    } else if constexpr (SPHERES) {
      if (test_sphere_leaf<COUNT>(cx, first, ref & kCountMask, r, sink, bound, skip_emitters, cnt)) return true;
    } else {
      if (test_leaf<COUNT>(tris, first, ref & kCountMask, r, sink, bound, cnt, cx.S->exact_index)) return true;
    }
    if (sp == 0) return false;
    const uint2 e = st.pop_deep(sp);
    ref = e.x;
    first = e.y;
  }
}

// The out-of-line walk gets COPIES of the ray, the sink, the tables and the stack handle: handing it the caller's own
// objects by reference would pin those — the hottest values of every kernel — in local memory for the whole kernel
// (ncu on an earlier build: 57 GB of local stores per pass-0 launch, every one written through to L2).
template <bool COUNT, class Sink, bool SPHERES = false>
__device__ __forceinline__ bool traverse_exact(const Ctx& cx, uint32_t root, const Ray& r, double& bound, Sink& sink, Stack& st,
                                               Cnt<COUNT>& cnt, bool skip_emitters = false) {
  Ctx cx_copy = cx;
  Ray r_copy = r;
  Sink sink_copy = sink;
  Stack st_copy = st;
  double bound_copy = bound;
  const bool stop = traverse_exact_impl<COUNT, Sink, SPHERES>(cx_copy, root, r_copy, bound_copy, sink_copy, st_copy, cnt, skip_emitters);
  sink = sink_copy;
  bound = bound_copy;
  return stop;
}

// Geometry.hs:70-79 (plane): hit iff |d.n| > 0 and time = n.(p-o) / (d.n) > 0.  The quotient is
// only formed when it can matter: opposite signs (or a zero numerator) give time <= 0 exactly, and
// |num| > limit*|den| gives time > limit (limit = best t so far, or the light distance with its slack).
__device__ __forceinline__ bool plane_time(const Ray& r, const DObject& ob, double limit, double& time) {
  const V3 p = ld3(ob.a), n = ld3(ob.b);
  const double dDotn = dot(r.d, n);
  const double num = dot(n, p - r.o);
  if (!(fabs(dDotn) > 0)) return false;
  if ((num > 0) != (dDotn > 0) && num == num) return false;  // quotient <= 0 (or -0): `time > 0` fails
  if (fabs(num) > limit * fabs(dDotn) * 1.000000000001) return false;
  time = num / dDotn;
  return time > 0;
}
// Geometry.hs:81-95 (sphere): first positive root.
__device__ __forceinline__ bool sphere_time(const Ray& r, const DObject& ob, double& time) {
  const V3 ct = ld3(ob.a);
  const double rad = ob.b[0];
  const double a = dot(r.d, r.d);
  const double b = 2.0 * dot(r.d, r.o - ct);
  const double c = sqrLen(r.o - ct) - rad * rad;
  const double delta = b * b - 4.0 * a * c;
  if (delta < 0.0) return false;
  const double t0 = 0.5 * ((-b) - sqrt(delta)) / a;
  if (t0 > 0) {
    time = t0;
    return true;
  }
  const double t1 = 0.5 * ((-b) + sqrt(delta)) / a;
  if (t1 > 0) {
    time = t1;
    return true;
  }
  return false;
}

// RayHs.hs:58-71 closestIntersection over the object list.
template <bool COUNT>
__device__ __forceinline__ void closest_hit(const Ctx& cx, const Ray& r, bool exact, Closest& best, Stack& st, Cnt<COUNT>& cnt) {
  const RayF f = make_rayf(r, *cx.S);
  best.t = __longlong_as_double(0x7ff0000000000000LL);
  best.u = best.v = 0;
  best.slot = 0;
  best.tris = cx.S->tris;
  best.obj = -1;
  const uint32_t sphere_root = cx.S->sphere_root;
  const uint32_t n = cx.S->n_lin;  // == n_objects, in scene order, unless the spheres live in the sphere tree
  for (uint32_t k = 0; k < n; k++) {
    const uint32_t i = sphere_root == kEmpty ? k : __ldg(cx.S->lin_objs + k);
    const DObject& ob = cx.objects[i];
    const int kind = ob.kind;
    if (kind == RH_OBJ_MESH) {
      const uint32_t root = ob.root;
      if (root == kEmpty) continue;
      best.cur_obj = (int)i;
      double bound = best.t * kPruneSlack;
      if (exact)
        traverse_exact<COUNT>(cx, root, r, bound, best, st, cnt);
      else
        traverse<COUNT>(cx, root, r, f, bound, best, st, cnt);
    } else {
      double time;
      RH_CNT(prim, 1);
      const bool hit = (kind == RH_OBJ_PLANE) ? plane_time(r, ob, best.t, time) : sphere_time(r, ob, time);
      if (hit && time < best.t) {
        best.t = time;
        best.obj = (int)i;
      }
    }
  }
  if (sphere_root != kEmpty) {
    double bound = best.t * kPruneSlack;
    if (exact)
      traverse_exact<COUNT, Closest, true>(cx, sphere_root, r, bound, best, st, cnt);
    else
      traverse<COUNT, Closest, true>(cx, sphere_root, r, f, bound, best, st, cnt);
  }
}

// Geometry.hs:39 Hit of the primitive closest_hit chose (object `ob` of kind `okind`): the point, the normal as the
// reference returns it (mesh normals interpolated, not renormalised: Mesh.hs:81) and, when `need_uv`, the uv.
// (query_closest_kernel; trace_kernel keeps the same lines inline, see there.)
template <bool COUNT>
__device__ __forceinline__ void rebuild_hit(const SceneView& S, const DObject& ob, int okind, const Ray& r, const Closest& best,
                                            bool need_uv, V3& p, V3& n, double& tu, double& tv, Cnt<COUNT>& cnt) {
  p = rayAt(r, best.t);
  if (okind == RH_OBJ_MESH) {
    const double* sh = (const double*)(S.shade + best.slot);
    RH_CNT(shade, 1);
    const double wu = best.u, wv = best.v, ww = 1 - best.u - best.v;
    // barycentricInterp u n1 v n2 (1-u-v) n0 = mul a p + mul b q + mul c r   (Mesh.hs:57, 81)
    n = mul(wu, ld3(sh + 3)) + mul(wv, ld3(sh + 6)) + mul(ww, ld3(sh));
    if (need_uv) {
      tu = wu * sh[11] + wv * sh[13] + ww * sh[9];
      tv = wu * sh[12] + wv * sh[14] + ww * sh[10];
    }
  } else if (okind == RH_OBJ_PLANE) {  // Geometry.hs:70-79
    n = ld3(ob.b);
    if (need_uv) {
      const V3 tg = ld3(ob.c);
      const V3 bt = cross(tg, n);
      const V3 rel = p - ld3(ob.a);
      tu = dot(tg, rel);
      tv = dot(bt, rel);
    }
  } else {  // Geometry.hs:83-96
    n = normalize(p - ld3(ob.a));
    if (need_uv) {
      tu = kPiInv * atan(n.z / n.x);
      tv = kPiInv * acos(n.y);
    }
  }
}

// RayHs.hs:74-87 shadowIntersection: true when some non-emitter object has a hit in front of the light.
// (General form over the object list; the kernels for <= 32 lights use the compact occluder tables instead.)
template <bool COUNT>
__device__ __forceinline__ bool occluded(const Ctx& cx, const Ray& r, bool exact, const rh_light& L, Stack& st, Cnt<COUNT>& cnt) {
  const RayF f = make_rayf(r, *cx.S);
  AnyHit sink;
  sink.directional = (L.kind == RH_LIGHT_DIRECTIONAL);
  sink.lpos = ld3(L.vec);
  sink.dl2 = sink.directional ? 0.0 : sqrDist(r.o, sink.lpos);
  // hits farther than the light cannot be in front of it; 1e-6 relative slack covers |d| != 1 rounding
  const double far = sink.directional ? __longlong_as_double(0x7ff0000000000000LL)
                                      : sqrt(sink.dl2) * 1.000001 / sqrt(dot(r.d, r.d));
  const uint32_t sphere_root = cx.S->sphere_root;
  const uint32_t n = cx.S->n_lin;
  for (uint32_t k = 0; k < n; k++) {
    const uint32_t i = sphere_root == kEmpty ? k : __ldg(cx.S->lin_objs + k);
    const DObject& ob = cx.objects[i];
    if (ob.is_emitter) continue;  // isOccluder, RayHs.hs:81-82
    const int kind = ob.kind;
    if (kind == RH_OBJ_MESH) {
      const uint32_t root = ob.root;
      if (root == kEmpty) continue;
      double bound = far;
      const bool hit = exact ? traverse_exact<COUNT>(cx, root, r, bound, sink, st, cnt)
                             : traverse<COUNT>(cx, root, r, f, bound, sink, st, cnt);
      if (hit) return true;
    } else {
      double time;
      RH_CNT(prim, 1);
      const bool hit = (kind == RH_OBJ_PLANE) ? plane_time(r, ob, far, time) : sphere_time(r, ob, time);
      if (hit && sink.in_front(r, time)) return true;
    }
  }
  if (sphere_root != kEmpty) {
    double bound = far;
    return exact ? traverse_exact<COUNT, AnyHit, true>(cx, sphere_root, r, bound, sink, st, cnt, true)
                 : traverse<COUNT, AnyHit, true>(cx, sphere_root, r, f, bound, sink, st, cnt, true);
  }
  return false;
}

// ------------------------------------------------------------------ Material.hs / Light.hs / ColorMap.hs
__device__ __forceinline__ double r0f(double n1, double n2) {  // Material.hs:22-24
  const double q = (n1 - n2) / (n1 + n2);
  return q * q;
}
__device__ __forceinline__ double fresnel(double ior, double cos0) {  // Material.hs:26-29
  const double r = r0f(1.0, ior);
  const double x = 1 - cos0;
  const double x2 = x * x;
  const double x5 = (x2 * x2) * x;  // GHC (^): square-and-multiply
  return r + (1 - r) * x5;
}

// Data.Fixed.mod' n d = n - fromInteger (floor (toRational n / toRational d)) * d   (exact rational floor)
__device__ __noinline__ double hs_mod1(double n, double d) {
  if (!isfinite(n) || !isfinite(d) || d == 0) return __longlong_as_double(0x7ff8000000000000LL);
  double q = floor(n / d);
  if (fabs(q) >= 4503599627370496.0) return n - q * d;
  if (d > 0) {
    while (__fma_rn(-q, d, n) < 0) q -= 1;
    while (__fma_rn(-(q + 1), d, n) >= 0) q += 1;
  } else {
    while (__fma_rn(-q, d, n) > 0) q -= 1;
    while (__fma_rn(-(q + 1), d, n) <= 0) q += 1;
  }
  return n - q * d;
}
__device__ __forceinline__ long long hs_mod_int(long long a, long long m) {
  long long r = a % m;
  return (r != 0 && ((r < 0) != (m < 0))) ? r + m : r;
}

// ColorMap.hs:18-58
template <bool COUNT>
__device__ __noinline__ V3 color_at(const SceneView& S, const rh_material& m, double u, double v, Cnt<COUNT>& cnt) {
  const V3 c1 = ld3(m.color1);
  if (m.cmap_kind == RH_CMAP_FLAT) return c1;
  if (m.cmap_kind == RH_CMAP_CHECKER) {
    const double s = m.size;
    return ((hs_mod1(u, s) - (0.5 * s)) * (hs_mod1(v, s) - (0.5 * s)) < 0) ? c1 : ld3(m.color2);
  }
  const rh_texture tx = S.textures[m.texture];
  const double* px = S.texels + 3 * tx.offset;
  const double uu = hs_mod1(u, 1) * (double)tx.w;  // toPixel / repeatUV
  const double vv = hs_mod1(v, 1) * (double)tx.h;
  const long long ui = (long long)rint(uu);  // round: half to even
  const long long vi = (long long)rint(vv);
  const long long x0 = hs_mod_int(ui - 1, tx.w), x1 = hs_mod_int(ui, tx.w);
  const long long y0 = hs_mod_int(vi - 1, tx.h), y1 = hs_mod_int(vi, tx.h);
  const double lx = uu - (double)(ui - 1) - 0.5;
  const double ly = vv - (double)(vi - 1) - 0.5;
  RH_CNT(texel, 4);
  const V3 c0 = ld3(px + 3 * (x0 + (long long)tx.w * y0));  // Bitmap.hs:17-18
  const V3 c1t = ld3(px + 3 * (x1 + (long long)tx.w * y0));
  const V3 c2 = ld3(px + 3 * (x0 + (long long)tx.w * y1));
  const V3 c3 = ld3(px + 3 * (x1 + (long long)tx.w * y1));
  const V3 cx0 = mul(lx, c1t) + mul(1 - lx, c0);  // bilinearInterp, ColorMap.hs:41-45
  const V3 cx1 = mul(lx, c3) + mul(1 - lx, c2);
  return mul(ly, cx1) + mul(1 - ly, cx0);
}

// ------------------------------------------------------------------ queues: slabs, warp-aggregated compaction
__device__ __forceinline__ uint64_t pack_bits(uint32_t sample, int depth, int kind, uint32_t mat) {
  return (uint64_t)sample | ((uint64_t)(depth & 0xff) << 32) | ((uint64_t)(kind & 0xff) << 40) | ((uint64_t)(mat & 0xffff) << 48);
}

// A warp's open slab of an output queue: entries [base, base + used) are written.  One per warp, in shared memory.
struct SlabWriter {
  uint32_t base, used, pushed;
  __device__ __forceinline__ void init() { base = kEmpty; used = 0; pushed = 0; }
};

// Slots for the lanes of ballot `m` (all 32 lanes call this, converged, with m != 0): the open slab first, then a new
// one reserved with ONE atomic on the queue's slab counter — one global atomic per kSlab entries instead of one per
// push.  The slab a push completes gets its fill count here; the last, partly filled one at slab_close.  Returns
// kEmpty for an entry that does not fit the queue (overflow is flagged; the host re-renders with larger queues).
// `live_from`: the queue is a ring of capacity / kSlab slabs addressed by a running counter; the slabs from `live_from` on
// are still in use (0 and a counter that starts at 0 for a queue that is simply filled once).
__device__ __forceinline__ uint32_t slab_reserve(SlabWriter& w, unsigned m, uint32_t lane, uint32_t* slab_counter, uint32_t* fill,
                                                 uint32_t capacity, uint32_t* overflow, uint32_t live_from = 0) {
  // `w` lives in the warp's shared memory: every lane reads it, then lane 0 writes the new state
  const uint32_t n = __popc(m), rank = __popc(m & ((1u << lane) - 1));
  __syncwarp();  // lane 0's update of the previous push is visible
  const uint32_t base = w.base, used = w.used;
  const uint32_t room = (base == kEmpty) ? 0u : kSlab - used;
  __syncwarp();  // every lane has read the state before lane 0 replaces it
  if (n <= room) {
    if (lane == 0) {
      w.used = used + n;
      w.pushed += n;
    }
    return base + used + rank;
  }
  uint32_t ns = 0;
  if (lane == 0) {
    if (base != kEmpty) fill[base / kSlab] = kSlab;  // this push fills the open slab to the brim
    ns = atomicAdd(slab_counter, 1u);
  }
  ns = __shfl_sync(kFull, ns, 0);
  const bool full = ns - live_from >= capacity / kSlab;
  ns %= capacity / kSlab;
  if (lane == 0) {
    if (full) *overflow = 1;
    w.base = full ? kEmpty : ns * kSlab;
    w.used = full ? 0u : n - room;
    w.pushed += n;
  }
  if (rank < room) return base + used + rank;
  return full ? kEmpty : ns * kSlab + (rank - room);
}
__device__ __forceinline__ void slab_close(const SlabWriter& w, uint32_t lane, uint32_t* fill, uint32_t* items) {
  __syncwarp();
  if (lane == 0) {
    if (w.base != kEmpty) fill[w.base / kSlab] = w.used;
    if (w.pushed) atomicAdd(items, w.pushed);
  }
}

// Work claim of a persistent warp: consecutive UNITS of kUnit work items (kSlab / kUnit per slab).  Guided
// self-scheduling: whole slabs (one atomic per 128 items) while plenty of work is left, then whole 32-item groups, and
// single units near the end of the queue and in small launches.  The secondary passes are short launches whose duration
// is set by their slowest warp, and a lone warp is latency-bound: its lanes walk in lock-step (a round lasts as long as
// its longest walk, ~1 us per node step with nothing to hide the loads behind), so near the end it is faster to spread
// 32 items over four warps with 8 lanes each than to give them to one (measured per warp with -DRH_WARP_TIMES: on one
// eighth of the bench frame the last percent of the warps ran 2-3x longer than the median with 32-item claims).
// Returns (first unit, number of units); first >= n_units: nothing left.
#ifndef RH_CLAIM_UNIT
#define RH_CLAIM_UNIT 8
#endif
#ifndef RH_CLAIM_DIV
#define RH_CLAIM_DIV 4  // a claim takes 1 / (RH_CLAIM_DIV x warps) of what is left (bench frame / one eighth of it: 2: 38.43 / 6.00 ms, 4: 38.31 / 5.91, 8: 39.39 / 6.22, 16: 42.09 / 7.35)
#endif
constexpr uint32_t kUnit = RH_CLAIM_UNIT;
constexpr uint32_t kSlabUnits = kSlab / kUnit, kGroupUnits = 32 / kUnit;
static_assert(kUnit >= 1 && kUnit <= 32 && 32 % kUnit == 0, "a claim unit divides a warp's 32 lanes");
// `seen`: where the cursor stood after this warp's previous claim (a lower bound of where it stands now; before the
// first claim: as if every warp ahead of this one had taken a slab) — the estimate of the work left costs no extra
// round trip to the cursor's cache line.
__device__ __forceinline__ uint2 claim_units(uint32_t* cursor, uint32_t n_units, uint32_t total_warps, uint32_t lane, uint32_t& seen) {
  uint2 c = make_uint2(0, 1);
  if (lane == 0) {
    const uint32_t left = seen < n_units ? n_units - seen : 0;
    uint32_t want = min(kSlabUnits, max(1u, left / ((uint32_t)RH_CLAIM_DIV * total_warps)));
    if (want >= kGroupUnits) want -= want % kGroupUnits;  // whole 32-item groups
    c.y = want;
    c.x = atomicAdd(cursor, c.y);
  }
  c.x = __shfl_sync(kFull, c.x, 0);
  c.y = __shfl_sync(kFull, c.y, 0);
  seen = c.x + c.y;
  return c;
}
// The next piece of a claim [u, end): at most 32 consecutive items of one slab.  Returns the slab, the first item's
// offset in it and the number of items, and advances u.
__device__ __forceinline__ void next_piece(uint32_t& u, uint32_t end, uint32_t& slab, uint32_t& off, uint32_t& n) {
  slab = u / kSlabUnits;
  const uint32_t uo = u % kSlabUnits, nu = min(min(end - u, kGroupUnits), kSlabUnits - uo);
  off = uo * kUnit;
  n = nu * kUnit;
  u += nu;
}

__device__ __forceinline__ void push_ray(bool has, const Ray& r, double w, uint64_t bits, const RayQueue& q, SlabWriter& sw,
                                         uint32_t* slab_counter, uint32_t* overflow, uint32_t lane) {
  const unsigned m = __ballot_sync(kFull, has);
  if (!m) return;
  const uint32_t idx = slab_reserve(sw, m, lane, slab_counter, q.fill, q.capacity, overflow);
  if (has && idx != kEmpty) {
    const size_t cap = q.capacity;
    q.plane[idx] = make_double2(r.o.x, r.o.y);
    q.plane[cap + idx] = make_double2(r.o.z, r.d.x);
    q.plane[2 * cap + idx] = make_double2(r.d.y, r.d.z);
    q.plane[3 * cap + idx] = make_double2(w, __longlong_as_double((long long)bits));
  }
}

// `walk` word of a hit-queue entry: the hit triangle's lit flags (16 bits), or kHitDirect: the entry's colour is a finished
// term (Emmit / ShowNormal / ShowUV) that is added as it is
constexpr uint32_t kHitDirect = 0x80000000u;
struct ShadowTask {
  V3 p, n, cd;
  double w;
  uint32_t sample;  // bit 31: add the 0.2*cd ambient term (Diffuse, RayHs.hs:111-114)
  uint32_t walk, settled;
};

__device__ __forceinline__ void push_shadow(bool has, const ShadowTask& t, const ShadowQueue& q, SlabWriter& sw,
                                            uint32_t* slab_counter, uint32_t* overflow, uint32_t lane, uint32_t live_from = 0) {
  const unsigned m = __ballot_sync(kFull, has);
  if (!m) return;
  const uint32_t idx = slab_reserve(sw, m, lane, slab_counter, q.fill, q.capacity, overflow, live_from);
  if (has && idx != kEmpty) {
    const size_t cap = q.capacity;
    q.plane[idx] = make_double2(t.p.x, t.p.y);
    q.plane[cap + idx] = make_double2(t.p.z, t.n.x);
    q.plane[2 * cap + idx] = make_double2(t.n.y, t.n.z);
    q.plane[3 * cap + idx] = make_double2(t.cd.x, t.cd.y);
    q.plane[4 * cap + idx] = make_double2(t.cd.z, t.w);
    q.sample[idx] = t.sample;
    q.walk[idx] = t.walk;
    if (q.settled) q.settled[idx] = t.settled;  // (the hit queue has no settled masks)
  }
}

__device__ __forceinline__ void accumulate(const ChunkParams& P, uint32_t sample, double w, V3 c) {
  double* a = P.accum + sample;
  atomicAdd(a, w * c.x);
  atomicAdd(a + P.accum_stride, w * c.y);
  atomicAdd(a + 2 * (size_t)P.accum_stride, w * c.z);
}

// ------------------------------------------------------------------ bulk async copies (TMA unit, 1-D form)
// cp.async.bulk.shared::cluster.global with mbarrier completion: one elected lane starts the copy of a contiguous
// tile, the data lands in shared memory without occupying registers or LSU slots, every lane waits on the mbarrier's
// phase before reading.  SASS: UBLKCP, SYNCS.ARRIVE.TRANS64, SYNCS.PHASECHK.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_global, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_global), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

// Image row of a shard-compact row (SURVEY 8e): band b = row / band_height goes to shard b mod G.
__device__ __forceinline__ uint32_t global_row(const ChunkParams& P, uint32_t local_row) {
  const uint32_t lb = local_row / P.band_height, rib = local_row % P.band_height;
  return (lb * P.shard_count + P.shard_index) * P.band_height + rib;
}

// Projection.hs:22-39 rayFromPixel with the per-frame constants hoisted into CameraParams.
__device__ __forceinline__ Ray camera_ray(const CameraParams& cam, double px, double py) {
  const double vx = cam.apw * (px - cam.half_w) / cam.w;
  const double vy = cam.aph * ((-py) + cam.half_h) / cam.h;
  V3 o, d;
  if (cam.projection == RH_PROJ_ORTHOGRAPHIC) {
    o = mk(vx, vy, 0);
    d = mk(0, 0, 1);
  } else {
    d = normalize(mk(vx, vy, cam.f));
    o = mk(0, 0, 0);
  }
  Ray r;
  r.o = o + ld3(cam.pos);
  r.d = mk(cam.m[0] * d.x + cam.m[1] * d.y + cam.m[2] * d.z, cam.m[3] * d.x + cam.m[4] * d.y + cam.m[5] * d.z,
           cam.m[6] * d.x + cam.m[7] * d.y + cam.m[8] * d.z);  // Mat.hs:40-44
  return r;
}

// Value k (0-based) of the SplitMix64 stream seeded with `seed`, as a double in [0, 1): the generator's state after
// k + 1 steps is seed + (k + 1) * gamma, so any value can be produced on its own (csrc/frontend.cpp SplitMix64).
__device__ __forceinline__ double splitmix01(unsigned long long seed, unsigned long long k) {
  unsigned long long z = seed + (k + 1ull) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

// ------------------------------------------------------------------ accumDiffuse (RayHs.hs:89-97): the light fold
// Light.hs:12-17
__device__ __forceinline__ void light_at(const rh_light& L, const V3& p, V3& ld, V3& lc) {
  if (L.kind == RH_LIGHT_DIRECTIONAL) {  // Light.hs:14
    ld = ld3(L.vec);
    lc = ld3(L.color);
  } else {  // Light.hs:15-17
    const V3 lp = ld3(L.vec);
    const double dd = sqrt(sqrDist(lp, p));
    const double s = 1.0 + dd / L.radius;
    const double falloff = 1.0 / (s * s);
    ld = mul(1 / dd, lp - p);
    lc = mul(falloff, ld3(L.color));
  }
}

// Light direction and shadow ray of a (hit, light) pair (Light.hs:12-17, RayHs.hs:93).  `far` bounds the distance from
// the ray origin to the light from above (|o - L| <= |o - p| + |p - L| = 1e-6 |ld| + dd); it only prunes — whether a hit
// is in front of the light is always decided by inFrontOfLight's own comparison (dl2 = +inf for a directional light).
struct LightPair {
  V3 ld, o, lp;
  double dd, far;
  bool directional;
};
__device__ __forceinline__ LightPair make_light_pair(const rh_light& L, const V3& p) {
  LightPair q;
  q.directional = (L.kind == RH_LIGHT_DIRECTIONAL);
  q.lp = ld3(L.vec);
  if (q.directional) {
    q.ld = q.lp;
    q.dd = 0;
    q.far = __longlong_as_double(0x7ff0000000000000LL);
  } else {
    const V3 dv = q.lp - p;
    q.dd = sqrt(sqrLen(dv));  // dist lightPos p = sqrt (sqrDist ..), Vec.hs:118-122: (lp - p).(lp - p)
    q.ld = mul(1 / q.dd, dv);
    q.far = (q.dd + kEps) * 1.000001;
  }
  q.o = p + mul(kEps, q.ld);  // rayEps, Geometry.hs:36
  return q;
}
__device__ __forceinline__ AnyHit make_any_hit(const LightPair& q) {
  AnyHit sink;
  sink.directional = q.directional;
  sink.lpos = q.lp;
  sink.dl2 = q.directional ? 0.0 : sqrDist(q.o, q.lp);
  return sink;
}

// Is the Lambert cull exact for this light?  diffuse (Material.hs:31-33) = (max (l.n) 0 / pi) * (cd (*) lc) is +-0 for
// l.n <= 0 only while cd (*) lc is finite: 0 * inf = NaN in the reference, which prints as channel 255.
__device__ __forceinline__ bool light_is_tame(const rh_light& L) {
  const bool colour = isfinite(L.color[0]) && isfinite(L.color[1]) && isfinite(L.color[2]);
  return colour && (L.kind == RH_LIGHT_DIRECTIONAL || L.radius >= 0);  // radius < 0 can make the falloff 1 / 0
}

// Planes and linear spheres of shadowIntersection (RayHs.hs:74-87) for one pair; true = occluded.
// The plane tests are straight-line: every plane gets the reference's two dot products (Geometry.hs:70-79), and a plane
// is dropped when `abs (d.n) > 0 && time > 0` is certain to fail or time is certain to lie beyond the light (the same
// three rejections as plane_time).  Planes that survive — none in a closed room — get the exact quotient and
// inFrontOfLight (RayHs.hs:84-87) in a cold loop.
// `skip`: planes (of the first 32) that the caller knows cannot lie between the hit and the light.
template <bool COUNT>
__device__ __forceinline__ bool primitives_occlude(const OccPlane* planes, uint32_t n_planes, const OccSphere* spheres,
                                                   uint32_t n_spheres, const LightPair& q, uint32_t skip, Cnt<COUNT>& cnt) {
  bool shadowed = false;
#pragma unroll 1
  for (uint32_t k0 = 0; k0 < n_planes && !shadowed; k0 += 32) {
    uint32_t maybe = 0;
    const uint32_t kn = min(32u, n_planes - k0);
    uint32_t todo = (kn == 32 ? kFull : (1u << kn) - 1u) & (k0 == 0 ? ~skip : kFull);
#pragma unroll 1
    while (todo) {
      const uint32_t k = __ffs(todo) - 1;
      todo &= todo - 1;
      const double2* pl = (const double2*)&planes[k0 + k];
      const double2 u0 = pl[0], u1 = pl[1], u2 = pl[2];  // (px,py) (pz,nx) (ny,nz)
      const V3 pp = mk(u0.x, u0.y, u1.x), pn = mk(u1.y, u2.x, u2.y);
      RH_CNT(prim, 1);
      const double den = dot(q.ld, pn);
      const double num = dot(pn, pp - q.o);
      const bool miss = !(fabs(den) > 0) | (((num > 0) != (den > 0)) & (num == num)) |
                        (fabs(num) > q.far * fabs(den) * 1.000000000001);
      maybe |= (miss ? 0u : 1u) << k;
    }
    if (maybe) {
      Ray r;
      r.o = q.o;
      r.d = q.ld;
      const AnyHit sink = make_any_hit(q);
      while (maybe) {  // cold: exact quotient and inFrontOfLight for the surviving planes
        const uint32_t k = k0 + __ffs(maybe) - 1;
        maybe &= maybe - 1;
        const V3 pp = ld3(planes[k].p), pn = ld3(planes[k].n);
        const double time = dot(pn, pp - r.o) / dot(r.d, pn);
        if (time > 0 && sink.in_front(r, time)) shadowed = true;
      }
    }
  }
  if (shadowed || !n_spheres) return shadowed;
  Ray r;
  r.o = q.o;
  r.d = q.ld;
  const AnyHit sink = make_any_hit(q);
  for (uint32_t k = 0; k < n_spheres && !shadowed; k++) {  // Geometry.hs:81-95
    const V3 ct = ld3(spheres[k].c);
    const double rad = spheres[k].r;
    RH_CNT(prim, 1);
    const double qa = dot(r.d, r.d);
    const double qb = 2.0 * dot(r.d, r.o - ct);
    const double qc = sqrLen(r.o - ct) - rad * rad;
    const double delta = qb * qb - 4.0 * qa * qc;
    if (delta < 0.0) continue;
    const double t0 = 0.5 * ((-qb) - sqrt(delta)) / qa;
    double time;
    if (t0 > 0) time = t0;
    else {
      const double t1 = 0.5 * ((-qb) + sqrt(delta)) / qa;
      if (!(t1 > 0)) continue;
      time = t1;
    }
    shadowed = sink.in_front(r, time);
  }
  return shadowed;
}

// Does the pair's ray have to walk a tree?  Only the part of the ray between its origin and the light can hold an
// occluder (inFrontOfLight).  The origin is within 1.000001e-6 of p in every coordinate, so when p and the light lie
// beyond the same face of a (padded) root box, that part is outside the box.  A mesh is not walked either when the hit
// lies on a triangle that nothing of its own mesh can shadow from this light (lit triangles, light_maps.cpp), or when
// the light's cube map says no triangle of the mesh can lie between p and the light.  What is left gets the float slab
// test of its root box (slot 0 of the super-root).
template <bool COUNT>
__device__ __forceinline__ bool roots_need_walk(const SmemTables& sm, const SceneView& S, bool exact_boxes, bool use_maps,
                                                uint32_t lit, uint32_t n_roots, uint32_t li, const V3& p, const LightPair& q,
                                                Cnt<COUNT>& cnt) {
  bool may = exact_boxes;
  uint32_t skip = 0;
  if ((lit >> li) & 1u) skip = 1u << (lit >> 12);  // (lit is 0 when the flags are switched off)
  for (uint32_t m = 0; m < n_roots; m++) {
    if ((skip >> m) & 1u) continue;
    const double* rb = sm.rootbox[m];
    const uint32_t side = (p.x < rb[0] ? 1u : 0u) | (p.y < rb[1] ? 2u : 0u) | (p.z < rb[2] ? 4u : 0u) |
                          (p.x > rb[3] ? 8u : 0u) | (p.y > rb[4] ? 16u : 0u) | (p.z > rb[5] ? 32u : 0u);
    may |= (side & sm.light_side[li][m]) == 0;
  }
  if (!may) return false;
  Ray r;
  r.o = q.o;
  r.d = q.ld;
  if (exact_boxes || needs_exact_walk(r, S)) return true;
  // the root boxes first (shared memory, ~60 instructions): only a pair whose ray enters a box asks that mesh's cube map
  // (a dependent L2 load)
  const RayF f = make_rayf(r, S);
  const float ffar = __double2float_ru(q.far);
  uint32_t enters = 0;
  for (uint32_t m = 0; m < n_roots; m++) {
    if ((skip >> m) & 1u) continue;
    const uint32_t root = sm.mesh_roots[m];
    const float4* np = root < S.n_smem_nodes ? (const float4*)&sm.nodes[root] : (const float4*)&S.wide32[root];
    const float4 b0 = np[0], b1 = np[1];
    float tm;
    RH_CNT(nodes, 1);
    RH_CNT(box, 1);
    if (slab32(f, b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, tm) && !(tm > ffar)) enters |= 1u << m;
  }
  if (!enters) return false;
  if (use_maps && !q.directional) {
    const uint32_t cell = light_map_cell(p, q.lp, S.light_map_res);
    const float dist_up = __double2float_ru(q.dd);
    if (cell != kEmpty)
      for (uint32_t m = 0; m < S.n_occ_meshes; m++) {
        if (!((enters >> m) & 1u)) continue;
        const uint32_t mi = sm.light_map[li][m];
        if (mi != kEmpty && light_map_clears(S, mi, cell, dist_up)) enters &= ~(1u << m);
      }
  }
  return enters != 0;
}

// The lights of one Diffuse / Plastic hit, everything that needs no tree walk: which lights add nothing (`settled`:
// l.n <= 0 — the Lambert term (Material.hs:31-33) is then exactly 0 whatever the query returns — or a plane / sphere
// occludes), which need a walk (`walk`), and, when none does, the fold itself (accumDiffuse's foldl in light order).
struct LightFold {
  uint32_t walk, settled, culled;
  V3 acc;
};
// FAST: the occluder tables are the staged shared-memory ones (SceneView::shadow_fast), read with LDS.
template <bool COUNT, bool FAST>
__device__ __forceinline__ LightFold fold_lights(const SmemTables& sm, const Ctx& cx, const ChunkParams& P, const V3& p, const V3& n,
                                                const V3& cd, uint32_t lit, Cnt<COUNT>& cnt) {
  const SceneView& S = *cx.S;
  LightFold F;
  F.walk = F.settled = F.culled = 0;
  F.acc = mk(0, 0, 0);  // foldl ... black lts
  const uint32_t n_lights = S.n_lights;
  constexpr bool fast = FAST;
  const OccPlane* planes = fast ? sm.planes : S.occ_planes;
  const OccSphere* spheres = fast ? sm.spheres : S.occ_spheres;
  const rh_light* lights = fast ? sm.lights : cx.lights;
  const uint32_t n_roots = S.n_occ_meshes + (S.sphere_root != kEmpty ? 1u : 0u);
  const bool use_maps = S.light_map_index != nullptr && !P.no_light_maps;
  const bool cd_finite = isfinite(cd.x) && isfinite(cd.y) && isfinite(cd.z);
  // Plane sides, once per hit instead of once per (hit, light).  f(x) = pn.(x - pp) is affine, so a plane can only hold a
  // point of the shadow ray between its origin o and a point light L when f(o) and f(L) differ in sign.  o is within
  // 1e-6 |ld| of the hit p, so |f(o) - f(p)| <= 1e-6 |pn|_1; with |f(p)| and |f(L)| both above the margin
  // |pn|_1 (1e-5 + 1e-12 (|x|_1 + |pp|_1)) — which also covers the roundings of f — and equal in sign, the reference's
  // own quotient n.(p-o)/(d.n) (Geometry.hs:70-79) is either negative (`time > 0` fails) or exceeds the distance to
  // the light by >= 1e-5, far beyond the roundings of inFrontOfLight's comparison (RayHs.hs:84-87) for lights nearer
  // than 1e9: the plane cannot occlude, and its two dot products are skipped.  The hit's own wall (f(p) ~ 0) and
  // everything near a plane still get the reference's test.
  uint32_t hit_front = 0, hit_behind = 0;
  if constexpr (FAST) {
    const double p1 = fabs(p.x) + fabs(p.y) + fabs(p.z);
    for (uint32_t k = 0; k < S.n_occ_planes; k++) {
      const double2* pl = (const double2*)&sm.planes[k];
      const double2 u0 = pl[0], u1 = pl[1], u2 = pl[2];  // (px,py) (pz,nx) (ny,nz)
      const double f = dot(mk(u1.y, u2.x, u2.y), p - mk(u0.x, u0.y, u1.x));
      const double m = sm.plane_margin[k][0] + sm.plane_margin[k][1] * p1;
      hit_front |= (f > m ? 1u : 0u) << k;
      hit_behind |= (f < -m ? 1u : 0u) << k;
    }
  }
  for (uint32_t li = 0; li < n_lights; li++) {
    const rh_light& L = lights[li];
    const LightPair q = make_light_pair(L, p);
    const double ldn = dot(q.ld, n);
    if (ldn <= 0 && cd_finite && light_is_tame(L)) {
      F.culled++;
      F.settled |= 1u << li;
      continue;
    }
    uint32_t skip = 0;
    if constexpr (FAST) {
      if (q.dd < 1e9) skip = (hit_front & sm.light_front[li]) | (hit_behind & sm.light_behind[li]);
    }
    if (primitives_occlude<COUNT>(planes, S.n_occ_planes, spheres, S.n_occ_spheres, q, skip, cnt)) {
      F.settled |= 1u << li;  // Just _ -> black
      continue;
    }
    if (n_roots) {
      // scenes beyond the staged tables (more than kOccMeshes meshes, kFastLights lights, ...) walk whenever there is a tree
      const bool need = fast ? roots_need_walk<COUNT>(sm, S, P.exact_boxes != 0, use_maps, lit, n_roots, li, p, q, cnt) : true;
      if (need) {
        F.walk |= 1u << li;
        continue;
      }
    }
    if (F.walk) continue;  // the shadow kernel redoes this hit's fold: no point in the term
    V3 lc = ld3(L.color);  // lightAt, Light.hs:14-17
    if (!q.directional) {
      const double s = 1.0 + q.dd / L.radius;
      lc = mul(1.0 / (s * s), lc);
    }
    F.acc = F.acc + mul(hs_max(ldn, 0) * kPiInv, cmul(cd, lc));  // diffuse, Material.hs:31-33
  }
  return F;
}

// The fold of a queued hit once its walks are done: `vis` bit l = light l adds nothing.
__device__ __forceinline__ V3 fold_visible(const Ctx& cx, uint32_t n_lights, uint32_t vis, const V3& p, const V3& n, const V3& cd) {
  V3 acc = mk(0, 0, 0);  // foldl ... black lts
  for (uint32_t li = 0; li < n_lights; li++) {
    if ((vis >> li) & 1u) continue;  // Just _ -> black (or l.n <= 0: the term is exactly 0)
    V3 ld, lc;
    light_at(cx.lights[li], p, ld, lc);
    acc = acc + mul(hs_max(dot(ld, n), 0) * kPiInv, cmul(cd, lc));  // diffuse, Material.hs:31-33
  }
  return acc;
}

// Index of a pixel sample's offset pair in the offset array, or false when the mode has no array.
__device__ __forceinline__ bool offset_slot(const ChunkParams& P, uint32_t item, size_t& idx, uint32_t& grow, uint32_t& col, uint32_t& s) {
  const uint32_t lp = item / P.spp;
  s = item - lp * P.spp;
  const uint32_t lrow = lp / P.width;
  col = lp - lrow * P.width;
  grow = global_row(P, P.first_row + lrow);
  if (P.offset_mode == RH_OFFSETS_TILED_F64)
    idx = ((size_t)(grow % P.offset_tile) * P.offset_tile + (col % P.offset_tile)) * P.spp + s;
  else if (P.offset_index == kOffIndexGlobal)
    idx = ((size_t)grow * P.width + col) * P.spp + s;
  else
    idx = item;
  return P.offset_mode == RH_OFFSETS_F64 || P.offset_mode == RH_OFFSETS_F32 || P.offset_mode == RH_OFFSETS_TILED_F64;
}

// One warp's staging tile for the NEXT batch of 32 work items: the four planes of a ray-queue batch (pass >= 1) or the
// f64 offset pairs of 32 pixel samples (pass 0, plane 0 only), filled by bulk async copies.
#if RH_TMA_STAGE >= 2
constexpr int kStagePlanes = 4;  // also the four planes of a ray-queue batch (passes >= 1)
#else
constexpr int kStagePlanes = 1;  // the sample offsets of pass 0 only: 512 bytes per warp
#endif
struct __align__(128) StageTile {
  double2 plane[kStagePlanes][32];
};
struct Staged {
  uint32_t first;   // first work item of the staged batch, kEmpty = nothing staged
  uint32_t parity;  // phase of the warp's mbarrier the next wait uses
};

// Start the copy of the batch of `n` items beginning at `first` (lane 0 only calls this).  Pass 0: only when the
// offsets are per-sample f64 pairs laid out in work-item order (P.offset_linear: chunk-local slices, or the full-frame
// array of an unsharded frame), so that the batch's pairs are one contiguous run.
// `dep`: a value derived from what this lane just read out of the tile; the copy's byte count is made to depend on
// it, so the warp's shared-memory reads of the previous batch have returned before the copy engine may overwrite them.
__device__ __forceinline__ bool stage_start(const ChunkParams& P, bool primary, uint32_t first, uint32_t n, StageTile* tile,
                                            unsigned long long* bar, uint32_t dep) {
  uint32_t zero;
  asm volatile("and.b32 %0, %1, 0;" : "=r"(zero) : "r"(dep));
  n += zero;
  if (primary) {
    if (!P.offset_linear) return false;
    mbar_expect(bar, n * 16u);
    bulk_g2s(tile->plane[0], (const double2*)P.offsets + P.offset_base + first, n * 16u, bar);
    return true;
  }
#if RH_TMA_STAGE >= 2
  const size_t cap = P.q_in.capacity;
  mbar_expect(bar, 4u * n * 16u);
#pragma unroll
  for (int k = 0; k < 4; k++) bulk_g2s(tile->plane[k], P.q_in.plane + (size_t)k * cap + first, n * 16u, bar);
  return true;
#else
  return false;
#endif
}

// Work item -> ray: the camera ray of a pixel sample (pass 0: pixelCoord, Image.hs:31-32, + sample offset,
// RayHs.hs:178-181) or a queued secondary ray with its weight and tags.  False for a padding row of the last band.
// `tile`: the item's batch was staged in shared memory (see stage_start), else it is read from global memory.
// RAYS (rh_trace_rays, P.offset_mode == kOffsetsRays): pass 0 reads caller-built rays instead; false past the chunk's rays.
template <bool RAYS>
__device__ __forceinline__ bool load_item(const ChunkParams& P, const CameraParams& cam, uint32_t item, bool primary,
                                          const StageTile* tile, uint32_t lane, Ray& r, double& w, uint32_t& sample, int& depth,
                                          int& kind, uint32_t& probe_mat) {
  r.o = r.d = mk(0, 0, 1);
  if (RAYS && primary) {
    if (item >= P.ray_items) return false;
    const double2* src = (const double2*)P.offsets + 3 * (P.offset_base + item);
    const double2 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
    r.o = mk(a.x, a.y, b.x);
    r.d = mk(b.y, c.x, c.y);
    return true;
  }
  if (primary) {
    size_t idx;
    uint32_t grow, col, s;
    const bool has_array = offset_slot(P, item, idx, grow, col, s);
    if (grow >= P.height) return false;
    double ox = 0, oy = 0;
    if (P.offset_mode == RH_OFFSETS_SPLITMIX64) {
      // values 2g and 2g+1 of the stream rh_sample_offsets_f64(seed, ...) writes (x before y, RayHs.hs:185-188)
      const unsigned long long g = ((unsigned long long)grow * P.width + col) * P.spp + s;
      ox = splitmix01(P.offset_seed, 2 * g) - 0.5;
      oy = splitmix01(P.offset_seed, 2 * g + 1) - 0.5;
    } else if (has_array) {
      if (P.offset_mode == RH_OFFSETS_F32) {
        const float2 o2 = __ldg((const float2*)P.offsets + idx);
        ox = (double)o2.x;
        oy = (double)o2.y;
      } else {
        const double2 o2 = tile ? tile->plane[0][lane] : __ldg((const double2*)P.offsets + idx);
        ox = o2.x;
        oy = o2.y;
      }
    }
    r = camera_ray(cam, (double)col + ox, (double)grow + oy);
    return true;
  }
  double2 a, b, c, d;
  if (RH_TMA_STAGE >= 2 && tile) {
    a = tile->plane[0][lane], b = tile->plane[1 % kStagePlanes][lane], c = tile->plane[2 % kStagePlanes][lane], d = tile->plane[3 % kStagePlanes][lane];
  } else {
    const size_t cap = P.q_in.capacity;
    a = P.q_in.plane[item], b = P.q_in.plane[cap + item], c = P.q_in.plane[2 * cap + item], d = P.q_in.plane[3 * cap + item];
  }
  r.o = mk(a.x, a.y, b.x);
  r.d = mk(b.y, c.x, c.y);
  w = d.x;
  const uint64_t bits = (uint64_t)__double_as_longlong(d.y);
  sample = (uint32_t)bits;
  depth = (int)((bits >> 32) & 0xff);
  kind = (int)((bits >> 40) & 0xff);
  probe_mat = (uint32_t)((bits >> 48) & 0x7fff);
  return true;
}

// ------------------------------------------------------------------ K1/K2/K4/K5
struct TraceWarpSmem {
#if RH_TMA_STAGE
  StageTile tile;
#endif
  unsigned long long bar;
  SlabWriter out_rays, out_shadow;  // the warp's open slabs of the two output queues
  unsigned long long pad_[12];
};
static_assert(sizeof(TraceWarpSmem) % 128 == 0, "staging tiles stay 128-byte aligned");
constexpr size_t kTraceSmem = sizeof(SmemTables) + (size_t)kShortStack * kTraceBlock * sizeof(uint2) +
                              (kTraceBlock / 32) * sizeof(TraceWarpSmem);
static_assert(sizeof(SmemTables) % 128 == 0 || !RH_TMA_STAGE, "staging tiles need 128-byte alignment after the tables");
static_assert(((size_t)kShortStack * kTraceBlock * sizeof(uint2)) % 128 == 0, "stack columns keep the alignment");
static_assert(kTraceSmem <= 227 * 1024, "trace kernel shared memory");

// RAYS: rh_trace_rays' instantiation (caller-built rays in pass 0, see load_item); the render's is RAYS = false.
template <bool COUNT, bool RAYS>
__global__ void __launch_bounds__(kTraceBlock, kTracePerSm) trace_kernel(const __grid_constant__ SceneView S,
                                                               const __grid_constant__ CameraParams cam,
                                                               const __grid_constant__ ChunkParams P) {
  SmemTables& sm = *reinterpret_cast<SmemTables*>(rh_smem);
  Ctx cx;
  stage_tables(sm, S, cx);
  Stack st = make_stack(rh_smem + sizeof(SmemTables), kTraceBlock, P);
  Cnt<COUNT> cnt;
  cnt.zero();
  const uint32_t lane = threadIdx.x & 31;
  const bool primary = (P.pass == 0);
  ChunkCtl* ctl = P.ctl;
  const uint32_t n_slabs = primary ? (P.n_samples + kSlab - 1) / kSlab : min(ctl->ray_slabs[P.pass], P.q_in.capacity / kSlab);
  // the hit queue is a ring: the slabs of pass `hit_live_pass` (this pass, or the one before it when that pass's hits may
  // still be under classification on the other stream) and later are in use
  const uint32_t hit_live_from = ctl->hit_start[P.hit_live_pass];
  uint32_t n_reflect = 0, n_probe = 0, n_exit = 0, n_shaded = 0;  // (per thread: far below 2^32)
  TraceWarpSmem& wsm = reinterpret_cast<TraceWarpSmem*>(rh_smem + sizeof(SmemTables) + (size_t)kShortStack * kTraceBlock * sizeof(uint2))[threadIdx.x >> 5];
  SlabWriter& out_rays = wsm.out_rays;  // warp-uniform state, kept out of the register file
  SlabWriter& out_shadow = wsm.out_shadow;
  if (lane == 0) {
    out_rays.init();
    out_shadow.init();
  }
#if RH_TMA_STAGE
  if (lane == 0) mbar_init(&wsm.bar);
  Staged staged;
  staged.first = kEmpty;
  staged.parity = 0;
#endif
  __syncwarp();

  const uint32_t n_units = n_slabs * kSlabUnits, total_warps = gridDim.x * (kTraceBlock / 32);
  uint32_t cursor_seen = (blockIdx.x * (kTraceBlock / 32) + (threadIdx.x >> 5)) * kSlabUnits;  // as if every warp ahead had claimed a slab
  for (;;) {
    const uint2 claim = claim_units(&ctl->trace_cursor[P.pass], n_units, total_warps, lane, cursor_seen);
    if (claim.x >= n_units) break;
    const uint32_t claim_end = min(claim.x + claim.y, n_units);
    for (uint32_t u = claim.x; u < claim_end;) {
      uint32_t slab, b, piece_n;
      next_piece(u, claim_end, slab, b, piece_n);
      const uint32_t slab_first = slab * kSlab;
      const uint32_t count = primary ? min(kSlab, P.n_samples - slab_first) : min(__ldg(P.q_in.fill + slab), kSlab);
      if (b >= count) continue;
      const uint32_t item = slab_first + b + lane;
      bool valid = lane < piece_n && b + lane < count;
      Ray r;
      double w = 1;
      uint32_t sample = item, probe_mat = 0;
      int depth = 0, kind = kRayNormal;
      const StageTile* tile = nullptr;
#if RH_TMA_STAGE
      if (staged.first == slab_first + b) {  // this batch was asked for while the previous one was traced
        mbar_wait(&wsm.bar, staged.parity);
        staged.parity ^= 1u;
        tile = &wsm.tile;
      }
#endif
      if (valid) valid = load_item<RAYS>(P, cam, item, primary, tile, lane, r, w, sample, depth, kind, probe_mat);
      else r.o = r.d = mk(0, 0, 1);
#if RH_TMA_STAGE
      // the tile is in registers now: ask for the next batch of this claim (same slab); it lands while this one is traced
      __syncwarp();
      staged.first = kEmpty;
      if (piece_n == 32 && b + 32 < count && u < claim_end && u % kSlabUnits != 0) {
        uint32_t ok = 0;
        const uint32_t dep = (uint32_t)(__double2loint(r.o.x) ^ __double2loint(r.d.x) ^ __double2loint(w));
        if (lane == 0) ok = stage_start(P, primary, slab_first + b + 32, min(32u, count - b - 32), &wsm.tile, &wsm.bar, dep) ? 1u : 0u;
        if (__shfl_sync(kFull, ok, 0)) staged.first = slab_first + b + 32;
      }
#endif

      Closest best;
      best.obj = -1;
      if (valid) {
        const bool exact = P.exact_boxes || needs_exact_walk(r, S);
        unsigned long long nodes_before = 0;
        if constexpr (COUNT) nodes_before = cnt.nodes;
        closest_hit<COUNT>(cx, r, exact, best, st, cnt);
        if constexpr (COUNT) {
          if (exact) atomicAdd(&P.counters->exact_closest, 1ull);
          atomicMax(&P.counters->max_closest_nodes, cnt.nodes - nodes_before);
        }
      }
      if (primary && valid && P.hit_ids) {
        int tri = -1;
        if (best.obj >= 0 && cx.objects[best.obj].kind == RH_OBJ_MESH) tri = (int)S.tris[best.slot].tri_id;
        P.hit_ids[(size_t)P.first_row * P.width * P.spp + item] = make_int2(best.obj, tri);
      }
      // RayHs.hs:149-154: a miss contributes black — nothing to do.
      const bool hit = valid && best.obj >= 0;

      // ---- shade (irradiance, RayHs.hs:107-147), in stages the whole warp walks through together so that every queue
      // push is one ballot; the recursion is unrolled into weighted child rays: every combine in the reference is
      // `mul scalar colour` + add, so a child carries the scalar product `w`.
      V3 p = mk(0, 0, 0), n = mk(0, 0, 1);
      double tu = 0, tv = 0;
      int mkind = -1, okind = -1;
      uint32_t mat_index = 0;
      if (hit) {
        // rebuild the Hit (Geometry.hs:39) of the winning primitive
        const DObject& ob = cx.objects[best.obj];
        mat_index = (uint32_t)ob.material;
        const rh_material& mat = cx.materials[mat_index];
        mkind = mat.kind;
        okind = ob.kind;
        const bool need_uv = (kind == kRayNormal) && (mkind == RH_MAT_SHOWUV ||
                                                      ((mkind == RH_MAT_DIFFUSE || mkind == RH_MAT_PLASTIC) && mat.cmap_kind != RH_CMAP_FLAT));
        // (the same rebuild as rebuild_hit, kept inline: calling it costs this kernel 8 bytes of stack frame and 32 bytes
        // of spill stores, DESIGN.md "Ray queries")
        p = rayAt(r, best.t);
        if (okind == RH_OBJ_MESH) {
          const double* sh = (const double*)(S.shade + best.slot);
          RH_CNT(shade, 1);
          const double wu = best.u, wv = best.v, ww = 1 - best.u - best.v;
          // barycentricInterp u n1 v n2 (1-u-v) n0 = mul a p + mul b q + mul c r   (Mesh.hs:57, 81)
          n = mul(wu, ld3(sh + 3)) + mul(wv, ld3(sh + 6)) + mul(ww, ld3(sh));
          if (need_uv) {
            tu = wu * sh[11] + wv * sh[13] + ww * sh[9];
            tv = wu * sh[12] + wv * sh[14] + ww * sh[10];
          }
        } else if (okind == RH_OBJ_PLANE) {  // Geometry.hs:70-79
          n = ld3(ob.b);
          if (need_uv) {
            const V3 tg = ld3(ob.c);
            const V3 bt = cross(tg, n);
            const V3 rel = p - ld3(ob.a);
            tu = dot(tg, rel);
            tv = dot(bt, rel);
          }
        } else {  // Geometry.hs:83-96
          n = normalize(p - ld3(ob.a));
          if (need_uv) {
            tu = kPiInv * atan(n.z / n.x);
            tv = kPiInv * acos(n.y);
          }
        }
      }
      const bool probe = hit && kind == kRayProbe;
      const bool surface = hit && kind != kRayProbe;

      // child ray A: the specular reflection (RayHs.hs:99-104) of Plastic / Mirror / Transparent, or — for the interior
      // probe of a Transparent hit (RayHs.hs:140-143) — the ray that leaves through the far interface
      {
        bool has = false, is_exit = false;
        Ray ra;
        ra.o = ra.d = mk(0, 0, 1);
        double wa = 0;
        uint64_t bits = 0;
        if (probe) {
          const double ior = cx.materials[probe_mat].ior;
          V3 outDir;
          if (refract(r.d, neg(n), ior, 1.0, outDir)) {
            has = is_exit = true;
            ra = rayEps(p, outDir);
            wa = w;
            bits = pack_bits(sample, depth, kRayNormal, 0);
          }
        } else if (surface && (mkind == RH_MAT_PLASTIC || mkind == RH_MAT_MIRROR || mkind == RH_MAT_TRANSPARENT) && depth < P.max_depth) {
          const double ior = cx.materials[mat_index].ior;
          const V3 rd = reflect(r.d, n);
          const double f = fresnel(ior, dot(n, neg(r.d)));
          has = true;
          ra = rayEps(p, rd);
          wa = w * (f * dot(rd, n));
          bits = pack_bits(sample, depth + 1, kRayNormal, 0);
        }
        if (has) {
          if (is_exit) n_exit++;
          else n_reflect++;
        }
        push_ray(has, ra, wa, bits, P.q_out, out_rays, &ctl->ray_slabs[P.pass + 1], &ctl->overflow, lane);
      }
      // child ray B: the interior probe of a Transparent hit (RayHs.hs:136-139)
      if (__any_sync(kFull, surface && mkind == RH_MAT_TRANSPARENT)) {
        bool has = false;
        Ray rb;
        rb.o = rb.d = mk(0, 0, 1);
        double wb = 0;
        uint64_t bits = 0;
        if (surface && mkind == RH_MAT_TRANSPARENT && depth != P.max_depth) {
          const double ior = cx.materials[mat_index].ior;
          V3 refDir;
          if (refract(r.d, n, 1.0, ior, refDir)) {
            has = true;
            rb = rayEps(p, refDir);
            wb = w * (1 - r0f(ior, 1.0));
            bits = pack_bits(sample, depth + 1, kRayProbe, mat_index);
            n_probe++;
          }
        }
        push_ray(has, rb, wb, bits, P.q_out, out_rays, &ctl->ray_slabs[P.pass + 1], &ctl->overflow, lane);
      }
      // Local terms that need no light (Emmit, ShowNormal, ShowUV: RayHs.hs:121-128) and Diffuse / Plastic hits, whose
      // ambient + accumDiffuse terms (RayHs.hs:111-119) classify_kernel folds: both go to the hit queue.  Every add to a
      // sample's accumulator is made by the shadow kernels, pass after pass, so the order of a sample's terms does not
      // depend on how far the next pass's trace kernel — which runs on its own stream — has got.
      {
        const bool lit_surface = surface && (mkind == RH_MAT_DIFFUSE || mkind == RH_MAT_PLASTIC);
        const bool direct = surface && (mkind == RH_MAT_EMMIT || mkind == RH_MAT_SHOWNORMAL || mkind == RH_MAT_SHOWUV);
        ShadowTask task;
        if (lit_surface) {
          n_shaded++;
          task.p = p;
          task.n = n;
          task.cd = color_at<COUNT>(S, cx.materials[mat_index], tu, tv, cnt);
          task.w = w;
          task.sample = sample | (mkind == RH_MAT_DIFFUSE ? 0x80000000u : 0u);
          // lit-triangle flags of the hit triangle (light_maps.cpp) travel in the `walk` word of the hit queue
          task.walk = (okind == RH_OBJ_MESH && S.lit_flags && !P.no_light_maps) ? (uint32_t)__ldg(S.lit_flags + best.slot) : 0u;
          task.settled = 0;
        } else if (direct) {
          task.p = p;
          task.n = n;
          task.cd = mkind == RH_MAT_EMMIT ? ld3(cx.materials[mat_index].color1) : (mkind == RH_MAT_SHOWNORMAL ? n : mk(tu, tv, 0));
          task.w = w;
          task.sample = sample;
          task.walk = kHitDirect;
          task.settled = 0;
        }
        push_shadow(lit_surface || direct, task, P.q_hits, out_shadow, &ctl->hit_slab_next, &ctl->overflow, lane, hit_live_from);
      }
    }
  }
  slab_close(out_rays, lane, P.q_out.fill, &ctl->ray_items[P.pass + 1]);
  slab_close(out_shadow, lane, P.q_hits.fill, &ctl->hit_items[P.pass]);

  // ray-class statistics (one ray per closestIntersection call, SURVEY 8d)
  const uint32_t per_thread[4] = {n_reflect, n_probe, n_exit, n_shaded};
  unsigned long long* const totals[4] = {&P.counters->rays_reflect, &P.counters->rays_probe, &P.counters->rays_exit,
                                         &P.counters->shaded_hits};
#pragma unroll
  for (int k = 0; k < 4; k++) {
    unsigned long long v = per_thread[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    if (lane == 0 && v) atomicAdd(totals[k], v);
  }
  flush_counters<COUNT>(cnt, P.counters, 0);
}

// ------------------------------------------------------------------ K3a: the light fold of every shaded hit
// One thread per Diffuse / Plastic hit of the pass: all its lights, everything that needs no tree (Lambert cull, planes,
// linear spheres, root boxes, lit triangles, cube maps).  A hit whose lights are all settled is folded and accumulated
// on the spot (accumDiffuse, RayHs.hs:89-97); a hit with a light whose shadow ray has to walk a tree goes to the walk
// queue with the two light masks.  Straight-line code, no stack, small enough for the instruction cache.
#ifndef RH_CLASSIFY_BLOCK
#define RH_CLASSIFY_BLOCK 256
#define RH_CLASSIFY_MINB 3  // 3 blocks of 256 per SM at 80 registers (measured on the bench frame: 23.6 ms of shadow work against 25.5 with 2 blocks at up to 128 registers and 26.8 with 4 at 64)
#endif
constexpr int kClassifyBlock = RH_CLASSIFY_BLOCK;
struct ClassifyWarpSmem {
  SlabWriter out;
  uint32_t pad_;
};
constexpr size_t kClassifySmem = sizeof(SmemTables) + (kClassifyBlock / 32) * sizeof(ClassifyWarpSmem);

template <bool COUNT, bool FAST>
__global__ void __launch_bounds__(kClassifyBlock, RH_CLASSIFY_MINB) classify_kernel(const __grid_constant__ SceneView S,
                                                                     const __grid_constant__ ChunkParams P) {
  SmemTables& sm = *reinterpret_cast<SmemTables*>(rh_smem);
  Ctx cx;
  stage_tables(sm, S, cx);
  const uint32_t lane = threadIdx.x & 31;
  SlabWriter& out = reinterpret_cast<ClassifyWarpSmem*>(rh_smem + sizeof(SmemTables))[threadIdx.x >> 5].out;
  if (lane == 0) out.init();
  __syncwarp();
  Cnt<COUNT> cnt;
  cnt.zero();
  ChunkCtl* ctl = P.ctl;
  const uint32_t ring_slabs = P.q_hits.capacity / kSlab, slab0 = ctl->hit_start[P.pass];  // this pass's slabs of the hit queue (a ring)
  const uint32_t n_slabs = min(ctl->hit_start[P.pass + 1] - slab0, ring_slabs);
  const size_t cap = P.q_hits.capacity;
  const double2* qp = P.q_hits.plane;
  uint32_t n_culled = 0, n_walk_pairs = 0;
  const uint32_t n_units = n_slabs * kSlabUnits, total_warps = gridDim.x * (kClassifyBlock / 32);
  uint32_t cursor_seen = (blockIdx.x * (kClassifyBlock / 32) + (threadIdx.x >> 5)) * kSlabUnits;
  for (;;) {
    const uint2 claim = claim_units(&ctl->hit_cursor[P.pass], n_units, total_warps, lane, cursor_seen);
    if (claim.x >= n_units) break;
    const uint32_t claim_end = min(claim.x + claim.y, n_units);
    for (uint32_t u = claim.x; u < claim_end;) {
      uint32_t slab, b, piece_n;
      next_piece(u, claim_end, slab, b, piece_n);
      slab = (slab + slab0) % ring_slabs;
      const uint32_t n_here = min(__ldg(P.q_hits.fill + slab), kSlab);
      if (b >= n_here) continue;
      const uint32_t item = slab * kSlab + b + lane;
      const bool valid = lane < piece_n && b + lane < n_here;
      ShadowTask task;
      bool queue = false;
      if (valid) {
        const double2 a = qp[item], bq = qp[cap + item], c = qp[2 * cap + item], d = qp[3 * cap + item], e = qp[4 * cap + item];
        task.sample = P.q_hits.sample[item];
        const uint32_t lit = P.q_hits.walk[item];
        task.p = mk(a.x, a.y, bq.x);
        task.n = mk(bq.y, c.x, c.y);
        task.cd = mk(d.x, d.y, e.x);
        task.w = e.y;
        LightFold F;
        if (lit & kHitDirect) {
          F.walk = F.settled = F.culled = 0;
          F.acc = task.cd;
        } else {
          F = fold_lights<COUNT, FAST>(sm, cx, P, task.p, task.n, task.cd, lit, cnt);
        }
        n_culled += F.culled;
        if (F.walk) {
          queue = true;
          n_walk_pairs += __popc(F.walk);
          task.walk = F.walk;
          task.settled = F.settled;
        } else {
          const V3 total = (task.sample & 0x80000000u) ? mul(0.2, task.cd) + F.acc : F.acc;  // Diffuse adds the ambient term, RayHs.hs:111-114
          accumulate(P, task.sample & 0x7fffffffu, task.w, total);
        }
      }
      push_shadow(queue, task, P.q_shadow, out, &ctl->shadow_slabs[P.pass], &ctl->overflow, lane);
    }
  }
  slab_close(out, lane, P.q_shadow.fill, &ctl->shadow_items[P.pass]);
  unsigned long long vc = n_culled, vw = n_walk_pairs;
  for (int o = 16; o > 0; o >>= 1) {
    vc += __shfl_xor_sync(kFull, vc, o);
    vw += __shfl_xor_sync(kFull, vw, o);
  }
  if (lane == 0) {
    if (vc) atomicAdd(&P.counters->shadow_culled, vc);
    if (vw) atomicAdd(&P.counters->shadow_walk_pairs, vw);
  }
  flush_counters<COUNT>(cnt, P.counters, 1);
}

// ------------------------------------------------------------------ K3: the tree walks of the queued hits
// The (hit, light) pair's any-hit walk over the occluding trees (RayHs.hs:74-87 for the mesh objects and the sphere
// tree; planes and linear spheres were settled by the trace kernel).  True = occluded.
template <bool COUNT>
__device__ __forceinline__ bool walk_pair(const Ctx& cx, const ChunkParams& P, const uint32_t* mesh_roots, uint32_t n_meshes,
                                          const rh_light& L, const V3& p, Stack& st, Cnt<COUNT>& cnt) {
  const SceneView& S = *cx.S;
  const LightPair q = make_light_pair(L, p);
  Ray r;
  r.o = q.o;
  r.d = q.ld;
  AnyHit sink = make_any_hit(q);
  const bool exact = P.exact_boxes || needs_exact_walk(r, S);
  const RayF f = make_rayf(r, S);
  bool hit = false;
  unsigned long long nodes_before = 0;
  if constexpr (COUNT) {
    nodes_before = cnt.nodes;
    if (exact) atomicAdd(&P.counters->exact_walks, 1ull);
  }
  for (uint32_t m = 0; m < n_meshes && !hit; m++) {
    double bound = q.far;
    hit = exact ? traverse_exact<COUNT>(cx, mesh_roots[m], r, bound, sink, st, cnt)
                : traverse<COUNT>(cx, mesh_roots[m], r, f, bound, sink, st, cnt);
  }
  if (!hit && S.sphere_root != kEmpty) {
    double bound = q.far;
    hit = exact ? traverse_exact<COUNT, AnyHit, true>(cx, S.sphere_root, r, bound, sink, st, cnt, true)
                : traverse<COUNT, AnyHit, true>(cx, S.sphere_root, r, f, bound, sink, st, cnt, true);
  }
  if constexpr (COUNT) {
    const unsigned long long nv = cnt.nodes - nodes_before;
    atomicMax(&P.counters->max_walk_nodes, nv);
    const int bin = min(19, 63 - __clzll((long long)(nv + 1))), row = min(P.pass, 3);
    atomicAdd(&P.counters->walk_hist[row][bin], 1ull);
    atomicAdd(&P.counters->walk_hist_nodes[row][bin], nv);
  }
  return hit;
}

// Pooled form, for coherent rays.  Each warp takes one slab of queued hits (<= 128, 4 per lane) and, light by light
// (rays towards one light from neighbouring samples stay coherent),
//   phase 1  appends the hits whose mask asks for a walk towards that light to a warp-local pool in shared memory
//            (ballot + prefix-popcount compaction);
//   phase 2  walks the pool in full rounds of 32, every lane on a ray that needs it; what is left over (< 32) stays
//            pooled and joins the next light's rays.  An occluded pair sets its bit in the hit's visibility word
//            (shared-memory atomicOr);
//   phase 3  every lane folds the lights of its own hits in order (accumDiffuse's foldl, RayHs.hs:89-97) with those
//            bits and adds w * (ambient + sum) to the sample.
constexpr int kShadowT = kSlab / 32;
struct ShadowWarpSmem {
  uint32_t vis[kSlab];        // bit li: light li adds nothing for this hit
  uint16_t pool[kSlab + 32];  // hit-in-slab | light << 8
};
static_assert(sizeof(ShadowWarpSmem) % 16 == 0, "the stack columns follow the per-warp regions");
static_assert(kSlab <= 256 && kMaskLights <= 256, "pool entries keep the hit index and the light in 8 bits each");
constexpr size_t kShadowSmem = sizeof(WalkTables) + (kShadowBlock / 32) * sizeof(ShadowWarpSmem) +
                               (size_t)kShortStack * kShadowBlock * sizeof(uint2);
static_assert(kShadowSmem <= 227 * 1024, "pooled shadow kernel shared memory");

template <bool COUNT>
__global__ void __launch_bounds__(kShadowBlock, kShadowPerSm) shadow_pooled_kernel(const __grid_constant__ SceneView S,
                                                                        const __grid_constant__ ChunkParams P) {
  WalkTables& sm = *reinterpret_cast<WalkTables*>(rh_smem);
  Ctx cx;
  stage_walk_tables(sm, S, cx);
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  ShadowWarpSmem& ws = reinterpret_cast<ShadowWarpSmem*>(rh_smem + sizeof(WalkTables))[warp];
  Stack st = make_stack(rh_smem + sizeof(WalkTables) + (kShadowBlock / 32) * sizeof(ShadowWarpSmem), kShadowBlock, P);
  const uint32_t n_lights = S.n_lights, n_meshes = S.n_occ_meshes;
  const uint32_t* mesh_roots = n_meshes <= (uint32_t)kOccMeshes ? sm.mesh_roots : S.occ_meshes;
  Cnt<COUNT> cnt;
  cnt.zero();
  ChunkCtl* ctl = P.ctl;
  const uint32_t n_slabs = min(ctl->shadow_slabs[P.pass], P.q_shadow.capacity / kSlab);
  const size_t cap = P.q_shadow.capacity;
  const double2* qp = P.q_shadow.plane;

  const uint32_t n_units = n_slabs * kSlabUnits, total_warps = gridDim.x * (kShadowBlock / 32);
  uint32_t seg_next = 0, seg_end = 0;  // the warp's claimed units not yet processed
  uint32_t cursor_seen = (blockIdx.x * (kShadowBlock / 32) + warp) * kSlabUnits;
#ifdef RH_WARP_TIMES
  unsigned long long dbg_t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0));
  uint32_t dbg_batches = 0, dbg_rounds = 0, dbg_walk_ns = 0, dbg_max_nodes = 0, dbg_max_tris = 0, dbg_pairs = 0;
#endif
  for (;;) {
    // a whole slab per claim while plenty of work is left (full pools), smaller pieces near the end of the queue
    if (seg_next == seg_end) {
      const uint2 claim = claim_units(&ctl->shadow_cursor[P.pass], n_units, total_warps, lane, cursor_seen);
      if (claim.x >= n_units) break;
      seg_next = claim.x;
      seg_end = min(claim.x + claim.y, n_units);
    }
    // the part of the claim that lies in one slab
    const uint32_t slab = seg_next / kSlabUnits, u_first = seg_next % kSlabUnits;
    const uint32_t u_count = min(seg_end - seg_next, kSlabUnits - u_first);
    seg_next += u_count;
    const uint32_t fill = min(__ldg(P.q_shadow.fill + slab), kSlab);
    if (u_first * kUnit >= fill) continue;
    const uint32_t base = slab * kSlab + u_first * kUnit, n_here = min(fill - u_first * kUnit, u_count * kUnit);
#ifdef RH_WARP_TIMES
    dbg_batches += (n_here + 31) / 32;
#endif
    uint32_t wm[kShadowT];
#pragma unroll
    for (int t = 0; t < kShadowT; t++) {
      const uint32_t j = t * 32 + lane;
      wm[t] = 0;
      if (j < n_here) {
        wm[t] = P.q_shadow.walk[base + j];
        ws.vis[j] = P.q_shadow.settled[base + j];
      }
    }
    __syncwarp();
    uint32_t pool_n = 0;
    for (uint32_t li = 0; li < n_lights; li++) {
      // ---- phase 1
#pragma unroll
      for (int t = 0; t < kShadowT; t++) {
        const bool need = (wm[t] >> li) & 1u;
        const unsigned m = __ballot_sync(kFull, need);
        if (need) ws.pool[pool_n + __popc(m & ((1u << lane) - 1))] = (uint16_t)((t * 32 + lane) | (li << 8));
        pool_n += __popc(m);
      }
      __syncwarp();
      // ---- phase 2: tree walks in full rounds; the last light also drains the remainder
      const bool last = (li + 1 == n_lights);
      const uint32_t n_full = last ? pool_n : (pool_n & ~31u);
#ifdef RH_WARP_TIMES
      dbg_rounds += (n_full + 31) / 32;
      dbg_pairs += n_full;
      unsigned long long dbg_w0;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_w0));
#endif
      for (uint32_t i = lane; i < n_full; i += 32) {
        const uint32_t e = ws.pool[i], j = e & 0xff, lw = e >> 8;
        const double2 a = qp[base + j], b = qp[cap + base + j];
#ifdef RH_WARP_TIMES
        unsigned dn0 = 0, dt0 = 0;
        if constexpr (!COUNT) { dn0 = cnt.dn; dt0 = cnt.dt; }
#endif
        if (walk_pair<COUNT>(cx, P, mesh_roots, n_meshes, cx.lights[lw], mk(a.x, a.y, b.x), st, cnt)) atomicOr(&ws.vis[j], 1u << lw);
#ifdef RH_WARP_TIMES
        if constexpr (!COUNT) {
          unsigned dn1 = cnt.dn - dn0, dt1 = cnt.dt - dt0;
          const unsigned act = __activemask();
          for (int o = 16; o; o >>= 1) {
            dn1 = max(dn1, __shfl_xor_sync(act, dn1, o));
            dt1 = max(dt1, __shfl_xor_sync(act, dt1, o));
          }
          dbg_max_nodes += dn1;
          dbg_max_tris += dt1;
        }
#endif
      }
#ifdef RH_WARP_TIMES
      __syncwarp();
      {
        unsigned long long dbg_w1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_w1));
        dbg_walk_ns += (uint32_t)(dbg_w1 - dbg_w0);
      }
#endif
      __syncwarp();
      const uint32_t rem = pool_n - n_full;
      uint16_t keep = 0;
      if (lane < rem) keep = ws.pool[n_full + lane];
      __syncwarp();
      if (lane < rem) ws.pool[lane] = keep;
      pool_n = rem;
      __syncwarp();
    }
    // ---- phase 3: accumDiffuse's fold over the lights, in order
#pragma unroll 1
    for (int t = 0; t < kShadowT; t++) {
      const uint32_t j = t * 32 + lane;
      if (j >= n_here) continue;
      const uint32_t item = base + j;
      const double2 a = qp[item], b = qp[cap + item], c = qp[2 * cap + item], d = qp[3 * cap + item], e = qp[4 * cap + item];
      const uint32_t sbits = P.q_shadow.sample[item];
      const V3 p = mk(a.x, a.y, b.x), n = mk(b.y, c.x, c.y), cd = mk(d.x, d.y, e.x);
      const V3 acc = fold_visible(cx, n_lights, ws.vis[j], p, n, cd);
      const V3 total = (sbits & 0x80000000u) ? mul(0.2, cd) + acc : acc;  // Diffuse adds the ambient term, RayHs.hs:111-114
      accumulate(P, sbits & 0x7fffffffu, e.y, total);
    }
    __syncwarp();
  }
#ifdef RH_WARP_TIMES
  {
    const uint32_t wi = blockIdx.x * (kShadowBlock / 32) + warp, row = min(P.pass, 3);
    if (lane == 0 && wi < 4096) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      P.counters->warp_begin[row][wi] = (unsigned int)dbg_t0;
      P.counters->warp_end[row][wi] = (unsigned int)t1 | 1u;
      P.counters->warp_batches[row][wi] = dbg_batches;
      P.counters->warp_rounds[row][wi] = dbg_rounds;
      P.counters->warp_walk_ns[row][wi] = dbg_walk_ns;
      P.counters->warp_max_nodes[row][wi] = dbg_max_nodes;
      P.counters->warp_max_tris[row][wi] = dbg_max_tris;
      P.counters->warp_pairs[row][wi] = dbg_pairs;
    }
  }
#endif
  flush_counters<COUNT>(cnt, P.counters, 1);
}

// Per-lane refill form, for incoherent rays (triangle soups: unoccluded rays walk hundreds of nodes while occluded ones
// stop after a few, and a pooled round lasts as long as its longest walk).  One queued hit per lane; a lane whose ray
// has ended starts the walk towards its hit's next light, or — when the hit has none left — folds the hit and takes
// the next one of the warp's slab, while its neighbours keep walking.  The loop is warp-uniform: votes decide between
// the refill, inner-node and leaf steps, so the lanes reconverge at every step by construction.
constexpr uint32_t kRefillMin = RH_REFILL_MIN;  // lanes without a ray in flight that trigger a refill step
constexpr int kWalkColumns = 12;                // per-thread doubles in shared memory: ray origin, direction, far, dl2, hit point, (spare)
constexpr size_t kWalkSmem = sizeof(WalkTables) + (size_t)kWalkColumns * kWalkBlock * sizeof(double) +
                             (size_t)kShortStack * kWalkBlock * sizeof(uint2);
static_assert(kWalkSmem <= 227 * 1024, "refill shadow kernel shared memory");

template <bool COUNT>
__global__ void __launch_bounds__(kWalkBlock, 1) shadow_refill_kernel(const __grid_constant__ SceneView S,
                                                                      const __grid_constant__ ChunkParams P) {
  WalkTables& sm = *reinterpret_cast<WalkTables*>(rh_smem);
  Ctx cx;
  stage_walk_tables(sm, S, cx);
  const uint32_t n_lights = S.n_lights, n_meshes = S.n_occ_meshes;
  const uint32_t n_roots = n_meshes + (S.sphere_root != kEmpty ? 1u : 0u);
  const uint32_t* mesh_roots = n_meshes <= (uint32_t)kOccMeshes ? sm.mesh_roots : S.occ_meshes;
  const rh_tri* tris = S.tris;
  // Lane state: what every inner-node step needs stays in registers (the float ray, the node reference, the stack
  // pointer); what only a leaf or the fold needs lives in a per-thread column of shared memory.
  double* lane_mem = reinterpret_cast<double*>(rh_smem + sizeof(WalkTables)) + threadIdx.x;
  auto lane_slot = [&](int k) -> double& { return lane_mem[k * kWalkBlock]; };  // 0-2 o, 3-5 d, 6 far, 7 dl2, 8-10 hit point
  Stack st = make_stack(rh_smem + sizeof(WalkTables) + (size_t)kWalkColumns * kWalkBlock * sizeof(double), kWalkBlock, P);
  Cnt<COUNT> cnt;
  cnt.zero();
  ChunkCtl* ctl = P.ctl;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t n_slabs = min(ctl->shadow_slabs[P.pass], P.q_shadow.capacity / kSlab);
  const size_t cap = P.q_shadow.capacity;
  const double2* qp = P.q_shadow.plane;

  uint32_t pos = 0, end = 0;  // this warp's claimed range of queued hits
  bool exhausted = false;
  bool walking = false, has_task = false, directional = false;
  uint32_t item = 0, rest = 0, vis = 0, cur = 0;  // the lane's hit, its lights still to walk, lights that add nothing, light in flight
  RayF f;
  f.ix = f.iy = f.iz = f.pix = f.piy = f.piz = f.mix = f.miy = f.miz = 0.f;
  float ffar = 0;
  uint32_t ref = 0;
  int sp = 0;

  for (;;) {
    // ---- refill: lanes without a ray in flight fold a finished hit, take a new one, start the next light
    const unsigned idle = __ballot_sync(kFull, !walking);
    if (__popc(idle) >= kRefillMin) {
      if (!walking && has_task && rest == 0) {  // all lights known: accumDiffuse's fold, in order
        const double2 bq = qp[cap + item], c = qp[2 * cap + item], d = qp[3 * cap + item], e = qp[4 * cap + item];
        const uint32_t sbits = P.q_shadow.sample[item];
        const V3 p = mk(lane_slot(8), lane_slot(9), lane_slot(10)), n = mk(bq.y, c.x, c.y), cd = mk(d.x, d.y, e.x);
        const V3 acc = fold_visible(cx, n_lights, vis, p, n, cd);
        const V3 total = (sbits & 0x80000000u) ? mul(0.2, cd) + acc : acc;  // Diffuse adds the ambient term, RayHs.hs:111-114
        accumulate(P, sbits & 0x7fffffffu, e.y, total);
        has_task = false;
      }
      const unsigned empty = __ballot_sync(kFull, !has_task);
      if (empty) {
        if (pos == end && !exhausted) {
          uint32_t s = 0;
          if (lane == 0) s = atomicAdd(&ctl->shadow_cursor[P.pass], 1u);
          s = __shfl_sync(kFull, s, 0);
          if (s >= n_slabs) exhausted = true;
          else {
            pos = s * kSlab;
            end = pos + min(__ldg(P.q_shadow.fill + s), kSlab);
          }
        }
        if (pos < end) {
          const uint32_t take = min((uint32_t)__popc(empty), end - pos);
          const uint32_t rank = __popc(empty & ((1u << lane) - 1));
          if (!has_task && rank < take) {
            item = pos + rank;
            rest = P.q_shadow.walk[item];
            vis = P.q_shadow.settled[item];
            const double2 a = qp[item], b = qp[cap + item];
            lane_slot(8) = a.x; lane_slot(9) = a.y; lane_slot(10) = b.x;
            has_task = true;
          }
          pos += take;
        } else if (exhausted && empty == kFull) {
          break;  // nothing in flight, nothing left to claim
        }
      }
      if (!walking && has_task && rest != 0) {  // the walk towards the hit's next light
        cur = __ffs(rest) - 1;
        rest &= rest - 1;
        const LightPair q = make_light_pair(cx.lights[cur], mk(lane_slot(8), lane_slot(9), lane_slot(10)));
        Ray r;
        r.o = q.o;
        r.d = q.ld;
        AnyHit sink = make_any_hit(q);
        if (P.exact_boxes || needs_exact_walk(r, S)) {
          // rare (SURVEY App. A-N1, far origins): the reference's own double boxes, run to the end right here
          if constexpr (COUNT) atomicAdd(&P.counters->exact_walks, 1ull);
          bool hit = false;
          for (uint32_t m = 0; m < n_roots && !hit; m++) {
            double bound = q.far;
            if (m < n_meshes) hit = traverse_exact<COUNT>(cx, mesh_roots[m], r, bound, sink, st, cnt);
            else hit = traverse_exact<COUNT, AnyHit, true>(cx, S.sphere_root, r, bound, sink, st, cnt, true);
          }
          if (hit) vis |= 1u << cur;
        } else if (n_roots) {
          lane_slot(0) = r.o.x; lane_slot(1) = r.o.y; lane_slot(2) = r.o.z;
          lane_slot(3) = r.d.x; lane_slot(4) = r.d.y; lane_slot(5) = r.d.z;
          lane_slot(6) = q.far;
          lane_slot(7) = sink.dl2;
          directional = q.directional;
          f = make_rayf(r, S);
          ffar = __double2float_ru(q.far);
          sp = 0;
          for (uint32_t m = n_roots; m-- > 1;)  // the other roots wait on the stack (entry distance 0), first mesh on top
            st.push(sp, m < n_meshes ? mesh_roots[m] : S.sphere_root, 0.f);
          ref = n_meshes ? mesh_roots[0] : S.sphere_root;
          walking = true;
        }
      }
    }
    // ---- inner nodes: step until every ray in flight holds a leaf (KDTree.hs:96-107 with the conservative float
    // boxes); RH_WALK_UNROLL steps per vote
    auto step = [&]() {
      if (!node_step<COUNT>(cx, ref, f, ffar, st, sp, cnt)) {
        if (sp == 0) walking = false;  // nothing in front of the light
        else ref = st.pop(sp).x;
      }
    };
    for (;;) {
      bool inner = walking && !(ref & kLeafBit);
      if (!__any_sync(kFull, inner)) break;
      if (inner) step();
#if RH_WALK_UNROLL > 1
      inner = walking && !(ref & kLeafBit);
      if (inner) step();
#endif
    }
    // ---- leaves: every ray in flight holds one (Mesh.hs:59-82 / Geometry.hs:81-95 per candidate)
    if (walking) {
      Ray r;
      r.o = mk(lane_slot(0), lane_slot(1), lane_slot(2));
      r.d = mk(lane_slot(3), lane_slot(4), lane_slot(5));
      double bound = lane_slot(6);
      AnyHit sink;
      sink.directional = directional;
      sink.lpos = mk(0, 0, 0);
      sink.dl2 = lane_slot(7);
      const uint32_t first = ref & kLeafFirstMask, count = ((ref >> kLeafCountShift) & (kLeafMaxCount - 1)) + 1;
      bool hit;
      if (ref & kSphereLeafBit) hit = test_sphere_leaf<COUNT>(cx, first, count, r, sink, bound, true, cnt);
      else hit = test_leaf<COUNT>(tris, first, count, r, sink, bound, cnt);
      if (hit) {
        vis |= 1u << cur;  // shadowIntersection = Just _
        walking = false;
      } else if (sp == 0) {
        walking = false;
      } else {
        ref = st.pop(sp).x;
      }
    }
  }
  flush_counters<COUNT>(cnt, P.counters, 1);
}

// Simple form, for scenes with more than 32 lights (the masks of a queued hit hold 32): every Diffuse / Plastic hit is
// queued unclassified; one hit per lane, lights in sequence, each query over the whole object list run to completion.
constexpr size_t kSimpleSmem = sizeof(SmemTables) + (size_t)kShortStack * kShadowBlock * sizeof(uint2);
template <bool COUNT>
__global__ void __launch_bounds__(kShadowBlock, 1) shadow_simple_kernel(const __grid_constant__ SceneView S,
                                                                        const __grid_constant__ ChunkParams P) {
  SmemTables& sm = *reinterpret_cast<SmemTables*>(rh_smem);
  Ctx cx;
  stage_tables(sm, S, cx);
  Stack st = make_stack(rh_smem + sizeof(SmemTables), kShadowBlock, P);
  Cnt<COUNT> cnt;
  cnt.zero();
  const uint32_t lane = threadIdx.x & 31;
  ChunkCtl* ctl = P.ctl;
  const uint32_t ring_slabs = P.q_hits.capacity / kSlab, slab0 = ctl->hit_start[P.pass];  // this pass's slabs of the hit queue (a ring)
  const uint32_t n_slabs = min(ctl->hit_start[P.pass + 1] - slab0, ring_slabs);
  const size_t cap = P.q_hits.capacity;
  unsigned long long n_culled = 0;
  for (;;) {
    uint32_t slab = 0;
    if (lane == 0) slab = atomicAdd(&ctl->hit_cursor[P.pass], 1u);
    slab = __shfl_sync(kFull, slab, 0);
    if (slab >= n_slabs) break;
    slab = (slab + slab0) % ring_slabs;
    const uint32_t n_here = min(__ldg(P.q_hits.fill + slab), kSlab);
    for (uint32_t j = lane; j < n_here; j += 32) {
      const uint32_t item = slab * kSlab + j;
      const double2 a = P.q_hits.plane[item], b = P.q_hits.plane[cap + item], c = P.q_hits.plane[2 * cap + item],
                    d = P.q_hits.plane[3 * cap + item], e = P.q_hits.plane[4 * cap + item];
      const uint32_t sbits = P.q_hits.sample[item];
      const V3 p = mk(a.x, a.y, b.x), n = mk(b.y, c.x, c.y), cd = mk(d.x, d.y, e.x);
      const double w = e.y;
      if (P.q_hits.walk[item] & kHitDirect) {  // a finished term (Emmit / ShowNormal / ShowUV)
        accumulate(P, sbits & 0x7fffffffu, w, cd);
        continue;
      }
      const bool cd_finite = isfinite(cd.x) && isfinite(cd.y) && isfinite(cd.z);
      V3 acc = mk(0, 0, 0);  // foldl ... black lts
      for (uint32_t li = 0; li < S.n_lights; li++) {
        const rh_light& L = cx.lights[li];
        V3 ld, lc;
        light_at(L, p, ld, lc);
        // diffuse (Material.hs:31-33) = (max (l.n) 0 / pi) * (cd (*) lc): exactly zero when l.n <= 0 (and the colours
        // are finite), whether or not the point is shadowed, so the occlusion query cannot change the sum
        const double ldn = dot(ld, n);
        if (ldn <= 0 && cd_finite && light_is_tame(L)) {
          n_culled++;
          continue;
        }
        const Ray sr = rayEps(p, ld);
        const bool shadowed = occluded<COUNT>(cx, sr, P.exact_boxes || needs_exact_walk(sr, S), L, st, cnt);
        if (!shadowed) acc = acc + mul(hs_max(ldn, 0) * kPiInv, cmul(cd, lc));
      }
      const V3 total = (sbits & 0x80000000u) ? mul(0.2, cd) + acc : acc;
      accumulate(P, sbits & 0x7fffffffu, w, total);
    }
  }
  for (int o = 16; o > 0; o >>= 1) n_culled += __shfl_xor_sync(kFull, n_culled, o);
  if (lane == 0 && n_culled) atomicAdd(&P.counters->shadow_culled, n_culled);
  flush_counters<COUNT>(cnt, P.counters, 1);
}

// ------------------------------------------------------------------ batched ray queries (caller-supplied rays)
// query_closest_kernel: closestIntersection (RayHs.hs:67-71) + the winner's Hit; query_shadow_kernel:
// shadowIntersection (RayHs.hs:74-87) towards one light through the general object-list form (`occluded`): the cube
// maps and lit-triangle flags only hold for rays aimed at a light from a shaded hit.  One ray per lane, persistent warps
// with the trace kernel's guided claims.  A warp's 32 rays (48 bytes each) arrive as coalesced 16-byte loads, three per
// lane, through the warp's shared-memory tile, and its 32 80-byte records leave the same way, five stores per lane.
constexpr int kQueryBlock = kTraceBlock;  // one block per SM: grid x block <= max_threads_per_launch (deep-stack scratch)
struct QueryWarpSmem {
  double2 tile[32 * sizeof(rh_hit) / sizeof(double2)];
};
static_assert(sizeof(rh_hit) == 80, "rh_hit is five 16-byte words");
constexpr size_t kQuerySmem = sizeof(SmemTables) + (size_t)kShortStack * kQueryBlock * sizeof(uint2) +
                              (kQueryBlock / 32) * sizeof(QueryWarpSmem);
static_assert(kQuerySmem <= 227 * 1024, "query kernel shared memory");

__device__ __forceinline__ Stack make_query_stack(const QueryParams& Q) {
  Stack s;
  s.col = reinterpret_cast<uint2*>(rh_smem + sizeof(SmemTables)) + threadIdx.x;
  s.stride = kQueryBlock;
  s.deep = Q.deep_stack + (size_t)blockIdx.x * kQueryBlock + threadIdx.x;
  s.deep_stride = Q.deep_stride;
  return s;
}
__device__ __forceinline__ double2* query_tile() {
  return reinterpret_cast<QueryWarpSmem*>(rh_smem + sizeof(SmemTables) + (size_t)kShortStack * kQueryBlock * sizeof(uint2))[threadIdx.x >> 5].tile;
}

// The claims of one warp: body(first, count) for pieces of at most 32 consecutive rays.
template <class Body>
__device__ __forceinline__ void claim_rays(const QueryParams& Q, uint32_t lane, Body&& body) {
  const uint32_t n_units = (Q.n + kSlab - 1) / kSlab * kSlabUnits, total_warps = gridDim.x * (kQueryBlock / 32);
  uint32_t seen = (blockIdx.x * (kQueryBlock / 32) + (threadIdx.x >> 5)) * kSlabUnits;
  for (;;) {
    const uint2 claim = claim_units(Q.cursor, n_units, total_warps, lane, seen);
    if (claim.x >= n_units) break;
    const uint32_t claim_end = min(claim.x + claim.y, n_units);
    for (uint32_t u = claim.x; u < claim_end;) {
      uint32_t slab, b, piece_n;
      next_piece(u, claim_end, slab, b, piece_n);
      const uint32_t first = slab * kSlab + b;
      if (first < Q.n) body(first, min(piece_n, Q.n - first));
    }
  }
}

// Ray `first + lane` of a piece (lanes >= count get whatever the tile holds and must not use it).
__device__ __forceinline__ Ray load_query_ray(const QueryParams& Q, uint32_t first, uint32_t count, double2* tile, uint32_t lane) {
  const double2* src = reinterpret_cast<const double2*>(Q.rays + (size_t)first * 6);
  __syncwarp();  // the tile's previous contents have been read
  for (uint32_t k = lane; k < 3 * count; k += 32) tile[k] = __ldcs(src + k);
  __syncwarp();
  const double2 a = tile[3 * lane], b = tile[3 * lane + 1], c = tile[3 * lane + 2];
  Ray r;
  r.o = mk(a.x, a.y, b.x);
  r.d = mk(b.y, c.x, c.y);
  return r;
}

__global__ void __launch_bounds__(kQueryBlock, 1) query_closest_kernel(const __grid_constant__ SceneView S,
                                                                       const __grid_constant__ QueryParams Q) {
  SmemTables& sm = *reinterpret_cast<SmemTables*>(rh_smem);
  Ctx cx;
  stage_tables(sm, S, cx);
  Stack st = make_query_stack(Q);
  Cnt<false> cnt;
  const uint32_t lane = threadIdx.x & 31;
  double2* tile = query_tile();
  claim_rays(Q, lane, [&](uint32_t first, uint32_t count) {
    const bool valid = lane < count;
    const Ray r = load_query_ray(Q, first, count, tile, lane);
    Closest best;
    best.obj = -1;
    if (valid) closest_hit<false>(cx, r, Q.exact_boxes || needs_exact_walk(r, S), best, st, cnt);
    double t = __longlong_as_double(0x7ff0000000000000LL);  // a miss: t = +inf, p = n = uv = 0, ids -1
    V3 p = mk(0, 0, 0), n = mk(0, 0, 0);
    double tu = 0, tv = 0;
    int tri = -1;
    if (best.obj >= 0) {
      const DObject& ob = cx.objects[best.obj];
      const int okind = ob.kind;
      t = best.t;
      rebuild_hit<false>(S, ob, okind, r, best, true, p, n, tu, tv, cnt);
      if (okind == RH_OBJ_MESH) tri = (int)S.tris[best.slot].tri_id;
    }
    __syncwarp();  // every lane has its ray out of the tile
    double2* rec = tile + 5 * lane;
    rec[0] = make_double2(t, p.x);
    rec[1] = make_double2(p.y, p.z);
    rec[2] = make_double2(n.x, n.y);
    rec[3] = make_double2(n.z, tu);
    rec[4] = make_double2(tv, __hiloint2double(tri, best.obj));
    __syncwarp();
    double2* dst = reinterpret_cast<double2*>(Q.hits + first);
    for (uint32_t k = lane; k < 5 * count; k += 32) __stcs(dst + k, tile[k]);
  });
}

__global__ void __launch_bounds__(kQueryBlock, 1) query_shadow_kernel(const __grid_constant__ SceneView S,
                                                                      const __grid_constant__ QueryParams Q) {
  SmemTables& sm = *reinterpret_cast<SmemTables*>(rh_smem);
  Ctx cx;
  stage_tables(sm, S, cx);
  Stack st = make_query_stack(Q);
  Cnt<false> cnt;
  const uint32_t lane = threadIdx.x & 31;
  double2* tile = query_tile();
  const rh_light& L = cx.lights[Q.light];
  claim_rays(Q, lane, [&](uint32_t first, uint32_t count) {
    const Ray r = load_query_ray(Q, first, count, tile, lane);
    if (lane < count)
      Q.occluded[first + lane] = occluded<false>(cx, r, Q.exact_boxes || needs_exact_walk(r, S), L, st, cnt) ? 1 : 0;
  });
}

// After pass k's trace kernel: its shaded hits are the slabs [hit_start[k], hit_start[k + 1]) of the hit queue.
__global__ void close_hit_range_kernel(ChunkCtl* ctl, int pass) { ctl->hit_start[pass + 1] = ctl->hit_slab_next; }

// ------------------------------------------------------------------ K6: average + toIntC (RayHs.hs:169-171, Image.hs:54-55)
__device__ __forceinline__ int to_int_c(double c, bool& negative) {
  const double v = 255 * hs_min(c, 1);  // hs_min NaN 1 = 1
  if (v < 0) {
    if (v <= -1) negative = true;
    return 0;
  }
  return min((int)v, 255);  // truncate toward zero, then the RGB8 clamp (SURVEY App. A-Q2)
}

__global__ void __launch_bounds__(kBlock) resolve_kernel(const __grid_constant__ ChunkParams P) {
  __shared__ __align__(16) uint8_t bytes[kBlock * 3];
  const uint32_t n_pixels = P.n_rows * P.width;
  const uint32_t lp = blockIdx.x * kBlock + threadIdx.x;
  bool negative = false;
  if (lp < n_pixels) {
    uint8_t r8 = 0, g8 = 0, b8 = 0;
    const uint32_t lrow = lp / P.width;
    if (global_row(P, P.first_row + lrow) < P.height) {
      double sr = 0, sg = 0, sb = 0;  // foldl (+) black
      const double* a = P.accum + (size_t)lp * P.spp;
      if ((P.spp & 1u) == 0 && (P.accum_stride & 1u) == 0) {
        // a pixel's samples are one contiguous run per plane: 16-byte loads halve the L1 wavefronts of this streaming
        // read (every lane of a warp is in a different 128-byte line); the sum stays in sample order
        const double2* a0 = (const double2*)a;
        const double2* a1 = (const double2*)(a + P.accum_stride);
        const double2* a2 = (const double2*)(a + 2 * (size_t)P.accum_stride);
        for (uint32_t s = 0; s < P.spp / 2; s++) {
          const double2 r2 = a0[s], g2 = a1[s], b2 = a2[s];
          sr = (sr + r2.x) + r2.y;
          sg = (sg + g2.x) + g2.y;
          sb = (sb + b2.x) + b2.y;
        }
      } else {
        for (uint32_t s = 0; s < P.spp; s++) {
          sr = sr + a[s];
          sg = sg + a[P.accum_stride + s];
          sb = sb + a[2 * (size_t)P.accum_stride + s];
        }
      }
      const double inv = 1.0 / (double)P.spp;
      r8 = (uint8_t)to_int_c(inv * sr, negative);
      g8 = (uint8_t)to_int_c(inv * sg, negative);
      b8 = (uint8_t)to_int_c(inv * sb, negative);
    }
    bytes[3 * threadIdx.x] = r8;
    bytes[3 * threadIdx.x + 1] = g8;
    bytes[3 * threadIdx.x + 2] = b8;
  }
  const unsigned neg = __ballot_sync(kFull, negative);
  if ((threadIdx.x & 31) == 0 && neg) atomicAdd(&P.counters->negative_channels, (unsigned long long)__popc(neg));
  __syncthreads();
  const uint32_t n_here = min((uint32_t)kBlock, n_pixels - blockIdx.x * kBlock) * 3;
  if (P.n_peers) {
    // Fused exchange: the block's bytes go straight into every shard's full frame (peer stores over NVLink), at the
    // image row of each byte.  Rows are whole multiples of 4 bytes and the block starts on a word when width % 4 == 0,
    // so a 32-bit word never straddles two rows; otherwise byte stores.
    const uint32_t row_bytes = P.width * 3;
    const size_t local0 = (size_t)blockIdx.x * kBlock * 3;  // byte offset inside the chunk's compact rows
    const bool words = (row_bytes & 3u) == 0 && (local0 & 3u) == 0;
    const uint32_t step = words ? 4u : 1u;
    for (uint32_t i = threadIdx.x * step; i < n_here; i += kBlock * step) {
      const size_t lb = local0 + i;
      const uint32_t lrow = (uint32_t)(lb / row_bytes), inrow = (uint32_t)(lb - (size_t)lrow * row_bytes);
      const uint32_t grow = global_row(P, P.first_row + lrow);
      if (grow >= P.height) continue;  // padding row of the last band
      const size_t at = (size_t)grow * row_bytes + inrow;
      if (words && i + 4 <= n_here) {
        const uint32_t v = *(const uint32_t*)(bytes + i);
        for (uint32_t g = 0; g < P.n_peers; g++) *(uint32_t*)(P.peer[g] + at) = v;
      } else {
        for (uint32_t k = 0; k < step && i + k < n_here; k++)
          for (uint32_t g = 0; g < P.n_peers; g++) P.peer[g][at + k] = bytes[i + k];
      }
    }
    return;
  }
  // coalesced store: the block's 384 bytes leave as 32-bit words when the destination allows it
  uint8_t* dst = P.rgb + ((size_t)P.first_row * P.width + (size_t)blockIdx.x * kBlock) * 3;
  if ((((uintptr_t)dst) & 3) == 0) {
    const uint32_t words = n_here / 4;
    if (threadIdx.x < words) ((uint32_t*)dst)[threadIdx.x] = ((const uint32_t*)bytes)[threadIdx.x];
    const uint32_t tail = words * 4 + threadIdx.x;
    if (tail < n_here) dst[tail] = bytes[tail];
  } else {
    for (uint32_t i = threadIdx.x; i < n_here; i += kBlock) dst[i] = bytes[i];
  }
}

// ------------------------------------------------------------------ K6': rh_trace_rays' colours (RayHs.hs:149-154)
// One ray per sample, so the accumulators are the colours traceRay returns: the three planes of a block's rays are read
// coalesced and leave interleaved as double[3] per ray, also coalesced, through shared memory.  No arithmetic.
__global__ void __launch_bounds__(kBlock) store_colors_kernel(const __grid_constant__ ChunkParams P, double* __restrict__ colors) {
  __shared__ double rgb[kBlock * 3];
  const uint32_t first = blockIdx.x * kBlock, n_here = min((uint32_t)kBlock, P.ray_items - first);
  if (threadIdx.x < n_here)
    for (int c = 0; c < 3; c++) rgb[3 * threadIdx.x + c] = P.accum[(size_t)c * P.accum_stride + first + threadIdx.x];
  __syncthreads();
  double* dst = colors + ((size_t)P.first_row * P.width + first) * 3;
  for (uint32_t i = threadIdx.x; i < 3 * n_here; i += kBlock) dst[i] = rgb[i];
}

// ------------------------------------------------------------------ K7: band de-interleave after the all-gather
__global__ void deinterleave_kernel(const uint8_t* __restrict__ gathered, uint8_t* __restrict__ out, uint32_t row_bytes,
                                    uint32_t height, uint32_t shard_count, uint32_t band_height, uint32_t rows_per_shard) {
  const uint32_t row = blockIdx.y;
  if (row >= height) return;
  const uint32_t band = row / band_height, rib = row % band_height;
  const uint32_t shard = band % shard_count, lrow = (band / shard_count) * band_height + rib;
  const uint8_t* src = gathered + ((size_t)shard * rows_per_shard + lrow) * row_bytes;
  uint8_t* dst = out + (size_t)row * row_bytes;
  if (((row_bytes & 3) == 0) && ((((uintptr_t)src) | ((uintptr_t)dst)) & 3) == 0) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < row_bytes / 4; i += gridDim.x * blockDim.x)
      ((uint32_t*)dst)[i] = ((const uint32_t*)src)[i];
  } else {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < row_bytes; i += gridDim.x * blockDim.x) dst[i] = src[i];
  }
}

// ------------------------------------------------------------------ micro-benchmarks (roofline denominators)
// Random 128-byte record gathers (the wide-node access pattern), `loads` independent records per thread.
__global__ void gather_bench_kernel(const double2* __restrict__ buf, uint64_t n_records, uint32_t loads, double2* sink) {
  uint64_t x = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull + 0x1234567ull;
  double2 acc = make_double2(0, 0);
  for (uint32_t i = 0; i < loads; i += 4) {
    uint64_t idx[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
      idx[k] = x % n_records;
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double2* p = buf + idx[k] * 8;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const double2 v = __ldg(p + j);
        acc.x += v.x;
        acc.y += v.y;
      }
    }
  }
  if (acc.x == 1.2345e300) sink[0] = acc;
}

__global__ void dfma_bench_kernel(double* sink, int iters) {
  double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
    a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 1.2345e300) sink[0] = s;
}

// Sequential 16-byte loads over a buffer (coalesced, every byte once per sweep): with a buffer that fits the 126 MB L2
// this is the L2 -> SM streaming rate, the denominator for `lts__t_bytes` of the traversal kernels.
__global__ void stream_bench_kernel(const double2* __restrict__ buf, uint64_t n_elems, double2* sink) {
  double2 acc = make_double2(0, 0);
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_elems; i += 4 * stride) {
    double2 v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) v[k] = (i + k * stride < n_elems) ? __ldg(buf + i + k * stride) : make_double2(0, 0);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      acc.x += v[k].x;
      acc.y += v[k].y;
    }
  }
  if (acc.x == 1.2345e300) sink[0] = acc;
}

}  // namespace

// ------------------------------------------------------------------ launchers
static int g_classify_grid[2] = {148, 148};
int configure_kernels() {
  cudaError_t e = cudaSuccess;
  auto set = [&](const void* fn, size_t bytes) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  };
  set((const void*)trace_kernel<true, false>, kTraceSmem);
  set((const void*)trace_kernel<false, false>, kTraceSmem);
  set((const void*)trace_kernel<false, true>, kTraceSmem);
  set((const void*)shadow_pooled_kernel<true>, kShadowSmem);
  set((const void*)shadow_pooled_kernel<false>, kShadowSmem);
  set((const void*)shadow_refill_kernel<true>, kWalkSmem);
  set((const void*)shadow_refill_kernel<false>, kWalkSmem);
  set((const void*)shadow_simple_kernel<true>, kSimpleSmem);
  set((const void*)shadow_simple_kernel<false>, kSimpleSmem);
  set((const void*)classify_kernel<true, true>, kClassifySmem);
  set((const void*)classify_kernel<false, true>, kClassifySmem);
  set((const void*)classify_kernel<true, false>, kClassifySmem);
  set((const void*)classify_kernel<false, false>, kClassifySmem);
  set((const void*)query_closest_kernel, kQuerySmem);
  set((const void*)query_shadow_kernel, kQuerySmem);
  if (e == cudaSuccess) {
    int dev = 0, sms = 0, nb = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    for (int c = 0; c < 2; c++) {
      if (c) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, classify_kernel<true, true>, kClassifyBlock, kClassifySmem);
      else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, classify_kernel<false, true>, kClassifyBlock, kClassifySmem);
      g_classify_grid[c] = sms * (nb > 0 ? nb : 1);
    }
  }
  return (int)e;
}
int max_threads_per_launch(int n_sms) {
  const int t = kTraceBlock * kTracePerSm, s = kShadowBlock * (kShadowPerSm > 1 ? kShadowPerSm : 1);  // (the simple kernel: one block)
  const int b = t > s ? (t > kWalkBlock ? t : kWalkBlock) : (s > kWalkBlock ? s : kWalkBlock);
  return n_sms * b;  // threads per SM of the largest traversal kernel
}
void launch_trace(const SceneView& S, const CameraParams& cam, const ChunkParams& P, bool count, int grid, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (P.offset_mode == kOffsetsRays) trace_kernel<false, true><<<grid * kTracePerSm, kTraceBlock, kTraceSmem, st>>>(S, cam, P);
  else if (count) trace_kernel<true, false><<<grid * kTracePerSm, kTraceBlock, kTraceSmem, st>>>(S, cam, P);
  else trace_kernel<false, false><<<grid * kTracePerSm, kTraceBlock, kTraceSmem, st>>>(S, cam, P);
  close_hit_range_kernel<<<1, 1, 0, st>>>(P.ctl, P.pass);
}
int launch_shadow(const SceneView& S, const ChunkParams& P, bool count, bool refill, int grid, void* stream, void* classified) {
  cudaStream_t st = (cudaStream_t)stream;
  if (S.n_lights > (uint32_t)kMaskLights) {
    if (count) shadow_simple_kernel<true><<<grid, kShadowBlock, kSimpleSmem, st>>>(S, P);
    else shadow_simple_kernel<false><<<grid, kShadowBlock, kSimpleSmem, st>>>(S, P);
    if (classified) cudaEventRecord((cudaEvent_t)classified, st);
    return 1;
  }
  // FAST: the occluder tables are the staged shared-memory ones (SceneView::shadow_fast)
  if (S.shadow_fast) {
    if (count) classify_kernel<true, true><<<g_classify_grid[1], kClassifyBlock, kClassifySmem, st>>>(S, P);
    else classify_kernel<false, true><<<g_classify_grid[0], kClassifyBlock, kClassifySmem, st>>>(S, P);
  } else {
    if (count) classify_kernel<true, false><<<g_classify_grid[1], kClassifyBlock, kClassifySmem, st>>>(S, P);
    else classify_kernel<false, false><<<g_classify_grid[0], kClassifyBlock, kClassifySmem, st>>>(S, P);
  }
  if (classified) cudaEventRecord((cudaEvent_t)classified, st);  // the pass's slabs of the hit queue are free again
  if (refill) {
    if (count) shadow_refill_kernel<true><<<grid, kWalkBlock, kWalkSmem, st>>>(S, P);
    else shadow_refill_kernel<false><<<grid, kWalkBlock, kWalkSmem, st>>>(S, P);
  } else {
    if (count) shadow_pooled_kernel<true><<<grid * kShadowPerSm, kShadowBlock, kShadowSmem, st>>>(S, P);
    else shadow_pooled_kernel<false><<<grid * kShadowPerSm, kShadowBlock, kShadowSmem, st>>>(S, P);
  }
  return 2;
}
void launch_resolve(const ChunkParams& P, void* stream) {
  const uint32_t n_pixels = P.n_rows * P.width;
  resolve_kernel<<<(n_pixels + kBlock - 1) / kBlock, kBlock, 0, (cudaStream_t)stream>>>(P);
}
void launch_store_colors(const ChunkParams& P, double* colors, void* stream) {
  store_colors_kernel<<<(P.ray_items + kBlock - 1) / kBlock, kBlock, 0, (cudaStream_t)stream>>>(P, colors);
}
void launch_query_closest(const SceneView& S, const QueryParams& Q, int grid, void* stream) {
  query_closest_kernel<<<grid, kQueryBlock, kQuerySmem, (cudaStream_t)stream>>>(S, Q);
}
void launch_query_shadow(const SceneView& S, const QueryParams& Q, int grid, void* stream) {
  query_shadow_kernel<<<grid, kQueryBlock, kQuerySmem, (cudaStream_t)stream>>>(S, Q);
}
void launch_deinterleave(const uint8_t* gathered, uint8_t* out, int width, int height, int shard_count, int band_height,
                         void* stream) {
  const uint32_t n_bands = (height + band_height - 1) / band_height;
  const uint32_t rows_per_shard = ((n_bands + shard_count - 1) / shard_count) * band_height;
  dim3 grid(4, height);
  deinterleave_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(gathered, out, (uint32_t)width * 3, height, shard_count,
                                                              band_height, rows_per_shard);
}
void launch_gather_bench(const double2* buf, uint64_t n_records, uint32_t loads_per_thread, double2* sink, int grid, int block,
                         void* stream) {
  gather_bench_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(buf, n_records, loads_per_thread, sink);
}
void launch_stream_bench(const double2* buf, uint64_t n_elems, double2* sink, int grid, int block, void* stream) {
  stream_bench_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(buf, n_elems, sink);
}
void launch_dfma_bench(double* sink, int iters, int grid, int block, void* stream) {
  dfma_bench_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(sink, iters);
}

}  // namespace rhd
