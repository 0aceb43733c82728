// device_types.cuh — HBM layouts and kernel parameter blocks of the ray-casting path.
// See DESIGN.md "Data layout in HBM".
#pragma once
#include <cstdint>

#include "../../include/rayhs_b200.h"

namespace rhd {

constexpr uint32_t kEmpty = 0xFFFFFFFFu;    // KDTree.hs:61 `Empty`
constexpr uint32_t kLeafBit = 0x80000000u;  // child reference is a leaf
constexpr uint32_t kSphereLeafBit = 0x40000000u;  // ... a leaf of the sphere tree: its slots index sphere_refs
constexpr uint32_t kCountMask = 0x3FFFFFFFu;      // exact (double) tree: low 30 bits of a leaf reference = triangle count
// Leaf reference of the float path's cull tree (WideNode32::child), self-contained so that a stacked subtree is ONE
// 32-bit word: kLeafBit | kSphereLeafBit? | (count - 1) << 27 | first slot.  Cull-tree leaves hold at most kSubLeaf
// triangles and sphere-tree leaves at most 4 spheres, so 3 bits of count and 27 bits of slot (134 M triangles) do.
constexpr uint32_t kLeafCountShift = 27, kLeafFirstMask = 0x07FFFFFFu, kLeafMaxCount = 8;
constexpr int kMaxDepth = 30;               // ray-tree depth limit accepted by rh_render (reference scenes use 3)
constexpr int kMaxPasses = 2 * kMaxDepth + 2;  // a Transparent hit inserts one probe pass per level (RayHs.hs:136-143)
constexpr int kStack = 112;                 // deepest stack a walk may need: tree depth <= 100 (KDTree.hs:76-77, 82) + roots
#ifndef RH_SHORT_STACK
#define RH_SHORT_STACK 8
#endif
// Traversal stack entries per thread held in SHARED memory (8 bytes each: subtree reference + float entry distance).
// Deeper entries — and the whole stack of the rare exact (double box) walk — go to the thread's column of a scratch
// area in global memory that the runtime sizes from the scene's tree depth.  No stack lives in local memory.
constexpr int kShortStack = RH_SHORT_STACK;
// Queue entries per slab: the unit a warp reserves (producer) or claims (consumer) with ONE global atomic.
constexpr uint32_t kSlab = 128;
#ifndef RH_SMEM_NODES
#define RH_SMEM_NODES 448
#endif
constexpr int kSmemNodes = RH_SMEM_NODES;   // top wide (fp32) nodes staged in shared memory (64 B each)
constexpr int kSmemObjects = 64;            // object / material tables staged when the scene has at most this many
constexpr int kSmemLights = 16;
constexpr int kBlock = 128;                // resolve kernel
constexpr int kMaxPeers = 16;
#ifndef RH_TRACE_BLOCK
#define RH_TRACE_BLOCK 768
#endif
#ifndef RH_SHADOW_BLOCK
#define RH_SHADOW_BLOCK 768
#endif
#ifndef RH_WALK_BLOCK
#define RH_WALK_BLOCK 640  // threads per block of the per-lane-refill shadow kernel (one block per SM)
#endif
#ifndef RH_WALK_UNROLL
#define RH_WALK_UNROLL 2
#endif
#ifndef RH_REFILL_MIN
#define RH_REFILL_MIN 16
#endif
#ifndef RH_TMA_STAGE
#define RH_TMA_STAGE 0  // trace kernel: the next batch's sample offsets (1) or also the next batch of queued rays (2) arrive by a bulk async copy (cp.async.bulk + mbarrier) while the current batch is traced; 0 = plain loads.  Measured on the bench frame: 0 = 41.3 ms, 1 = 42.4 ms, 2 = 42.8 ms — the loads it replaces are one coalesced LDG.128 per lane whose latency the other warps of the SM already hide, while the tile, the mbarrier handshake and the shared memory taken from L1 cost more than they save: off by default
#endif
#ifndef RH_TRACE_PER_SM
#define RH_TRACE_PER_SM 1   // resident blocks per SM of the trace kernel (block size x this = threads per SM)
#endif
#ifndef RH_SHADOW_PER_SM
#define RH_SHADOW_PER_SM 1  // ... of the pooled shadow kernel
#endif
constexpr int kTracePerSm = RH_TRACE_PER_SM, kShadowPerSm = RH_SHADOW_PER_SM;
constexpr int kTraceBlock = RH_TRACE_BLOCK;    // tables staged once per block
constexpr int kShadowBlock = RH_SHADOW_BLOCK;
constexpr int kWalkBlock = RH_WALK_BLOCK;

// 128-byte "wide" node of the EXACT walk: one record per inner node of the reference's own tree (KDTree.hs:59-61)
// holding BOTH child boxes in double, so every box is tested exactly once, as in KDTree.hs:96-107 (box test at every
// Node and Leaf).  A synthetic super-root per mesh carries the root's own box in slot 0.  Level order over all meshes.
struct __align__(16) WideNode {
  double box[12];     // child0 lo.xyz hi.xyz, child1 lo.xyz hi.xyz
  uint32_t child[2];  // kEmpty | kLeafBit|count | wide-node index
  uint32_t first[2];  // leaf child: first triangle slot
  uint32_t refine;    // bit c: child c's box is not a box the reference tests (sphere tree): the exact walk passes it
  uint32_t pad_[3];
};
#ifndef RH_STREAM_CHUNK_MI
#define RH_STREAM_CHUNK_MI 16  // chunk size (Mi samples) when the sample offsets stream in from the host
#define RH_STREAM_FIRST_MI 4   // ... and of the first chunk, whose upload nothing overlaps
#endif
#ifndef RH_LANES
#define RH_LANES 2  // chunks in flight (streams with their own queues); 1 = strictly one chunk after the other
#endif
#ifndef RH_SUBLEAF
#define RH_SUBLEAF 4  // triangles per leaf of the float path's cull tree (measured: 3-4 best of 2, 3, 4, 6, 8)
#endif
constexpr uint32_t kSubLeaf = RH_SUBLEAF;
static_assert(kSubLeaf <= kLeafMaxCount, "cull-tree leaf count must fit the packed leaf reference");
static_assert(sizeof(WideNode) == 128, "WideNode must be 128 bytes");

// 64-byte node of the float path's cull tree: two child boxes rounded OUTWARD to float, relative to SceneView::center.
// The fp32 slab test on it is conservative (never rejects a box the double test of KDTree.hs:39-56 accepts, see
// kernels.cu), so it only decides which triangles get the exact double test.  child: kEmpty | packed leaf reference
// (see kLeafCountShift) | node index.
struct __align__(16) WideNode32 {
  float box[12];
  uint32_t child[2];
  uint32_t pad_[2];
};
static_assert(sizeof(WideNode32) == 64, "WideNode32 must be 64 bytes");

// Object table entry (device copy of rh_object with the wide super-root index).
struct __align__(16) DObject {
  double a[3], b[3], c[3];
  int32_t kind;
  int32_t material;
  uint32_t root;  // wide-node index of the mesh's super-root or kEmpty
  uint32_t is_emitter;
};
static_assert(sizeof(DObject) == 96, "DObject must be 96 bytes");

// Occluder tables (shadowIntersection, RayHs.hs:74-82): the non-emitter planes and the non-emitter spheres that are
// not in the sphere tree, as compact records, and the super-roots of the non-emitter, non-empty meshes.
struct OccPlane { double p[3], n[3]; };   // Geometry.hs:62
struct OccSphere { double c[3], r; };     // Geometry.hs:63
constexpr int kOccPlanes = 16, kOccSpheres = 16, kOccMeshes = 8, kFastLights = 12;
constexpr int kMaskLights = 32;  // lights whose per-hit state fits the 32-bit walk / settled masks of a shadow task

struct SceneView {
  const WideNode* wide;      // exact double boxes: rays with a zero direction component, RH_FLAG_EXACT_BOXES
  const WideNode32* wide32;  // conservative float boxes: everything else
  const rh_tri* tris;
  const rh_tri_shade* shade;
  const DObject* objects;
  const rh_material* materials;
  const rh_light* lights;
  const rh_texture* textures;
  const double* texels;
  const uint32_t* lin_objs;     // objects scanned linearly in scene order (RayHs.hs:64-71): all of them, or all but the spheres
  const uint32_t* sphere_refs;  // sphere tree leaves: object indices
  const uint32_t* exact_index;  // exact walk: slot of the reference tree's leaves -> slot in tris / shade (null: identical)
  uint32_t n_lin;
  uint32_t sphere_root;         // super-root of the sphere tree or kEmpty (spheres are in lin_objs then)
  const OccPlane* occ_planes;
  const OccSphere* occ_spheres;
  const uint32_t* occ_meshes;
  uint32_t n_occ_planes, n_occ_spheres, n_occ_meshes;
  uint32_t shadow_fast;         // the occluder tables and the lights fit the shared-memory tables (root boxes, light sides, cube maps usable)
  uint32_t n_wide, n_tris, n_objects, n_materials, n_lights, n_textures;
  uint32_t n_smem_nodes;    // min(n_wide, kSmemNodes)
  uint32_t tables_in_smem;  // objects/materials/lights fit the staged tables
  float abs_max;            // largest |coordinate - center| of any tree box (pads the fp32 slab test)
  uint32_t light_map_res;   // cells per edge of a cube-map face
  double center[3];         // the float boxes of wide32 are stored relative to this point
  // Per (point light, occluder mesh) cube maps of the nearest possible occluder distance (light_maps.cpp): map k is
  // light_maps[k * 6 * res * res ..], face-major; light_map_index[light * kOccMeshes + mesh] = k or kEmpty.
  // Null when the scene has none (no point light, no mesh, maps useless or switched off).
  const float* light_maps;
  const uint32_t* light_map_index;
  // Lit triangles (light_maps.cpp), per triangle slot: bit l = nothing of the triangle's own mesh can shadow a point
  // of it from light l (l < 12, point or directional); bits 12-15 = the mesh's index in occ_meshes.  Null when the
  // scene has none.
  const uint16_t* lit_flags;
};

// Camera with everything `rayFromPixel` recomputes per pixel hoisted to the host
// (Projection.hs:22-46, Mat.hs:89-93): the values are identical, they are just computed once.
struct CameraParams {
  double m[9];  // lookAt matrix rows (Mat.hs:83-93)
  double pos[3];
  double w, h, half_w, half_h, apw, aph, f;
  int32_t projection;
  int32_t pad_;
};

// Per-chunk control block in device memory (zeroed before each chunk).
struct ChunkCtl {
  uint32_t ray_slabs[kMaxPasses + 2];     // slabs reserved in the ray queue that pass k consumes
  // The hit queue is a ring of slabs addressed by ONE running counter over all passes of a chunk: pass k's shaded hits
  // are the slabs [hit_start[k], hit_start[k + 1]) (mod the ring), so that pass k + 1's trace kernel can append while
  // pass k's hits are still being classified on the other stream; pass k + 2 reuses pass k's slabs.  hit_start[k + 1] is
  // written when pass k's trace kernel has ended.
  uint32_t hit_start[kMaxPasses + 3];
  uint32_t shadow_slabs[kMaxPasses + 2];  // slabs of hits whose shadow rays have to walk a tree (walk queue)
  uint32_t trace_cursor[kMaxPasses + 2];  // persistent-warp work cursors, in claim units
  uint32_t hit_cursor[kMaxPasses + 2];
  uint32_t shadow_cursor[kMaxPasses + 2];
  uint32_t ray_items[kMaxPasses + 2];     // entries in those slabs (statistics; one atomic per warp per launch)
  uint32_t hit_items[kMaxPasses + 2];
  uint32_t shadow_items[kMaxPasses + 2];
  uint32_t overflow;
  uint32_t hit_slab_next;                 // the hit queue's slab counter
  uint32_t pad_[1];
};

// Frame-level counters (zeroed per rh_render).
struct KernelCounters {  // RH_FLAG_COUNT only
  unsigned long long box_tests, tri_tests, prim_tests, node_visits, shade_fetches, texel_fetches, global_node_visits, tri_records;
};
struct FrameCounters {
  unsigned long long rays_reflect, rays_probe, rays_exit, negative_channels;
  unsigned long long shaded_hits;    // Diffuse / Plastic hits: each is one accumDiffuse fold over all lights (RayHs.hs:89-97)
  unsigned long long shadow_culled;  // (hit, light) pairs with l.n <= 0: Lambert term is exactly 0, query skipped
  unsigned long long shadow_walk_pairs;  // (hit, light) pairs that went to a tree walk
  unsigned long long exact_walks;    // RH_FLAG_COUNT: shadow rays that took the exact (double box) walk
  unsigned long long max_walk_nodes; // RH_FLAG_COUNT: most node records one shadow ray visited
  unsigned long long exact_closest;  // RH_FLAG_COUNT: closest-hit rays that took the exact walk
  unsigned long long max_closest_nodes;
  unsigned long long deep_pushes;    // RH_FLAG_COUNT: stack entries that went beyond the shared-memory short stack
  KernelCounters k[2];  // 0 = trace_kernel, 1 = shadow kernels
  // RH_FLAG_COUNT: shadow walks by floor(log2(node records visited + 1)), per pass (last row: passes >= 3), and the nodes they visited
  unsigned long long walk_hist[4][20], walk_hist_nodes[4][20];
#ifdef RH_WARP_TIMES
  // diagnostic build (-DRH_WARP_TIMES): per warp of the pooled shadow kernel and pass (row 3: passes >= 3): the low 32 bits of its first
  // and last globaltimer reading (ns), batches of 32 hits it processed, walk rounds it ran
  unsigned int warp_begin[4][4096], warp_end[4][4096], warp_batches[4][4096], warp_rounds[4][4096];
  // ... ns inside the walk rounds, and over its rounds the sums of the longest lane's node steps / triangle tests
  unsigned int warp_walk_ns[4][4096], warp_max_nodes[4][4096], warp_max_tris[4][4096], warp_pairs[4][4096];
#endif
};

// Queues are arrays of slabs of kSlab entries; slab s holds fill[s] <= kSlab valid entries at [s * kSlab ..).  A warp
// reserves a slab with one atomic and fills it privately; the consumer claims whole slabs.
// SoA-of-16-byte planes so that a warp's compacted pushes are fully coalesced.
// Ray queue: 4 planes (ox,oy) (oz,dx) (dy,dz) (weight, bits).
// bits = sample | depth << 32 | kind << 40 | material << 48.
struct RayQueue {
  double2* plane;  // plane k at plane + k*capacity
  uint32_t* fill;  // entries per slab
  uint32_t capacity;  // entries (a multiple of kSlab)
};
// Hit queue (every shaded Diffuse / Plastic hit of a pass) and walk queue (the hits with a light whose shadow ray has
// to walk a tree): 5 planes (px,py) (pz,nx) (ny,nz) (cr,cg) (cb,w) + sample ids (bit 31 = ambient term) + two words.
struct ShadowQueue {
  double2* plane;
  uint32_t* sample;
  uint32_t* walk;     // walk queue: bit l = the shadow ray towards light l has to walk a tree; hit queue: the lit-triangle flags of the hit triangle
  uint32_t* settled;  // walk queue: bit l = light l adds nothing (l.n <= 0, or a plane / sphere occludes)
  uint32_t* fill;
  uint32_t capacity;
};

enum { kRayNormal = 0, kRayProbe = 1 };
enum { kOffIndexLocal = 0, kOffIndexGlobal = 1 };
// ChunkParams::offset_mode of rh_trace_rays (not an RH_OFFSETS_* value): the pass-0 work items are caller-built rays,
// double[6] = origin, direction, at `offsets` (ray of item i: offset_base + i), instead of camera rays.
constexpr int kOffsetsRays = 16;

struct ChunkParams {
  uint32_t first_row;     // first local (shard-compact) row of the chunk
  uint32_t n_rows;        // rows in the chunk
  uint32_t n_samples;     // n_rows * width * spp
  uint32_t spp;
  uint32_t width, height;
  uint32_t shard_index, shard_count, band_height;
  int32_t max_depth;
  int32_t offset_mode;    // RH_OFFSETS_*
  int32_t offset_index;   // kOffIndex*: per-pixel offsets indexed by chunk-local or full-frame pixel
  int32_t offset_tile;
  int32_t pass;           // wavefront pass (0 = primary)
  int32_t exact_boxes;    // RH_FLAG_EXACT_BOXES: double slab test for every ray (validation)
  int32_t no_light_maps;  // RH_FLAG_NO_LIGHT_MAPS: shadow rays ignore the lights' cube maps (validation, A/B)
  int32_t hit_live_pass;  // the hit queue (a ring) still holds the hits of this pass and later ones (pass, or pass - 1 when pipelined)
  uint32_t ray_items;     // kOffsetsRays: pass-0 items of the chunk that are rays (the rest of its last row is padding)
  const void* offsets;    // device
  uint32_t offset_linear; // f64 pairs in work-item order: pair of item i at offsets[offset_base + i] (bulk-copy staging)
  uint32_t pad5_;
  unsigned long long offset_base;
  unsigned long long offset_seed;  // RH_OFFSETS_SPLITMIX64
  double* accum;          // 3 planes of accum_stride (r,g,b), chunk-local sample order
  uint32_t accum_stride;
  uint32_t deep_stride;   // threads the deep-stack scratch has a column for (>= grid * block of every launch)
  uint2* deep_stack;      // [entry][thread]: stack entries beyond the short stack, and the exact walk's whole stack
  int2* hit_ids;          // shard-compact [pixel][spp] (object, tri) or null
  uint8_t* rgb;           // shard-compact framebuffer (or null with peer frames)
  uint8_t* peer[kMaxPeers];  // RH_FLAG_PEER_FRAMES: full frames of all shards
  uint32_t n_peers;
  uint32_t pad4_;
  ChunkCtl* ctl;
  FrameCounters* counters;
  RayQueue q_in, q_out;
  ShadowQueue q_hits, q_shadow;
};

// One launch of the batched ray queries (rh_closest_intersection / rh_shadow_intersection) over rays [0, n).
struct QueryParams {
  const double* rays;  // device, double[n][6] = origin, direction; 16-byte aligned
  rh_hit* hits;        // closest: one record per ray; 16-byte aligned
  uint8_t* occluded;   // shadow: 0 / 1 per ray
  uint32_t n;
  uint32_t light;      // shadow: index into the light table
  int32_t exact_boxes; // RH_FLAG_EXACT_BOXES: double slab test for every ray
  uint32_t deep_stride;
  uint2* deep_stack;   // the render's deep-stack scratch (>= grid * block columns)
  uint32_t* cursor;    // claim cursor, zero before the launch
};

// Launchers (kernels.cu).  `count` selects the instrumented instantiation (box/tri counters); launch_trace runs the
// uninstrumented ray instantiation for P.offset_mode == kOffsetsRays.
// (followed by a one-thread kernel that closes the pass's range of the hit queue, ChunkCtl::hit_start)
void launch_trace(const SceneView& S, const CameraParams& cam, const ChunkParams& P, bool count, int grid, void* stream);
// classify_kernel, then the walks of the hits it queued — refill: the per-lane-refill kernel (incoherent rays) instead of
// the pooled one (coherent rays).  Returns the number of launches.
// `classified`: a cudaEvent_t recorded after the classify kernel (or null).
int launch_shadow(const SceneView& S, const ChunkParams& P, bool count, bool refill, int grid, void* stream, void* classified);
void launch_resolve(const ChunkParams& P, void* stream);
// rh_trace_rays' end of a chunk instead of the resolve: the accumulators of its rays to colors (double[n][3], all rays)
void launch_store_colors(const ChunkParams& P, double* colors, void* stream);
// query_closest_kernel / query_shadow_kernel: `grid` blocks of one SM each
void launch_query_closest(const SceneView& S, const QueryParams& Q, int grid, void* stream);
void launch_query_shadow(const SceneView& S, const QueryParams& Q, int grid, void* stream);
void launch_deinterleave(const uint8_t* gathered, uint8_t* out, int width, int height, int shard_count, int band_height,
                         void* stream);
int configure_kernels();  // opt in to > 48 KB dynamic shared memory; returns a cudaError_t
int max_threads_per_launch(int n_sms);  // largest grid * block of the trace / shadow kernels (sizes the deep-stack scratch)
// setup_kernels.cu: the light-space tables of rh_scene_create, built on the device (return a cudaError_t)
int preload_setup_kernels();
int device_light_map(const double L[3], const rh_tri* d_tris, const uint32_t* d_slots, size_t n, int R, float* d_out, double min_empty,
                     unsigned long long* d_words, int* useful, double* empty_fraction, void* stream);
int device_lit_flags(const rh_tri* d_tris, const WideNode32* d_nodes, const double center[3], uint32_t root, const uint32_t* d_slots,
                     uint32_t n_slots, const rh_light* d_lights, uint32_t n_lights, uint32_t mesh, uint16_t* d_lit,
                     unsigned long long* d_flagged, void* stream);
// micro-benchmarks
void launch_gather_bench(const double2* buf, uint64_t n_records, uint32_t loads_per_thread, double2* sink, int grid, int block,
                         void* stream);
void launch_stream_bench(const double2* buf, uint64_t n_elems, double2* sink, int grid, int block, void* stream);
void launch_dfma_bench(double* sink, int iters, int grid, int block, void* stream);

}  // namespace rhd
