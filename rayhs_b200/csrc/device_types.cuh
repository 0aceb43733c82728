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
constexpr int kMaxGroups = 16;   // light groups of rh_render_light_groups
constexpr uint32_t kMaxViews = 65536;  // cameras of one rh_render_views call

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
  int32_t projection;  // RH_PROJ_*; a thin lens of radius 0 is RH_PROJ_PERSPECTIVE here
  int32_t pad_;
  double lens_r, focus;  // RH_PROJ_THIN_LENS: aperture radius R and focus distance F
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

// rh_render_adaptive's pass-0 source: P.spp samples of each entry of a list of the shard's pixels.  The frame's rows
// are rows of the list (P.width entries each; P.ray_items pass-0 items of the chunk are real, the rest of its last row is
// padding), so P's geometry is the list's; the image's is here.
struct PixelList {
  const uint32_t* pixels;  // shard-compact pixel index of each entry, ascending; null: not a list frame
  const uint32_t* counts;  // n_p: pixel p's samples continue the stream at pixel * stream_spp + counts[p]
  uint32_t width, height, shard_index, shard_count, band_height;  // the image and the shard's bands
};

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
  uint32_t reserved_;     // padding: keeps the offsets of the fields below
  uint32_t stream_spp;    // RH_OFFSETS_SPLITMIX64: samples per pixel of the stream (rh_render: spp) ...
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
  uint32_t stream_base;   // ... and the stream's first sample this call traces (rh_render: 0)
  ChunkCtl* ctl;
  FrameCounters* counters;
  RayQueue q_in, q_out;
  ShadowQueue q_hits, q_shadow;
  PixelList list;         // rh_render_adaptive (after the render's fields: their offsets stay as they were)
  // rh_render_light_groups (after the render's fields: their offsets stay as they were): the shadow kernels also add a
  // hit's terms split by light group to (n_groups + 1) x 3 planes of group_stride doubles, chunk-local sample order
  // (plane 3 g + c: group g, channel c; group n_groups: the remainder).  Null for every other frame.
  double* groups;
  uint32_t group_stride;
  uint32_t n_groups;
  uint32_t group_mask[kMaxGroups];  // bit l: light l is in group g
  // rh_render_views (after the render's fields: their offsets stay as they were): the frame's local rows are
  // [view][view_rows]; pass 0 builds local row r's rays with cams[r / view_rows] and, with view_seeds, SplitMix64 seed
  // view_seeds[r / view_rows].  view_rows 0 (cams null): not a views frame.
  const CameraParams* cams;
  const unsigned long long* view_seeds;
  uint32_t view_rows;
};

// rh_render_accumulate's end of a chunk instead of the resolve: the running per-pixel sums of the accumulator.
struct AccumParams {
  const double* sum_in;  // 3 planes (r, g, b) of `plane` doubles, shard-compact pixel order; not read when n_before == 0
  double* sum_out;       // the same layout: sum_in + this call's samples, in sample order
  double* linear;        // shard-compact double[pixel][3] = sum / n_total, or null
  size_t plane;
  uint32_t n_before;     // samples in sum_in
  uint32_t n_total;      // n_before + spp
};

// rh_render_adaptive's state and the buffers of one call: the selection, the sink of the list frame, the commit and the
// output.  State and output are in shard-compact pixel order; the list and the staging are indexed by list entry.
struct AdaptiveParams {
  uint32_t* counts;        // n_p, one plane
  double* sum;             // S: 3 planes (r, g, b) of `plane` doubles
  double* sumsq;           // Q: the same layout
  uint32_t* list;          // active pixels, ascending (select writes it)
  double* stage;           // 6 planes of `plane` doubles by entry: new S (r, g, b), new Q (r, g, b) (sink writes, commit reads)
  uint32_t* warp_masks;    // select: bit i of word w = pixel 32 w + i is active
  uint32_t* block_counts;  // select: active pixels per block, then their exclusive prefix
  uint32_t* n_active;      // select: the total
  unsigned long long* negative;  // output: pixels with a negative channel (RGB8 only)
  uint8_t* rgb;            // output, or null
  double* linear;          // output, or null
  size_t plane;            // pixels of the shard's rows: rows * width
  uint32_t width, height, shard_index, shard_count, band_height;  // the image and the shard's bands
  uint32_t spp, stream_spp, min_spp;
  double tt;               // threshold * threshold
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

// rh_render_features' outputs of one launch, indexed by the launch's pixels (pixel 0 = first pixel of ChunkParams::
// first_row); any may be null.
struct FeatureParams {
  double* albedo;   // double[pixel][3]
  double* normal;   // double[pixel][3]
  double* depth;    // double[pixel]
  uint32_t* hits;   // uint32[pixel]
  int2* hit_ids;    // int2[pixel][spp]
};

// Launchers (kernels.cu).  `count` selects the instrumented instantiation (box/tri counters); launch_trace runs the
// uninstrumented ray instantiation for P.offset_mode == kOffsetsRays, the pixel-list one when P.list.pixels is set and
// the uninstrumented views one when P.cams is set.
// (followed by a one-thread kernel that closes the pass's range of the hit queue, ChunkCtl::hit_start)
void launch_trace(const SceneView& S, const CameraParams& cam, const ChunkParams& P, bool count, int grid, void* stream);
// classify_kernel, then the walks of the hits it queued — refill: the per-lane-refill kernel (incoherent rays) instead of
// the pooled one (coherent rays).  Returns the number of launches.  P.groups set: the instantiations that also add the
// light-group terms (count must be false).
// `classified`: a cudaEvent_t recorded after the classify kernel (or null).
int launch_shadow(const SceneView& S, const ChunkParams& P, bool count, bool refill, int grid, void* stream, void* classified,
                  bool sphere_lights);
void launch_resolve(const ChunkParams& P, void* stream);
// rh_render_light_groups' sink, beside the resolve: each group's (and the remainder's) per-sample sums of the chunk,
// folded per pixel in sample order and times 1 / spp, to out + g * out_group_stride + (out_px0 + pixel) * 3, where
// pixel is chunk-local (padding rows: 0)
void launch_light_groups_resolve(const ChunkParams& P, double* out, size_t out_group_stride, size_t out_px0, void* stream);
// rh_render_views' end of a chunk instead of the resolve: resolve_kernel's RGB8 (P.rgb, may be null) and, to
// linear + (first_row * width + pixel) * 3 (may be null), the linear colours toIntC is applied to, with the padding
// rows of each view decided per view (0 in both outputs)
void launch_views_resolve(const ChunkParams& P, double* linear, void* stream);
// rh_trace_rays' end of a chunk instead of the resolve: the accumulators of its rays to colors (double[n][3], all rays)
void launch_store_colors(const ChunkParams& P, double* colors, void* stream);
// rh_render_accumulate's end of a chunk instead of the resolve: adds the chunk's samples to the running sums and writes
// RGB8 (P.rgb, may be null) and the linear colours (A.linear, may be null) of the new sums
void launch_accumulate_resolve(const ChunkParams& P, const AccumParams& A, void* stream);
// rh_render_adaptive: the selection (evaluates the rule per pixel, writes the active pixels to A.list in pixel order
// and their number to A.n_active); the sink of a list frame's chunk (the entries' new S and Q to A.stage); the commit of
// a completed frame (A.stage into the state, n_p += spp for the first n_active entries); the output (RGB8 and linear
// colours of every pixel, either optional)
void launch_adaptive_select(const AdaptiveParams& A, void* stream);
void launch_adaptive_fold(const ChunkParams& P, const AdaptiveParams& A, void* stream);
void launch_adaptive_commit(const AdaptiveParams& A, uint32_t n_active, void* stream);
void launch_adaptive_output(const AdaptiveParams& A, void* stream);
// rh_adaptive_state: three planes of `plane` doubles to double[plane][3]
void launch_adaptive_interleave(const double* planes, size_t plane, double* out, void* stream);
constexpr int kSelectBlock = 256;  // pixels per block of the selection
// query_closest_kernel / query_shadow_kernel: `grid` blocks of one SM each
void launch_query_closest(const SceneView& S, const QueryParams& Q, int grid, void* stream);
void launch_query_shadow(const SceneView& S, const QueryParams& Q, int grid, void* stream);
// feature_kernel (rh_render_features): the Q.n pixels of the rows of P (first_row, width, spp, offsets and the shard as
// for the render's pass 0; Q: claim cursor, deep stack, exact boxes) into F; `grid` blocks of one SM each
void launch_features(const SceneView& S, const CameraParams& cam, const ChunkParams& P, const QueryParams& Q, const FeatureParams& F,
                     int grid, void* stream);
void launch_deinterleave(const uint8_t* gathered, uint8_t* out, int width, int height, int shard_count, int band_height,
                         void* stream);
int configure_kernels();  // opt in to > 48 KB dynamic shared memory; returns a cudaError_t
int max_threads_per_launch(int n_sms);  // largest grid * block of the trace / shadow kernels (sizes the deep-stack scratch)
// setup_kernels.cu: the light-space tables of rh_scene_create, built on the device (return a cudaError_t)
int preload_setup_kernels();
int device_light_map(const double L[3], const rh_tri* d_tris, const uint32_t* d_slots, size_t n, int R, float* d_out, double min_empty,
                     unsigned long long* d_words, int* useful, double* empty_fraction, void* stream);
int device_lit_flags(const rh_tri* d_tris, const WideNode32* d_nodes, const double center[3], uint32_t root, const uint32_t* d_slots,
                     uint32_t n_slots, const rh_light* d_lights, uint32_t n_lights, uint32_t mask, uint32_t no_query, uint32_t mesh,
                     uint16_t* d_lit, unsigned long long* d_flagged, void* stream);
// micro-benchmarks
void launch_gather_bench(const double2* buf, uint64_t n_records, uint32_t loads_per_thread, double2* sink, int grid, int block,
                         void* stream);
void launch_stream_bench(const double2* buf, uint64_t n_elems, double2* sink, int grid, int block, void* stream);
void launch_dfma_bench(double* sink, int iters, int grid, int block, void* stream);

}  // namespace rhd
