/*
 * rayhs_b200.h — C ABI of the B200-native ray-casting path of RayHs.
 *
 * This header is the drop-in boundary.  The reference (oilandrust/rayhs) has no
 * FFI; the seam is `rayTrace :: Rendering -> Image` (src/RayHs.hs:161-166),
 * called from `main` (src/RayHs.hs:229-231).  A Haskell host binds these entry
 * points with `foreign import ccall safe` (see INTEGRATION.md) after flattening
 * its Scene (src/Scene.hs:8-10) at `buildGeometry` / `buildMaterial`
 * (src/Descriptors.hs:50-55, src/MaterialDescriptors.hs:34-45).
 *
 * Plain C only: pointers, sizes, POD structs.  No torch / C++ types.
 * All floating point data is IEEE double, like the reference (src/Vec.hs:29-31).
 * Every array pointer handed in must be 32-byte aligned when it is a node,
 * triangle or shading-record array (the library copies; the caller keeps
 * ownership of all host memory).
 *
 * Return convention: 0 = RH_OK, negative = error class; text through
 * rh_last_error() (thread-local).  The library never exits or aborts.
 */
#ifndef RAYHS_B200_H
#define RAYHS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RH_ABI_VERSION 2

/* ---- error classes -------------------------------------------------- */
enum {
  RH_OK = 0,
  RH_ERR_ARG = -1,      /* bad argument / malformed scene             */
  RH_ERR_CUDA = -2,     /* CUDA runtime failure (no GPU, launch, ...)  */
  RH_ERR_NCCL = -3,     /* NCCL failure                                */
  RH_ERR_OOM = -4,      /* host or device allocation failed            */
  RH_ERR_STATE = -5,    /* rh_init not called / called twice           */
  RH_ERR_IO = -6,       /* front end: file missing / parse error       */
  RH_ERR_OVERFLOW = -7  /* internal ray queue overflow (not recoverable by chunk split) */
};

/* ---- kinds ---------------------------------------------------------- */
/* Geometry.hs:62-63 (Plane | Sphere), KDTree.hs:59-61 (mesh tree)       */
enum { RH_OBJ_PLANE = 0, RH_OBJ_SPHERE = 1, RH_OBJ_MESH = 2 };
/* Material.hs:13-20                                                      */
enum {
  RH_MAT_MIRROR = 0, RH_MAT_DIFFUSE = 1, RH_MAT_PLASTIC = 2, RH_MAT_EMMIT = 3,
  RH_MAT_TRANSPARENT = 4, RH_MAT_SHOWNORMAL = 5, RH_MAT_SHOWUV = 6
};
/* ColorMap.hs:11-16                                                      */
enum { RH_CMAP_FLAT = 0, RH_CMAP_CHECKER = 1, RH_CMAP_TEXTURE = 2 };
/* Light.hs:8-10                                                          */
enum { RH_LIGHT_DIRECTIONAL = 0, RH_LIGHT_POINT = 1 };
/* Projection.hs:10-15                                                    */
enum { RH_PROJ_ORTHOGRAPHIC = 0, RH_PROJ_PERSPECTIVE = 1 };
/* sample-offset formats for rh_render (RayHs.hs:173-188)                 */
enum {
  RH_OFFSETS_NONE = 0,     /* 1 sample at the integer pixel coordinate (generatePixels, Image.hs:34-36) */
  RH_OFFSETS_F64 = 1,      /* double[w*h][spp][2], pixel-major, values already (x-0.5, y-0.5)          */
  RH_OFFSETS_F32 = 2,      /* float [w*h][spp][2], same order                                          */
  RH_OFFSETS_TILED_F64 = 3, /* double[tile*tile][spp][2], tile period given in rh_render_opts (declared deviation) */
  RH_OFFSETS_SPLITMIX64 = 4 /* `offsets` points at ONE uint64 seed (host memory): the kernel regenerates the stream of
                               rh_sample_offsets_f64(seed, ...) in place — SplitMix64 is counter-based, so value k of
                               the stream needs no predecessor — instead of reading 16 bytes per sample.  Same values,
                               same image; for hosts whose stream is this generator (SURVEY 8c/8f-4). */
};

#define RH_NO_NODE 0xFFFFFFFFu /* KDTree.hs:61 `Empty` */

/* ---- tables shared by the raw and the flat scene -------------------- */

/* Material.hs:13-20 + ColorMap.hs:11-16 folded into one 96-byte record.
 * Emmit: ce in color1.  Flat: colour in color1.  Checker: color1/color2/size
 * (ColorMap.hs:21-24: color1 where the product is negative).             */
typedef struct rh_material {
  int32_t kind;       /* RH_MAT_*                                        */
  int32_t cmap_kind;  /* RH_CMAP_* (diffuse / plastic only)              */
  double ior;
  double color1[3];
  double color2[3];
  double size;
  int32_t texture;    /* index into textures[] or -1                      */
  int32_t pad_;
  double pad2_[2];
} rh_material;

/* Light.hs:8-10.  vec = direction (un-normalised, Light.hs:14) or position. */
typedef struct rh_light {
  int32_t kind;  /* RH_LIGHT_* */
  int32_t pad_;
  double vec[3];
  double color[3];
  double radius;
} rh_light;

/* Bitmap.hs:13-15.  Texels are RGB triples of double (= byte/255, Bitmap.hs:28-29),
 * row-major, first PPM row first; `offset` counts texels into the shared texel array. */
typedef struct rh_texture {
  int32_t w, h;
  uint64_t offset;
} rh_texture;

/* Projection.hs:17-20 + 10-15 */
typedef struct rh_camera {
  double position[3];
  double target[3];
  double up[3];
  int32_t projection; /* RH_PROJ_* */
  int32_t pad_;
  double fovy;        /* perspective only                       */
  double proj_width;  /* parsed but unused by the reference     */
  double proj_height; /* (Projection.hs:34)                     */
  double near_;
} rh_camera;

/* ---- raw scene: what the front end holds BEFORE the tree build ------ */
/* One entry per Scene.shapes element (Scene.hs:8), in scene order.
 * plane : a = point, b = normal, c = tangent        (Geometry.hs:62)
 * sphere: a = center, b[0] = radius                 (Geometry.hs:63)
 * mesh  : vertices after Mesh.transform (Mesh.hs:89-101); positions/normals
 *         are double[n_verts][3], uvs double[n_verts][2], indices uint32[n_indices]
 *         grouped in threes (Mesh.hs:105-109).                                    */
typedef struct rh_raw_object {
  int32_t kind;
  int32_t material;
  double a[3], b[3], c[3];
  uint32_t n_verts;
  uint32_t n_indices;
  const double* positions;
  const double* normals;
  const double* uvs;
  const uint32_t* indices;
} rh_raw_object;

typedef struct rh_raw_scene {
  uint32_t n_objects;
  uint32_t n_materials;
  uint32_t n_lights;
  uint32_t n_textures;
  const rh_raw_object* objects;
  const rh_material* materials;
  const rh_light* lights;
  const rh_texture* textures;
  const double* texels; /* RGB triples */
  uint64_t n_texels;
} rh_raw_scene;

/* ---- flat scene: what crosses into the CUDA library ----------------- */

/* 64-byte tree node (KDTree.hs:59-61).  Inner: left/right = node indices or
 * RH_NO_NODE for `Empty`.  Leaf: left = first triangle, right = count.
 * leaf_index numbers the leaves of one mesh in left-to-right DFS order; it
 * carries the reference's tie rule (KDTree.hs:109-115) across any traversal order. */
typedef struct rh_node {
  double lo[3];
  double hi[3];
  uint32_t left;
  uint32_t right;
  uint32_t leaf_index;
  uint32_t is_leaf;
} rh_node;

/* 80-byte intersection record: p0, e1 = p1 - p0, e2 = p2 - p0 (Mesh.hs:70-71),
 * stored in leaf order.  tri_id = index in the mesh's `triangles` list (Mesh.hs:105-109). */
typedef struct rh_tri {
  double p0[3];
  double e1[3];
  double e2[3];
  uint32_t tri_id;
  uint32_t pad_;
} rh_tri;

/* 128-byte shading record, same order as rh_tri; read only for the winning hit
 * (Mesh.hs:81-82). */
typedef struct rh_tri_shade {
  double n0[3], n1[3], n2[3];
  double uv0[2], uv1[2], uv2[2];
  double pad_;
} rh_tri_shade;

typedef struct rh_object {
  int32_t kind;
  int32_t material;
  double a[3], b[3], c[3];
  uint32_t root;     /* mesh: root node index or RH_NO_NODE */
  uint32_t n_leaves; /* mesh: number of leaves              */
  uint32_t depth;    /* mesh: tree depth (root = 0)         */
  uint32_t pad_;
} rh_object;

typedef struct rh_scene_desc {
  uint32_t n_objects, n_materials, n_lights, n_textures;
  uint32_t n_nodes, n_tris;
  const rh_object* objects;
  const rh_material* materials;
  const rh_light* lights;
  const rh_texture* textures;
  const double* texels;
  uint64_t n_texels;
  const rh_node* nodes;          /* 32-byte aligned */
  const rh_tri* tris;            /* 32-byte aligned */
  const rh_tri_shade* tri_shade; /* 32-byte aligned */
} rh_scene_desc;

/* ---- render call ---------------------------------------------------- */

typedef struct rh_render_opts {
  int32_t width, height;  /* RayHs.hs:43-44 */
  int32_t max_depth;      /* RayHs.hs:45    */
  int32_t spp;            /* >= 1; RayHs.hs:175 hard-codes 64 */
  int32_t offset_mode;    /* RH_OFFSETS_*   */
  int32_t offset_tile;    /* period in pixels for RH_OFFSETS_TILED_F64 */
  const void* offsets;    /* host pointer, layout per offset_mode; may be NULL for RH_OFFSETS_NONE */
  /* image partition (SURVEY 8e): this call renders the rows whose band
   * (row / band_height) satisfies band % shard_count == shard_index.      */
  int32_t shard_index;    /* 0 .. shard_count-1 */
  int32_t shard_count;    /* >= 1               */
  int32_t band_height;    /* rows per band; 0 = library default */
  int32_t chunk_samples;  /* wavefront chunk size in pixel samples; 0 = default */
  int32_t flags;          /* RH_FLAG_* */
  int32_t n_peer_frames;  /* RH_FLAG_PEER_FRAMES: entries of peer_frames (= shard_count) */
  /* RH_FLAG_PEER_FRAMES (fused exchange, SURVEY 8e / 8f-4): host array of n_peer_frames DEVICE pointers, one full
   * [height][width][3] frame per shard of the job (this shard's own included), all addressable from this device
   * (rh_peer_alloc / rh_peer_open).  The resolve kernel stores every finished row straight into all of them, so after
   * all shards have returned (and one barrier) every GPU holds the complete frame: no all-gather, no de-interleave.
   * rgb_out may then be NULL. */
  void* const* peer_frames;
} rh_render_opts;

enum {
  RH_FLAG_HIT_IDS = 1,      /* also produce primary hit ids (see rh_render) */
  RH_FLAG_DEVICE_OUT = 2,   /* rgb_out / hit_ids_out are DEVICE pointers on the current device */
  RH_FLAG_DEVICE_OFFSETS = 4, /* offsets is a DEVICE pointer (already uploaded, full-frame layout) */
  RH_FLAG_COUNT = 8,         /* run the instrumented kernels: fills box_tests .. texel_fetches (slower) */
  RH_FLAG_PROFILE = 16,      /* bracket every launch with CUDA events: fills ms_trace / ms_shadow / ms_resolve */
  RH_FLAG_EXACT_BOXES = 32,  /* validation: the reference's double slab test at every box instead of the
                                conservative float cull (same image; see DESIGN.md) */
  /* Shadow-walk schedule (same image either way; DESIGN.md "Kernels").  Default: the library times both on the
   * first large frames of a scene (warm-up, pooled, refill) and keeps the faster one for that scene. */
  RH_FLAG_SHADOW_POOLED = 64, /* tree walks of the queued hits in warp-local rounds of 32, pooled per light (coherent rays) */
  RH_FLAG_SHADOW_SPLIT = 128, /* one queued hit per lane, per-lane refill when a ray ends (incoherent rays: triangle soups) */
  RH_FLAG_PEER_FRAMES = 256,  /* store the finished rows into rh_render_opts.peer_frames (see there) */
  /* 512 and 1024 selected the closest-hit schedule in ABI version 1; ignored since (one closest-hit kernel). */
  RH_FLAG_SHARD_OFFSETS = 4096, /* RH_OFFSETS_F64 / F32 with shard_count > 1: `offsets` holds only THIS shard's rows, in
                                   shard-compact order ([rh_shard_rows][width][spp][2]), instead of the full frame   */
  RH_FLAG_NO_LIGHT_MAPS = 2048 /* validation / A-B: shadow rays ignore the per-light cube maps of nearest possible
                                  occluder distance that rh_scene_create builds (same image; DESIGN.md "Light maps") */
};

/* Counts follow SURVEY 8d: one ray per closestIntersection (RayHs.hs:67) or
 * shadowIntersection (RayHs.hs:74) call. */
typedef struct rh_stats {
  uint64_t rays_primary;
  uint64_t rays_reflect;  /* specular children, RayHs.hs:99-104                */
  uint64_t rays_probe;    /* interior probe of Transparent, RayHs.hs:140        */
  uint64_t rays_exit;     /* transmitted child, RayHs.hs:143                    */
  uint64_t rays_shadow;   /* RayHs.hs:93                                        */
  uint64_t rays_shadow_culled; /* of rays_shadow: light at or below the shading horizon (l.n <= 0), Lambert term
                                  exactly 0, occlusion query skipped                                   */
  uint64_t shadow_tasks;  /* shaded Diffuse/Plastic hits (each folds over all lights) */
  uint64_t shadow_tasks_queued; /* of those: hits with a light whose shadow ray had to walk a tree (the others fold in the trace kernel) */
  uint64_t shadow_walk_pairs;   /* (hit, light) pairs that walked a tree                                  */
  uint64_t deep_stack_pushes;   /* RH_FLAG_COUNT only: traversal-stack entries beyond the shared-memory short stack */
  uint64_t queued_rays;   /* ray-queue entries written and read back (reflect + probe + exit) */
  /* RH_FLAG_COUNT only; the first six are the closest-hit (trace) kernel's */
  uint64_t box_tests;     /* child boxes tested                                  */
  uint64_t tri_tests;     /* triangle records tested                             */
  uint64_t prim_tests;    /* sphere / plane tests                                */
  uint64_t shade_fetches; /* winning triangle shading records read               */
  uint64_t texel_fetches;
  uint64_t node_visits;   /* 128-byte wide-node records read                     */
  uint64_t shadow_box_tests; /* the same four for the shadow (any-hit) kernel    */
  uint64_t shadow_tri_tests;
  uint64_t shadow_prim_tests;
  uint64_t shadow_node_visits;
  uint64_t node_visits_global;        /* node records fetched from global memory (not the staged top levels), counted once
                                         per warp instruction: lanes that visit the same node share one fetch          */
  uint64_t shadow_node_visits_global;
  uint64_t tri_records;               /* triangle records fetched, counted the same way                              */
  uint64_t shadow_tri_records;
  uint64_t upload_bytes;  /* sample-offset bytes copied host -> device           */
  double ms_total;        /* CUDA events around the whole call's device work (uploads and read-back included) */
  double ms_trace;        /* RH_FLAG_PROFILE only: closest-hit + shade kernels   */
  double ms_shadow;       /* RH_FLAG_PROFILE only: shadow any-hit kernels        */
  double ms_resolve;      /* RH_FLAG_PROFILE only: average + quantise            */
  uint32_t trace_launches;
  uint32_t shadow_launches;
  uint32_t kernel_launches;
  uint32_t chunks;
  uint32_t negative_channels; /* pixels with a channel whose toIntC is < 0 before the RGB8 clamp (App. A-Q2) */
  uint32_t queue_factor;      /* ray-queue capacity / chunk samples that was needed */
  uint32_t shadow_split;      /* 1: this frame used the per-lane-refill shadow kernel (RH_FLAG_SHADOW_SPLIT or auto) */
  uint32_t reserved_;
} rh_stats;

typedef struct rh_scene rh_scene; /* opaque; owns device copies */

/* Library / device bring-up.  device < 0: use the current CUDA device. */
int rh_init(int device);
void rh_shutdown(void);
const char* rh_last_error(void);
int rh_abi_version(void);
/* Number of kernels this library has launched since rh_init (for gpu_launches). */
uint64_t rh_launch_count(void);

/* Upload a flat scene.  Copies everything; host arrays may be freed after return. */
int rh_scene_create(const rh_scene_desc* desc, rh_scene** out);
void rh_scene_destroy(rh_scene* scene);
/* What rh_scene_create did: setup_ms3 = milliseconds for {cull / sphere trees + flattening, light-space tables (cube
 * maps, lit-triangle flags), uploads}; info4 = {object / material / light tables staged in shared memory, occluder
 * tables staged, deepest tree, deep-stack entries per thread}.  Either pointer may be NULL. */
int rh_scene_info(const rh_scene* scene, double* setup_ms3, int32_t* info4);
/* Bytes of the scene's gathered records in HBM: bytes5 = {cull-tree nodes (float boxes), triangle records, shading
 * records, texels, light-space tables (cube maps + lit flags)}.  bench.py bounds the HBM-compulsory share of the
 * gathers with it (a record has to cross HBM at most once per launch while the set fits the L2). */
int rh_scene_record_bytes(const rh_scene* scene, uint64_t* bytes5);
/* The light-space tables rh_scene_create built on the device, copied back (validation: tests compare them with the host
 * builders rh_light_map_build / rh_lit_triangles).  info4 = {cube maps, cells per face edge, lit flags present (0/1),
 * triangle slots}.  maps_out: maps * 6 * res * res floats; index_out: n_lights * 8 words (light * 8 + occluder mesh ->
 * map or 0xFFFFFFFF); lit_out: one uint16 per triangle slot.  Any pointer may be NULL. */
int rh_scene_light_tables(const rh_scene* scene, uint32_t* info4, float* maps_out, uint32_t* index_out, uint16_t* lit_out);

/* Replaces `rayTrace` (RayHs.hs:161-166) / `distributedRayTrace` (RayHs.hs:190-195).
 * rgb_out: RGB8, row-major.  For shard_count == 1 it is width*height*3 bytes.
 * For shard_count > 1 it is the COMPACT band buffer of this shard:
 * rh_shard_rows(...) rows of width*3 bytes (assemble with rh_assemble_bands or
 * an all-gather + rh_deinterleave_bands).
 * hit_ids_out (RH_FLAG_HIT_IDS): int32[rows*width*spp][2] = (object index,
 * triangle id | -1), (-1,-1) for a miss; may be NULL otherwise.
 * Quantisation = toIntC (Image.hs:54-55) clamped into 0..255.               */
int rh_render(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts,
              uint8_t* rgb_out, int32_t* hit_ids_out, rh_stats* stats);

/* ---- batched ray queries -------------------------------------------- */
/* Geometry.hs:39 Hit + the object and triangle that produced it (80 bytes). */
typedef struct rh_hit {
  double t;          /* +inf on a miss                                                                   */
  double p[3];       /* rayAt r t (Geometry.hs:29); 0 on a miss                                           */
  double n[3];       /* as the reference returns it: mesh normals interpolated, not renormalised (Mesh.hs:81) */
  double uv[2];      /* mesh: Mesh.hs:81-82, plane: Geometry.hs:70-79, sphere: Geometry.hs:96             */
  int32_t object;    /* scene index, -1 on a miss                                                         */
  int32_t tri;       /* tri_id (index in the mesh's triangles), -1 for planes / spheres / a miss          */
} rh_hit;

/* Replaces `closestIntersection` (RayHs.hs:67-71) for n caller-built rays: the closest hit over the object list, the
 * first object of the list winning a tie in t.  rays: double[n][6] = origin, direction (any length, zero components
 * allowed: the reference's arithmetic decides them).  hits_out: n records.  flags: RH_FLAG_DEVICE_OUT (rays and
 * hits_out are DEVICE pointers on the current device, 16-byte aligned) and RH_FLAG_EXACT_BOXES (validation: the
 * reference's double slab test at every box); any other bit is RH_ERR_ARG.  Host buffers are copied through device
 * scratch in bounded chunks, so any n works.  n == 0 is RH_OK; a null pointer with n > 0 is RH_ERR_ARG.  The call
 * returns when the results are written.  Sphere uv goes through CUDA's atan / acos (DESIGN.md §3: within a few ulp of
 * glibc's); every other value is bit-identical to the reference's. */
int rh_closest_intersection(const rh_scene* scene, const double* rays, uint64_t n, rh_hit* hits_out, int32_t flags);
/* Replaces `shadowIntersection` (RayHs.hs:74-87) towards light `light` (index into the scene's lights; out of range is
 * RH_ERR_ARG): occluded_out[i] = 1 when some non-emitter object (isOccluder, RayHs.hs:81-82) has a hit on ray i in
 * front of the light (inFrontOfLight, RayHs.hs:84-87: for a point light strictly nearer to the ray origin than the
 * light, for a directional light any hit), else 0.  The caller builds the ray, as accumDiffuse does with
 * `rayEps p ld` (RayHs.hs:93).  rays, flags, n and the buffers as for rh_closest_intersection (occluded_out needs no
 * alignment). */
int rh_shadow_intersection(const rh_scene* scene, uint32_t light, const double* rays, uint64_t n, uint8_t* occluded_out,
                           int32_t flags);

/* ---- radiance queries ----------------------------------------------- */
typedef struct rh_trace_opts {
  int32_t max_depth;   /* 0 .. 30, as rh_render_opts.max_depth                                                      */
  int32_t flags;       /* RH_FLAG_DEVICE_OUT | RH_FLAG_HIT_IDS | RH_FLAG_EXACT_BOXES | RH_FLAG_SHADOW_POOLED |
                          RH_FLAG_SHADOW_SPLIT | RH_FLAG_NO_LIGHT_MAPS; any other bit is RH_ERR_ARG                    */
  uint32_t chunk_rays; /* 0 = library default; else rays per wavefront chunk, in whole rows of 4096 rays (at least one) */
  uint32_t reserved_;
} rh_trace_opts;

/* Replaces `traceRay sc 0 max_depth r` (RayHs.hs:149-154) for n caller-built rays: the full Whitted radiance of each
 * ray (shadows, reflection, refraction, textures, the depth limit), as rh_render computes it for a camera ray.
 * `traceRay sc d maxD` depends on d and maxD only through maxD - d (specular: depth < maxDepth; Transparent:
 * d /= maxDepth), so a ray that starts at depth d is traced with max_depth = maxD - d.
 * rays: double[n][6] = origin, direction, as for rh_closest_intersection.
 * colors_out: double[n][3], the linear colour traceRay returns: not averaged, not clamped, no toIntC.  (rh_render's RGB8
 * of a camera ray at spp = 1 is toIntC of this value.)  Colours are sums of light terms in the wavefront's order, so
 * they may differ from the reference's in the last bits (DESIGN.md §3).
 * hit_ids_out (RH_FLAG_HIT_IDS): int32[n][2] = (object, tri) of the ray's own closest hit, as rh_render writes them.
 * RH_FLAG_DEVICE_OUT: rays, colors_out and hit_ids_out are DEVICE pointers on the current device (rays 16-byte aligned,
 * colours and ids 8-byte aligned); else host buffers, streamed through device scratch.  The shadow-walk flags force a
 * schedule; without them the call uses the one the scene's renders chose, else the pooled one.  The call never changes
 * what later rh_render calls of the scene do.  n == 0 is RH_OK; a null buffer with n > 0 is RH_ERR_ARG.
 * stats (optional): rays_primary = n, the other ray counts, queue_factor, shadow_split, chunks and ms_total as
 * rh_render fills them. */
int rh_trace_rays(const rh_scene* scene, const double* rays, uint64_t n, const rh_trace_opts* opts, double* colors_out,
                  int32_t* hit_ids_out, rh_stats* stats);

/* Rows owned by one shard (equal for all shards: bands are padded). */
int rh_shard_rows(int height, int shard_count, int band_height);
int rh_default_band_height(int height, int shard_count);

/* Device-side de-interleave after an all-gather: gathered = [shard][rows_per_shard][w][3]
 * (device), out = [h][w][3] (device).  Runs on the library stream and synchronises. */
int rh_deinterleave_bands(const uint8_t* gathered_dev, uint8_t* out_dev, int width, int height,
                          int shard_count, int band_height);

/* ---- several GPUs from ONE process (the Haskell host is one OS process; SURVEY 8e) ----
 * rh_multi_init opens devices 0 .. n_gpus-1 and enables peer access to device 0; rh_multi_scene_create replicates the
 * scene on all of them; rh_multi_render renders shard g of the interleaved row bands on GPU g (one host thread per GPU),
 * every resolve kernel storing its rows straight into ONE full frame on device 0 (peer stores over NVLink,
 * RH_FLAG_PEER_FRAMES), and copies that frame to rgb_out (host, width*height*3).  opts: shard_index / shard_count /
 * peer_frames are ignored (set by the library), RH_FLAG_HIT_IDS and the DEVICE flags are refused; host sample offsets
 * are uploaded per shard.  stats: ray counts summed over the shards, ms_total = the slowest shard.  Independent of
 * rh_init / rh_render (both contexts may exist). */
typedef struct rh_multi_scene rh_multi_scene;
int rh_multi_init(int n_gpus);
void rh_multi_shutdown(void);
int rh_multi_gpu_count(void);
int rh_multi_scene_create(const rh_scene_desc* desc, rh_multi_scene** out);
void rh_multi_scene_destroy(rh_multi_scene* scene);
int rh_multi_render(const rh_multi_scene* scene, const rh_camera* camera, const rh_render_opts* opts, uint8_t* rgb_out,
                    rh_stats* stats);

/* Frames shared between the processes of one job (one process per GPU): rh_peer_alloc allocates device memory on this
 * process's device and returns its CUDA IPC handle (64 bytes, to be sent to the other processes by any means);
 * rh_peer_open maps another process's allocation into this one (peer access over NVLink).  Close before the owner frees. */
#define RH_PEER_HANDLE_BYTES 64
int rh_peer_alloc(size_t bytes, void** dev_ptr_out, unsigned char handle_out[RH_PEER_HANDLE_BYTES]);
int rh_peer_open(const unsigned char handle[RH_PEER_HANDLE_BYTES], void** dev_ptr_out);
int rh_peer_close(void* dev_ptr);
int rh_peer_free(void* dev_ptr);

/* Micro-benchmarks used by bench.py for the roofline denominators (SURVEY 8d):
 * random 32-byte-aligned 64-byte gathers over `bytes` of device memory; returns GB/s. */
int rh_bench_gather(uint64_t bytes, int iters, double* gbs_out);
/* Coalesced 16-byte loads sweeping `bytes` of device memory `iters` times; with bytes below the L2 size this is the
 * L2 -> SM streaming rate (the denominator for the traversal kernels' lts__t_bytes); returns GB/s. */
int rh_bench_stream(uint64_t bytes, int iters, double* gbs_out);
/* Dependent DFMA chains on all SMs; returns TFLOP/s (2 flop per DFMA). */
int rh_bench_dfma(int iters, double* tflops_out);

/* ---- host-side front end (C++; stands in for the Haskell one) ------- */
/* KDTree.hs:68-90 build + flattening into the arrays above.              */
typedef struct rh_flat_scene rh_flat_scene; /* opaque; owns host arrays */
int rh_flatten(const rh_raw_scene* raw, rh_flat_scene** out);
const rh_scene_desc* rh_flat_desc(const rh_flat_scene* flat);
void rh_flat_destroy(rh_flat_scene* flat);

/* JSON.hs:22-141 + Descriptors.hs:39-55 + Mesh.hs:118-221 + Bitmap.hs:20-37. */
typedef struct rh_loaded rh_loaded; /* opaque; owns a raw scene + camera + size */
int rh_load_json(const char* json_path, const char* base_dir, rh_loaded** out);
/* binary pack of a loaded scene (fixtures for boxes without the data files) */
int rh_load_pack(const char* pack_path, rh_loaded** out);
int rh_save_pack(const rh_loaded* loaded, const char* pack_path);
/* SURVEY 8d config C5: n_tris random triangles + n_spheres spheres + floor, dragon.json camera/lights */
int rh_make_synthetic(uint64_t n_tris, uint32_t n_spheres, uint64_t seed, rh_loaded** out);
const rh_raw_scene* rh_loaded_raw(const rh_loaded* l);
const rh_camera* rh_loaded_camera(const rh_loaded* l);
void rh_loaded_size(const rh_loaded* l, int32_t* width, int32_t* height, int32_t* max_depth);
void rh_loaded_destroy(rh_loaded* l);

/* Sample offsets (RayHs.hs:173-188 shape; SplitMix64 stream, SURVEY 8d):
 * fills out[n_pixels][spp][2] with (x-0.5, y-0.5), x drawn before y. */
void rh_sample_offsets_f64(uint64_t seed, uint64_t n_pixels, int spp, double* out);
void rh_sample_offsets_f32(uint64_t seed, uint64_t n_pixels, int spp, float* out);
/* The same stream from pixel `first_pixel` on (SplitMix64 is counter-based): what a shard needs of a frame whose full
 * stream does not fit the host (configs[4]: 34 GB). */
void rh_sample_offsets_f64_at(uint64_t seed, uint64_t first_pixel, uint64_t n_pixels, int spp, double* out);

/* P3 writer byte-identical to Image.hs:60-75. */
int rh_write_ppm(const char* path, const uint8_t* rgb, int width, int height);

/* Validation hook (host only, no GPU): the cube map rh_scene_create builds for one point light and the triangles of
 * one mesh — per cell a lower bound of the distance from the light to every triangle that covers a direction of the
 * cell, +inf where none does.  The shadow kernels skip a mesh's tree walk when |p - L| is below the bound of the cell
 * of p - L: no triangle found there could be in front of the light (inFrontOfLight, RayHs.hs:84-87).  The reference
 * has no counterpart; the hook exists so that tests can check the map against brute-force shadow queries.
 * out: 6 * res * res floats, face 2k + (v[k] < 0) of the largest |v[k]|, rows of `res` cells, cell coordinates
 * (v[a], v[b]) / |v[k]| with (a, b) = (1,2), (0,2), (0,1) for k = 0, 1, 2.  *useful = 0 when the library would not
 * use the map (a triangle touches the light, or almost no cell is empty). */
int rh_light_map_build(const double light_pos[3], const rh_tri* tris, uint32_t n_tris, int res, float* out, int* useful,
                       double* empty_fraction);

/* Validation hook (host only): the "lit triangle" flags rh_scene_create computes per light and mesh.  out[i] = 1 when
 * no other triangle of tris[0 .. n_tris) can shadow any point of triangle i from the light: nothing else meets the hull
 * of the triangle and the light (RH_LIGHT_POINT; light_pos = its position) or the prism over the triangle along the
 * light's vector (RH_LIGHT_DIRECTIONAL; light_pos = that vector) above 1e-8 of the triangle's plane (a shadow ray
 * starts 1e-6 along the light direction and counts hits from t = 1e-6 on: Geometry.hs:36, Mesh.hs:76), and the light
 * is not grazing.  The shadow kernels skip the walk of a hit's own mesh for such a triangle.  Brute force here
 * (O(n^2)); the library walks the mesh's tree. */
int rh_lit_triangles(int light_kind, const double light_pos[3], const rh_tri* tris, uint32_t n_tris, uint8_t* out);
/* Host-only validation hook: the cull tree rh_scene_create builds over one mesh's triangles (binned SAH, at most 4
 * triangles per leaf, several host threads), refitted to exact padded boxes.  order_out[n_tris]: new slot -> given
 * triangle; nodes_out (room for 2 * n_tris records; leaves: left = first new slot, right = count; inner nodes: child
 * indices) ; *n_nodes_out, *depth_out.  Needs no GPU. */
int rh_cull_tree_build(const rh_tri* tris, uint32_t n_tris, uint32_t* order_out, rh_node* nodes_out, uint32_t* n_nodes_out,
                       uint32_t* depth_out);

#ifdef __cplusplus
}
#endif
#endif /* RAYHS_B200_H */
