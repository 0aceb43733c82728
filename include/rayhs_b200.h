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
/* Light.hs:8-10, and RH_LIGHT_SPHERE (a point light that emits from a ball; see rh_light) */
enum { RH_LIGHT_DIRECTIONAL = 0, RH_LIGHT_POINT = 1, RH_LIGHT_SPHERE = 2 };
/* Projection.hs:10-15, and RH_PROJ_THIN_LENS (a perspective camera with a circular thin lens; see rh_camera) */
enum { RH_PROJ_ORTHOGRAPHIC = 0, RH_PROJ_PERSPECTIVE = 1, RH_PROJ_THIN_LENS = 2 };
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

/* Light.hs:8-10.  vec = direction (un-normalised, Light.hs:14) or position.
 *
 * RH_LIGHT_SPHERE: a point light whose radius is also the radius r of the ball it emits from (the reference's falloff
 * c / (1 + d/r)^2 is the inverse-square law of such a ball): vec is the centre, color and radius mean what they mean
 * for RH_LIGHT_POINT.  radius must be finite and >= 0, else rh_scene_create and rh_scene_update return RH_ERR_ARG.
 * Each shading point samples one point of the ball per light, all in IEEE double in this order, without fused
 * multiply-add.  For the point p that accumDiffuse (RayHs.hs:89-97) receives and light index l:
 *   1. key = bits(p.x) ^ mix64(bits(p.y) ^ mix64(bits(p.z) ^ mix64(l))), with bits the IEEE-754 bit pattern, l as a
 *      uint64 and mix64 SplitMix64's output function (as for RH_PROJ_THIN_LENS, see rh_camera);
 *   2. for j = 0 .. 15: a = 2 U(key, 3j) - 1, b = 2 U(key, 3j + 1) - 1, c = 2 U(key, 3j + 2) - 1, with U(key, k) value k
 *      of the SplitMix64 stream seeded with key, as a double in [0, 1) (as for the lens); the first triple with
 *      ((a*a) + (b*b)) + (c*c) < 1 is taken; if none is, a = b = c = 0 (the centre);
 *   3. L' = (vec[0] + r*a, vec[1] + r*b, vec[2] + r*c);
 *   4. the pair (p, l) is then exactly an RH_LIGHT_POINT at L' with the same color and radius: lightAt (Light.hs:15-17)
 *      gives the direction and the falloff, the shadow ray is rayEps p ld, and inFrontOfLight (RayHs.hs:84-87) compares
 *      against L'.
 * The sample depends on p and l only, so every entry point that shades the same hit uses the same light point, and K
 * accumulate calls of s samples still equal one call of K*s samples.  The penumbra converges as the camera samples of
 * a pixel land on different points.  The points are a hash, not stratified: with RH_OFFSETS_NONE a hit point has one
 * fixed light point.  A radius of 0 gives RH_LIGHT_POINT's image.  rh_shadow_intersection takes caller-built rays and
 * compares a sphere light's hits against its centre, as for a point light. */
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

/* Projection.hs:17-20 + 10-15.
 *
 * RH_PROJ_THIN_LENS: position, target, up and fovy as for RH_PROJ_PERSPECTIVE; proj_width is the lens (aperture)
 * radius R >= 0 in world units, proj_height the focus distance F > 0 (the plane perpendicular to the view axis at
 * distance F from position is in focus); near_ is ignored.  R, F and fovy must be finite, else the render returns
 * RH_ERR_ARG.  The ray of image position (px, py) (the same doubles the pinhole ray is built from, col + ox and
 * row + oy), all in IEEE double in this order, without fused multiply-add:
 *   1. vx, vy, f, d = normalize(vx, vy, f), M = lookAt(position, target, up) and p = position, as RH_PROJ_PERSPECTIVE;
 *   2. R == 0: the perspective ray, bit for bit;
 *   3. lens sample: mix64(z) = SplitMix64's output function (z ^= z >> 30; z *= 0xBF58476D1CE4E5B9; z ^= z >> 27;
 *      z *= 0x94D049BB133111EB; z ^= z >> 31, mod 2^64); key = bits(px) ^ mix64(bits(py)) (IEEE-754 bit patterns);
 *      U(key, k) = value k of the SplitMix64 stream seeded with key, as a double in [0, 1) (RH_OFFSETS_SPLITMIX64's
 *      generator).  For j = 0 .. 15: a = 2 U(key, 2j) - 1, b = 2 U(key, 2j + 1) - 1; the first pair with
 *      (a*a) + (b*b) < 1 is taken; if none is, a = b = 0;
 *   4. in camera space L = (R*a, R*b, 0), s = F / d.z, P = (s*d.x, s*d.y, s*d.z), e = normalize(P - L);
 *   5. origin = apply(M, L) + p, direction = apply(M, e).
 * The lens point depends on the image position only, so every entry point that casts rh_render's camera rays casts
 * the same lens rays.  It is a hash, not stratified, whatever the pixel offsets are; with RH_OFFSETS_NONE a pixel has
 * one fixed lens point.  The reference's perspective camera never reads proj_width or proj_height, so the layout is
 * unchanged. */
typedef struct rh_camera {
  double position[3];
  double target[3];
  double up[3];
  int32_t projection; /* RH_PROJ_* */
  int32_t pad_;
  double fovy;        /* perspective and thin lens                              */
  double proj_width;  /* perspective: parsed but unused by the reference        */
  double proj_height; /* (Projection.hs:34); thin lens: R and F, see above      */
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

/* ---- scene updates --------------------------------------------------- */
/* What rh_scene_update rebuilt (24 bytes). */
typedef struct rh_update_info {
  uint32_t colours_only;      /* 1: nothing but light color / radius and material color1 / color2 / size changed  */
  uint32_t occluders_rebuilt; /* 1: the set of emitter objects changed (occluder tables and all light tables rebuilt) */
  uint32_t maps_rasterised;   /* cube maps built anew                                                                */
  uint32_t maps_kept;         /* cube maps carried over from the previous tables by device copies                    */
  uint64_t lit_queries;       /* (triangle, light) lit-triangle queries made                                          */
} rh_update_info;
/* Replaces the scene's material and light tables in place; the geometry (objects, their material indices, meshes,
 * textures) stays.  materials: n_materials entries, which must equal the scene's material count, or NULL (keep the
 * table); lights: n_lights entries (n_lights may differ from the scene's; 0 removes every light), or NULL (keep the
 * table, n_lights ignored).  Entries are checked as rh_scene_create checks them.  After RH_OK every call on the scene
 * behaves as on rh_scene_create of the same description with the new tables (set-up times aside), including
 * rh_scene_info's info4, rh_scene_light_tables and rh_scene_record_bytes.  Only what the edit touches is rebuilt: an
 * update of colours only (light color / radius, material color1 / color2 / size) uploads the two tables; one that turns
 * an object into an emitter or back rebuilds the occluder tables and every light table; any other rebuilds the cube
 * maps of the lights that are new or moved (kind or vec) and their lit-triangle bits, and carries the other maps over.
 * Beyond a colours-only update the scene's learned state (shadow schedule, queue factor, row costs) starts over as a
 * fresh scene's.  An update that changes no byte is a no-op.  Every other update makes rh_render_accumulate and
 * rh_render_adaptive refuse a state whose view was fixed before it (reset it first).  The call returns when the device
 * work is done and must not overlap another call on the scene.  On failure (argument, RH_ERR_OOM, RH_ERR_CUDA) the
 * scene is unchanged and usable: the new tables are built beside the old ones and swapped in at the end, so the peak
 * memory is both sets.  info (optional): what was rebuilt. */
int rh_scene_update(rh_scene* scene, const rh_material* materials, uint32_t n_materials, const rh_light* lights,
                    uint32_t n_lights, rh_update_info* info);

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

/* ---- progressive rendering ------------------------------------------ */
/* Running per-pixel sums of the sample colours of one frame (or of one shard's rows of it: the rows rh_render's
 * shard_index / shard_count / band_height select, band_height 0 resolved as rh_render resolves it), kept on the device
 * between calls.  2 x 24 bytes per pixel of those rows.  stream_spp: samples per pixel of the SplitMix64 stream that
 * RH_OFFSETS_SPLITMIX64 calls draw from (0: such calls are refused).  Needs rh_init (else RH_ERR_STATE). */
typedef struct rh_accum rh_accum; /* opaque */
int rh_accum_create(int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                    rh_accum** out);
/* Back to 0 samples; the next call may use another scene, camera or max_depth. */
int rh_accum_reset(rh_accum* acc);
void rh_accum_destroy(rh_accum* acc);
/* Traces opts->spp new samples per pixel exactly as rh_render would, adds them to the accumulator's sums in sample
 * order (continuing `foldl (+) black`, RayHs.hs:169-171: K calls of s samples leave the sums of one call of K*s
 * samples), so that the accumulator's count N grows by spp, then writes what the caller asked for:
 *   rgb_out    RGB8 = toIntC((1/N) sum), clamped as rh_render clamps it;
 *   linear_out double[rows][width][3] = (1/N) sum, the value toIntC is applied to (not clamped).
 * Either may be NULL (neither: the call only accumulates).  Layouts are shard-compact, as for rh_render.
 * Offsets: RH_OFFSETS_NONE / F64 / F32 / TILED_F64 give THIS call's samples ([pixels][spp][2] or the [tile^2][spp][2]
 * tile), host or device, RH_FLAG_SHARD_OFFSETS as for rh_render; so slicing one stream [pixels][S][2] into
 * consecutive sample ranges reproduces the one-shot S-sample frame.  RH_OFFSETS_SPLITMIX64 draws values 2g and 2g + 1
 * with g = pixel * stream_spp + N_before + s: the stream of rh_sample_offsets_f64(seed, n_pixels, stream_spp, ...);
 * N_before + spp > stream_spp is RH_ERR_ARG.  hit_ids_out (RH_FLAG_HIT_IDS): this call's samples, int32[rows][width]
 * [spp][2].  RH_FLAG_DEVICE_OUT applies to all three outputs (linear_out 8-byte aligned).  The other flags behave as
 * in rh_render and may change from call to call; RH_FLAG_PEER_FRAMES is refused.
 * The first call after create or reset records the scene, the camera bytes and max_depth; a later call with others is
 * RH_ERR_ARG (reset first), and so is a call after an rh_scene_update of that scene that changed bytes.  opts must
 * match the accumulator's size and shard.  A call that fails (argument, CUDA or
 * RH_ERR_OVERFLOW) leaves the sums and N unchanged.  For the scene's learned state (shadow schedule, queue factor, row
 * costs) the call is a render.  stats: this call's samples; negative_channels counts its RGB8 output. */
int rh_render_accumulate(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, rh_accum* acc,
                         uint8_t* rgb_out, double* linear_out, int32_t* hit_ids_out, rh_stats* stats);

/* ---- adaptive sampling ---------------------------------------------- */
/* Progressive rendering that traces new samples only for the pixels whose standard error is still above a threshold,
 * each pixel continuing its own slice of the SplitMix64 stream.  State per pixel p of the shard's rows (shard-compact
 * order, rows selected as for rh_accum_create), kept on the device between calls (52 bytes per pixel, plus 52 bytes
 * per pixel of list and staging space):
 *   n_p      samples so far;
 *   S_p[c]   foldl (+) 0 of the sample colours in sample order (the sum rh_render_accumulate keeps);
 *   Q_p[c]   foldl (+) 0 of x * x, each square rounded and then added, in sample order.
 * stream_spp >= 1: samples per pixel of the stream (no pixel goes past it).  Needs rh_init (else RH_ERR_STATE). */
typedef struct rh_adaptive rh_adaptive; /* opaque */
typedef struct rh_adaptive_opts {
  double threshold;   /* >= 0, linear colour units: bound on each channel's standard error of the mean */
  uint32_t min_spp;   /* >= 2: pixels with fewer samples are always traced                            */
  uint32_t reserved_; /* must be 0                                                                     */
} rh_adaptive_opts;   /* 16 bytes */
int rh_adaptive_create(int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                       rh_adaptive** out);
/* All counts and sums back to 0; the next call may use another scene, camera or max_depth. */
int rh_adaptive_reset(rh_adaptive* ad);
void rh_adaptive_destroy(rh_adaptive* ad); /* NULL is a no-op */
/* One round of adaptive sampling.  opts->offset_mode must be RH_OFFSETS_SPLITMIX64 (opts->offsets: the seed); sample s of
 * this call for pixel p draws values 2g and 2g + 1 with g = pixel * stream_spp + n_p + s (pixel: full-image index), the
 * index rh_render_accumulate uses with the pixel's own count in place of N.  So a pixel that ends with n samples holds
 * exactly the sums, and gives exactly the bytes, of an n-sample rh_render_accumulate (or rh_render) of that stream.
 * Selection, on the state before the call, in this operation order (IEEE double, no fused multiply-add):
 *   tt = threshold * threshold;  nn = (double)n * (double)(n - 1);  d_c = Q_c - S_c * (S_c / n)
 *   p is active  iff  n + spp <= stream_spp  and  (n < min_spp  or  d_c > tt * nn for some channel c).
 * (A NaN d_c does not keep a pixel active; a negative d_c from cancellation counts as converged.)  Each active pixel gets
 * opts->spp new samples; the others are not traced and keep their state.  *n_active_out (optional): active pixels.  A
 * call with no active pixel traces nothing, returns RH_OK and still writes the outputs, which cover every pixel of the
 * shard's rows, shard-compact:
 *   rgb_out    RGB8 = toIntC((1/n_p) S_p), clamped as rh_render clamps it (0 for a pixel with no sample yet);
 *   linear_out double[rows][width][3] = (1/n_p) S_p (0 for a pixel with no sample yet).
 * Either may be NULL.  RH_FLAG_DEVICE_OUT applies to both (linear_out 8-byte aligned).  RH_FLAG_HIT_IDS,
 * RH_FLAG_PEER_FRAMES, RH_FLAG_SHARD_OFFSETS and RH_FLAG_DEVICE_OFFSETS are RH_ERR_ARG; RH_FLAG_EXACT_BOXES,
 * RH_FLAG_NO_LIGHT_MAPS, the shadow-schedule flags, RH_FLAG_COUNT, RH_FLAG_PROFILE and chunk_samples behave as in
 * rh_render (chunk_samples counts the samples of the active pixels).  threshold and min_spp may change from call to
 * call.  The first call after create or reset records the scene, the camera bytes and max_depth; a later call with
 * others is RH_ERR_ARG (reset first), and so is a call after an rh_scene_update of that scene that changed bytes.
 * opts must match the state's size and shard.  A call that fails (argument, CUDA
 * or RH_ERR_OVERFLOW) leaves every n_p, S_p and Q_p unchanged; a queue-overflow retry inside the call counts no sample
 * twice.  The call uses the scene's decided shadow schedule and queue factor (else the pooled schedule and factor 2)
 * and changes neither them nor the row costs, as rh_trace_rays does.  stats: rays_primary = n_active * spp, the other
 * ray counts this call's; chunks, queue_factor, shadow_split and ms_total (the whole call) as in rh_render;
 * negative_channels counts the RGB8 output; RH_FLAG_PROFILE: ms_resolve also holds the selection, commit and output
 * kernels. */
int rh_render_adaptive(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts,
                       const rh_adaptive_opts* aopts, rh_adaptive* ad, uint8_t* rgb_out, double* linear_out,
                       uint64_t* n_active_out, rh_stats* stats);
/* Copies the state out: counts_out uint32[rows][width] = n_p, sums_out / sumsq_out double[rows][width][3] = S_p / Q_p.
 * Any pointer may be NULL.  flags: 0 (host buffers) or RH_FLAG_DEVICE_OUT (device buffers, the doubles 8-byte aligned). */
int rh_adaptive_state(const rh_adaptive* ad, uint32_t* counts_out, double* sums_out, double* sumsq_out, int32_t flags);

/* ---- feature buffers ------------------------------------------------ */
/* Per-pixel buffers of the camera rays' first hits, for denoisers (albedo, normal) and compositing (depth, coverage).
 * Layouts are shard-compact rows, as rh_render's rgb_out; any pointer may be NULL. */
typedef struct rh_features {
  double* albedo;        /* double[rows][width][3], or NULL                                        */
  double* normal;        /* double[rows][width][3], or NULL                                        */
  double* depth;         /* double[rows][width], or NULL                                           */
  uint32_t* hits;        /* uint32[rows][width], or NULL                                           */
  uint32_t stream_spp;   /* RH_OFFSETS_SPLITMIX64 only: samples per pixel of the stream; 0 = opts->spp */
  uint32_t stream_base;  /* RH_OFFSETS_SPLITMIX64 only: the pixel's first stream sample this call uses */
} rh_features;           /* 40 bytes */
/* Casts exactly the camera rays rh_render casts for the same scene, camera and opts (offset modes, device and shard
 * offsets, shard and band selection), without shading them.  RH_OFFSETS_SPLITMIX64: sample s of pixel p uses stream
 * index g = p * stream_spp + stream_base + s, the index rh_render_accumulate uses; stream_base + spp > stream_spp, or a
 * nonzero stream field with another offset mode, is RH_ERR_ARG.  Each ray's closest hit is the one rh_render's
 * RH_FLAG_HIT_IDS reports.  Per sample s: t_s and n_s as rh_closest_intersection's rh_hit gives them (mesh normals
 * interpolated, not renormalised); the albedo a_s is colorAt of the material at the hit's uv for Diffuse and Plastic
 * (the colour the render shades with, textures included), color1 for Emmit, n_s for ShowNormal, (u, v, 0) for ShowUV and
 * (1, 1, 1) for Mirror and Transparent; a miss has a_s = n_s = 0 and no t_s.  Per pixel, with foldl (+) 0 over the
 * samples in sample order, per channel, in IEEE double without fused multiply-add, and inv = 1.0 / spp:
 *   albedo = inv * sum a_s;   normal = inv * sum n_s (not renormalised: a half-covered pixel has a shorter normal);
 *   hits = h, the samples that hit;   depth = (1.0 / h) * (sum of t_s over the hitting samples), +inf when h = 0.
 * Padding rows of the last band are pixels without hits.  hit_ids_out (RH_FLAG_HIT_IDS): int32[rows][width][spp][2] as
 * rh_render writes it.  RH_FLAG_DEVICE_OUT: every output is a device pointer on the current device, 8-byte aligned;
 * else host buffers, written through device scratch in bounded chunks (so are host offsets).  RH_FLAG_DEVICE_OFFSETS,
 * RH_FLAG_SHARD_OFFSETS and RH_FLAG_EXACT_BOXES behave as in rh_render; the shadow-schedule flags, RH_FLAG_NO_LIGHT_MAPS,
 * chunk_samples and max_depth (checked as in rh_render) have no effect, so a render's opts can be passed unchanged;
 * RH_FLAG_PEER_FRAMES, RH_FLAG_COUNT and RH_FLAG_PROFILE are RH_ERR_ARG, and so is a call that asks for no output.  The
 * call neither reads nor changes the scene's learned state (shadow schedule, queue factor, row costs), reflects the
 * scene's latest rh_scene_update, and returns when the outputs are written.  stats: rays_primary (the samples traced),
 * chunks, kernel_launches and ms_total; every other field 0. */
int rh_render_features(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, const rh_features* features,
                       int32_t* hit_ids_out, rh_stats* stats);

/* ---- light groups --------------------------------------------------- */
/* One linear image per group of lights, plus one of everything else (the remainder), for relighting in compositing:
 * scaling group g's image by k_g is scaling those lights' colours by k_g. */
typedef struct rh_light_groups {
  const uint8_t* group_of_light; /* n_lights entries (host memory), each < n_groups; may be NULL for a scene without lights */
  uint32_t n_groups;             /* 1 .. 16                                                                 */
  uint32_t reserved_;            /* must be 0                                                               */
  double* out;                   /* double[n_groups + 1][rows][width][3], shard-compact rows; last = remainder */
} rh_light_groups;               /* 24 bytes */
/* Renders exactly as rh_render does for the same scene, camera and opts (the same rays, every offset mode, device and
 * shard offsets, shard and band selection) and also writes the light groups.  Per shaded hit with weight w:
 *   group g:   w * foldl (+) black [diffuse_l | l <- lights in order, group_of_light[l] == g, l visible], added only when
 *              one of g's lights is visible; culled (l.n <= 0) and occluded pairs add nothing, as in the render;
 *   remainder: Diffuse's ambient term w * 0.2 cd, and every finished term (Emmit, ShowNormal, ShowUV, and the NaN terms of
 *              tainted rays).
 * A sample's group sums add these terms in pass order; a pixel is foldl (+) 0 of its samples in sample order, times
 * inv = 1.0 / spp, in IEEE double without fused multiply-add.  Padding rows of the last band are 0.  So the groups and
 * the remainder add up to the render's linear colour only up to rounding, group g is linear in its lights' colours
 * only up to rounding, and Transparent forks wobble in the last bit as everywhere else; a group without lights is 0.
 * rgb_out (optional: may be NULL) receives rh_render's bytes and hit_ids_out (RH_FLAG_HIT_IDS) its ids.
 * RH_FLAG_DEVICE_OUT covers all outputs (out 8-byte aligned); host outputs go through device scratch in bounded chunks.
 * RH_FLAG_PEER_FRAMES and RH_FLAG_COUNT are RH_ERR_ARG, and so is a scene with more than 32 lights; RH_FLAG_EXACT_BOXES,
 * RH_FLAG_NO_LIGHT_MAPS, the shadow-schedule flags, RH_FLAG_PROFILE and chunk_samples behave as in rh_render.  The call
 * uses the scene's decided shadow schedule and queue factor (else pooled and 2) and changes neither of them nor the row
 * costs.  stats as rh_render fills them (negative_channels counts rgb_out).  A call refused for its arguments writes
 * nothing. */
int rh_render_light_groups(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts,
                           const rh_light_groups* groups, uint8_t* rgb_out, int32_t* hit_ids_out, rh_stats* stats);

/* ---- camera batches ------------------------------------------------- */
/* Many views of one scene in one wavefront (cube-map faces, stereo pairs and rigs, thumbnails, multi-view image sets). */
typedef struct rh_views {
  const rh_camera* cameras; /* n_views cameras (host memory)                                                     */
  uint32_t n_views;         /* 1 .. 65536                                                                        */
  uint32_t reserved_;       /* must be 0                                                                         */
  const uint64_t* seeds;    /* RH_OFFSETS_SPLITMIX64 only: n_views seeds (host), or NULL = every view uses
                               *opts->offsets; non-NULL with another offset mode is RH_ERR_ARG                     */
} rh_views;                 /* 24 bytes */
/* View v is exactly rh_render(scene, &cameras[v], opts'), where opts' is opts with *offsets = seeds[v] when seeds is
 * given: the same rays (every offset mode, host, device and shard-compact offsets, shard and band selection), bytes,
 * hit ids and ray counts, up to the 1-LSB wobble of Transparent forks that two rh_render calls already show.  All views
 * share width, height, spp, max_depth and the offsets; the cameras may differ in anything, projection included.
 * Outputs are view-major over shard-compact rows (rows = rh_shard_rows(height, shard_count, band_height)):
 *   rgb_out      uint8[n_views][rows][width][3], as rh_render writes it (padding rows of the last band: 0);
 *   linear_out   double[n_views][rows][width][3], the colour toIntC is applied to: the linear_out a single
 *                rh_render_accumulate call on a freshly created accumulator writes for that view (padding rows: 0);
 *   hit_ids_out  (RH_FLAG_HIT_IDS) int32[n_views][rows][width][spp][2].
 * rgb_out and linear_out are each optional (NULL), but not both.  RH_FLAG_DEVICE_OUT covers all three outputs
 * (linear_out 8-byte aligned).  RH_FLAG_DEVICE_OFFSETS, RH_FLAG_SHARD_OFFSETS, RH_FLAG_EXACT_BOXES,
 * RH_FLAG_NO_LIGHT_MAPS, the shadow-schedule flags, RH_FLAG_PROFILE and chunk_samples behave as in rh_render; host
 * per-pixel offsets (F64 / F32) are uploaded once per call to device scratch (RH_ERR_OOM when they do not fit).
 * RH_ERR_ARG: RH_FLAG_PEER_FRAMES, RH_FLAG_COUNT, n_views 0 or above 65536, a null cameras, a nonzero reserved_, a
 * camera with an unknown projection (the message names the view), seeds with an offset mode other than SplitMix64, and
 * rh_render's own checks.  The call uses the scene's decided shadow schedule (else pooled).  Its queues start at the
 * larger of the scene's queue factor (else 2) and the factor the scene's last views call needed, reduced while the
 * queues would outgrow the memory the library plans for a chunk, and grow by the overflow retry; the call remembers
 * its own factor for the next views call.  It changes neither the schedule, nor the queue factor renders use, nor the
 * row costs.  stats: ray counts summed over the views (rays_primary = n_views times one
 * view's), negative_channels of rgb_out, and chunks, queue_factor, shadow_split and ms_total as rh_render fills
 * them (ms_total includes the upload of the camera table, the seeds and host offsets).  A call refused for its arguments writes nothing. */
int rh_render_views(const rh_scene* scene, const rh_views* views, const rh_render_opts* opts, uint8_t* rgb_out,
                    double* linear_out, int32_t* hit_ids_out, rh_stats* stats);

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
/* rh_scene_update on every replica: all are prepared before any is swapped in, so the update takes on every GPU or on
 * none.  info: replica 0's. */
int rh_multi_scene_update(rh_multi_scene* scene, const rh_material* materials, uint32_t n_materials, const rh_light* lights,
                          uint32_t n_lights, rh_update_info* info);
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
