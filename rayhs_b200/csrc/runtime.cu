// runtime.cu — host side of librayhs_b200: device bring-up, scene upload, and the wavefront
// schedule behind rh_render (the replacement for `rayTrace`, RayHs.hs:161-166, and
// `distributedRayTrace`, RayHs.hs:190-195).  C ABI in include/rayhs_b200.h.
//
// Schedule per chunk of rows (all launches asynchronous on one stream, no host round trip
// between passes — queue lengths stay in device memory and the kernels are persistent):
//   pass 0      trace_kernel(primary)  -> shadow tasks, child rays
//               shadow_kernel
//   pass 1..2D  trace_kernel(queued)   -> shadow tasks, child rays     (D = maxDepth; a Transparent
//               shadow_kernel                                            hit adds one probe pass per level)
//   resolve_kernel -> RGB8
// Sample offsets for chunk k+1 are uploaded on a second stream while chunk k is traced.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <initializer_list>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.h"
#include "device_types.cuh"
#include "light_geom.h"
#include "render_plan.h"
#include "scene_update.h"

namespace rh {
static thread_local std::string g_err;
int set_error(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
}  // namespace rh

using namespace rhd;

namespace {

std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_contexts{0};  // device contexts opened so far (names each one: an address can be reused)

#define RH_CUDA(expr)                                                                                     \
  do {                                                                                                    \
    cudaError_t e_ = (expr);                                                                              \
    if (e_ != cudaSuccess) {                                                                              \
      int code_ = (e_ == cudaErrorMemoryAllocation) ? RH_ERR_OOM : RH_ERR_CUDA;                           \
      return rh::set_error(code_, std::string(#expr) + ": " + cudaGetErrorString(e_));                    \
    }                                                                                                     \
  } while (0)

// A growable device buffer.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int reserve(size_t n) {
    if (n <= bytes) return RH_OK;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    RH_CUDA(cudaMalloc(&p, n));
    bytes = n;
    return RH_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
};

// Everything the library owns on one GPU.
struct Device {
  int dev = -1;
  uint64_t context = 0;
  int n_sms = 0;
  size_t total_mem = 0;
  cudaStream_t stream = nullptr;       // kernels (lane 0)
  cudaStream_t stream2 = nullptr;      // kernels of every second chunk when two chunks are in flight (lane 1)
  cudaStream_t copy_stream = nullptr;  // sample-offset uploads
  // Per lane: the stream of the shadow kernels (classify + walks) when a chunk's passes are pipelined — the trace kernel of
  // pass k + 1 runs beside the shadow kernels of pass k — with an event per pass (trace done) and one per chunk (shadows done)
  cudaStream_t shadow_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_trace[2][kMaxPasses + 2] = {}, ev_classified[2][kMaxPasses + 2] = {}, ev_shadows[2] = {nullptr, nullptr};
  cudaEvent_t ev_lane = nullptr;
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
  std::vector<cudaEvent_t> ev_up, ev_done;  // one pair per slot of the offset upload ring
  // per-lane scratch: a chunk's accumulators and queues
  struct Scratch {
    DevBuf accum, rayq[2], rayq_fill[2], hitq, hitq_words, shq, shq_words, deep, deep_shadow;
    DevBuf groups, group_out;  // rh_render_light_groups: per-sample group sums; one chunk of host output
  } lane[2];
  DevBuf ctl, counters, offsets, rgb, ids, linear;
  DevBuf query;  // ray queries: claim cursor, then (host buffers) one chunk of rays and of results
  DevBuf views;  // rh_render_views: the camera table, then the seeds
  void* pinned = nullptr;  // ctl + counters read-back
  size_t pinned_bytes = 0;
  int max_threads = 0;  // largest grid * block of the traversal kernels (one block per SM)
  std::vector<cudaEvent_t> prof_events;

  int open(int device) {
    dev = device;
    context = ++g_contexts;
    RH_CUDA(cudaSetDevice(dev));
    cudaDeviceProp prop;
    RH_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10)
      return rh::set_error(RH_ERR_CUDA, std::string("rayhs_b200 needs an sm_100 device, found ") + prop.name);
    n_sms = prop.multiProcessorCount;
    total_mem = prop.totalGlobalMem;
    RH_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    RH_CUDA(cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
    RH_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    for (int l = 0; l < 2; l++) {
      RH_CUDA(cudaStreamCreateWithFlags(&shadow_stream[l], cudaStreamNonBlocking));
      RH_CUDA(cudaEventCreateWithFlags(&ev_shadows[l], cudaEventDisableTiming));
      for (cudaEvent_t& e : ev_trace[l]) RH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      for (cudaEvent_t& e : ev_classified[l]) RH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    RH_CUDA(cudaEventCreateWithFlags(&ev_lane, cudaEventDisableTiming));
    RH_CUDA(cudaEventCreate(&ev_begin));
    RH_CUDA(cudaEventCreate(&ev_end));
    RH_CUDA((cudaError_t)configure_kernels());
    RH_CUDA((cudaError_t)preload_setup_kernels());
    max_threads = max_threads_per_launch(n_sms);
    RH_CUDA(cudaGetLastError());
    return RH_OK;
  }
  void close() {
    if (dev < 0) return;
    cudaSetDevice(dev);
    for (Scratch& sc : lane)
      for (DevBuf* b : {&sc.accum, &sc.rayq[0], &sc.rayq[1], &sc.rayq_fill[0], &sc.rayq_fill[1], &sc.hitq, &sc.hitq_words, &sc.shq, &sc.shq_words, &sc.deep, &sc.deep_shadow,
                        &sc.groups, &sc.group_out})
        b->release();
    for (int l = 0; l < 2; l++) {
      if (shadow_stream[l]) cudaStreamDestroy(shadow_stream[l]);
      shadow_stream[l] = nullptr;
      if (ev_shadows[l]) cudaEventDestroy(ev_shadows[l]);
      ev_shadows[l] = nullptr;
      for (cudaEvent_t& e : ev_trace[l]) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
      }
      for (cudaEvent_t& e : ev_classified[l]) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
      }
    }
    for (DevBuf* b : {&ctl, &counters, &offsets, &rgb, &ids, &linear, &query, &views})
      b->release();
    if (pinned) cudaFreeHost(pinned);
    pinned = nullptr;
    pinned_bytes = 0;
    for (cudaEvent_t e : prof_events) cudaEventDestroy(e);
    prof_events.clear();
    for (cudaEvent_t e : {ev_begin, ev_end, ev_lane})
      if (e) cudaEventDestroy(e);
    if (stream2) cudaStreamDestroy(stream2);
    stream2 = nullptr;
    for (cudaEvent_t e : ev_up) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_done) cudaEventDestroy(e);
    ev_up.clear();
    ev_done.clear();
    if (stream) cudaStreamDestroy(stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    stream = copy_stream = nullptr;
    dev = -1;
  }
};

std::mutex g_mu;
std::unique_ptr<Device> g_dev;  // rh_init

}  // namespace

struct rh_scene {
  Device* device = nullptr;
  DevBuf wide, wide32, tris, shade, objects, materials, lights, textures, texels, lin_objs, sphere_refs, occ_planes, occ_spheres, occ_meshes, exact_index, light_maps, light_map_index, lit_flags;
  SceneView view{};
  uint32_t max_tree_depth = 0;
  uint32_t deep_entries = 1;     // per-thread entries of the deep-stack scratch this scene's walks can need
  bool refill_possible = true;   // the per-lane-refill shadow kernel stacks every tree root: not with hundreds of meshes
  bool has_transparent = false;  // some material is Transparent (Material.hs:18): frames need the probe passes
  bool has_sphere_lights = false;  // some light is RH_LIGHT_SPHERE: frames run the shadow kernels that sample the balls
  // Shadow-walk schedule of this scene: 0 = undecided, 1 = pooled, 2 = per-lane refill.  Decided by timing one large
  // frame with each (render_on); frames too small to time use the pooled kernel and do not count, and after
  // kTuneGiveUp of those the scene stays pooled.
  mutable int shadow_mode = 0;
  mutable int tune_frames = 0, tune_small_frames = 0;
  mutable double tune_ns_per_pair[2] = {0, 0};
  // set-up times of rh_scene_create (milliseconds)
  double ms_trees = 0, ms_light_tables = 0, ms_upload = 0;
  uint32_t n_light_maps = 0;     // cube maps in light_maps
  // Per-chunk kernel time of the last frame that streamed its sample offsets from the host (key: the chunk plan).
  // The next such frame processes its chunks in descending cost per sample, so that the uploads of the cheap chunks
  // hide behind the kernels of the expensive ones instead of the other way round.
  mutable std::vector<int> cost_key;      // {W, H, spp, shards, shard, band height} the row costs belong to
  mutable std::vector<float> row_cost;    // kernel ms per local row (its chunk's time / its chunk's rows)
  mutable uint32_t queue_factor = 2;          // the queue capacity factor the scene's last frame needed
  mutable uint32_t views_queue_factor = 2;    // ... and its last rh_render_views frame (which leaves the one above alone)
  mutable bool stream_compute_bound = false;  // ... and in that frame the kernels, not the upload, finished last
  // What derive_tables needs to rebuild the material- and light-derived tables for rh_scene_update (DESIGN.md "Scene
  // updates"), on the host: the object records, the linear object list, the sphere-tree root, both tree depths, the
  // texture table, the current material and light tables, and each mesh's triangle slots (4 bytes per triangle) in
  // the order the light-table builders walk its cull tree.
  std::vector<DObject> objs_host;
  std::vector<uint32_t> lin_objs_host;
  uint32_t sphere_root = kEmpty, ref_depth = 0, cull_depth = 0;
  std::vector<rh_texture> textures_host;
  uint64_t n_texels = 0;
  std::vector<rh_material> materials_host;
  std::vector<rh_light> lights_host;
  std::vector<uint32_t> mesh_slots;  // object i's slots: mesh_slots[slot_begin[i] .. slot_begin[i + 1])
  std::vector<size_t> slot_begin;
  // The light tables as derive_tables left them: the cube-map resolution (0: no tables), the host copy of
  // light_map_index, per occluder mesh whether it got lit-triangle queries, and whether the device builders made them.
  uint32_t tables_res = 0;
  std::vector<uint32_t> map_index_host;
  std::vector<uint8_t> mesh_lit;
  bool tables_on_device = false;
  uint64_t generation = 0;  // rh_scene_update calls that changed bytes
};

// What the per-pixel states of several calls (rh_accum, rh_adaptive) share: the frame (or shard of it) they cover, the
// device context they live on, the SplitMix64 stream they draw from and the view their first call fixed.
struct ShardState {
  Device* device = nullptr;
  uint64_t context = 0;  // device->context when the state was created
  int dev = -1;
  int width = 0, height = 0, shard_index = 0, shard_count = 1, band_height = 1, rows_local = 0;
  uint32_t stream_spp = 0;  // RH_OFFSETS_SPLITMIX64: samples per pixel of the stream the calls draw from
  size_t plane = 0;         // doubles per colour plane: rows_local * width
  const rh_scene* scene = nullptr;
  uint64_t scene_generation = 0;  // scene->generation when the view was fixed
  rh_camera camera{};
  int32_t max_depth = 0;
};

// Running per-pixel sums of one progressive frame (or of one shard's rows of it): two buffers of three planes of doubles,
// `cur` holding the sums of the n samples so far.  A call's sink reads buffer cur and writes the other; the call flips
// them and adds its samples to n only after a frame that completed, so a failed call or an overflow retry leaves the
// sums as they were.  The first call after create or reset fixes the view (scene, camera, max_depth).
struct rh_accum : ShardState {
  DevBuf sums;              // [2][3][plane]
  int cur = 0;
  uint32_t n = 0;
};

// Adaptive sampling state of one frame (or shard): per pixel the count n_p and the sums S_p and Q_p (state), and the
// per-call space: the list of active pixels and the staged new sums of its entries (work), the selection's scratch.
// A call's sink writes only the staging; the commit moves it into the state after a frame that completed, so a failed
// call or an overflow retry leaves the state as it was.  The first call after create or reset fixes the view.
struct rh_adaptive : ShardState {
  DevBuf state;    // counts uint32[plane] (padded to 8 bytes), S double[3][plane], Q double[3][plane]
  DevBuf work;     // list uint32[plane] (padded to 8 bytes), staging double[6][plane]
  DevBuf scratch;  // negative-channel counter, n_active, block counts, warp masks
  AdaptiveParams A{};  // the pointers into the three buffers and the geometry
  bool fixed = false;  // the view is fixed
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // call begin, selection end, commit begin, call end
};

namespace {

// ------------------------------------------------------------------ scene upload
// Top-level spheres.  The reference scans the object list linearly (RayHs.hs:64-71), which is what the
// kernels do too while the list is short.  A scene with many spheres (SURVEY 8d config C5: 1 000) gets a
// bounding-volume tree over them instead, walked like a mesh tree with the conservative float boxes; its
// leaves hold object indices and every candidate still gets the reference's exact double test
// (Geometry.hs:81-95).  The winner is the same: smallest time, lowest object index on a tie (RayHs.hs:67-71).
// Boxes are padded so that a ray the reference's rounded discriminant accepts cannot miss the box.
constexpr int kLightMapRes = 512;                       // cells per edge of a cube-map face (6.3 MB per map)
constexpr size_t kLightMapBudget = (size_t)256 << 20;   // all maps of a scene; the resolution halves until they fit
constexpr size_t kLitMaxQueriesDevice = 48000000;        // the same bound for the GPU builder (dragon: 82 k queries in ~2 ms)
constexpr size_t kLitMaxQueries = 1200000;              // (triangles x lights) of a mesh beyond which it gets no lit-triangle flags (host time: ~10 us per query)
constexpr double kLightMapMinEmpty = 0.02;              // a map with fewer empty cells than this is not worth its lookups
constexpr uint32_t kSphereTreeMin = 16;  // fewer spheres than this stay in the linear object list
constexpr uint32_t kSphereLeaf = 4;
constexpr uint32_t kSphereTreeFlag = 4;  // WideNode::refine bit 2: the record belongs to the sphere tree

struct SphereTree {
  std::vector<rh_node> nodes;
  std::vector<uint32_t> refs;  // object indices in leaf order
  uint32_t depth = 0;
  struct Item { uint32_t obj; double c[3], lo[3], hi[3]; };

  uint32_t build(std::vector<Item>& it, size_t b, size_t e, uint32_t d) {
    depth = std::max(depth, d);
    const double inf = std::numeric_limits<double>::infinity();
    rh_node nd{};
    double clo[3] = {inf, inf, inf}, chi[3] = {-inf, -inf, -inf};
    for (int k = 0; k < 3; k++) { nd.lo[k] = inf; nd.hi[k] = -inf; }
    for (size_t i = b; i < e; i++)
      for (int k = 0; k < 3; k++) {
        nd.lo[k] = std::min(nd.lo[k], it[i].lo[k]);
        nd.hi[k] = std::max(nd.hi[k], it[i].hi[k]);
        clo[k] = std::min(clo[k], it[i].c[k]);
        chi[k] = std::max(chi[k], it[i].c[k]);
      }
    const uint32_t self = (uint32_t)nodes.size();
    nodes.push_back(nd);
    if (e - b <= kSphereLeaf) {
      nodes[self].is_leaf = 1;
      nodes[self].left = (uint32_t)refs.size();
      nodes[self].right = (uint32_t)(e - b);
      std::sort(it.begin() + b, it.begin() + e, [](const Item& x, const Item& y) { return x.obj < y.obj; });
      for (size_t i = b; i < e; i++) refs.push_back(it[i].obj);
      return self;
    }
    int axis = 0;
    for (int k = 1; k < 3; k++)
      if (chi[k] - clo[k] > chi[axis] - clo[axis]) axis = k;
    const size_t mid = b + (e - b) / 2;
    std::nth_element(it.begin() + b, it.begin() + mid, it.begin() + e,
                     [axis](const Item& x, const Item& y) { return x.c[axis] < y.c[axis] || (x.c[axis] == y.c[axis] && x.obj < y.obj); });
    const uint32_t l = build(it, b, mid, d + 1);
    const uint32_t r = build(it, mid, e, d + 1);
    nodes[self].left = l;
    nodes[self].right = r;
    return self;
  }

  // Returns false (no tree) when there are too few spheres or one of them is not finite.
  bool run(const rh_scene_desc& d) {
    std::vector<Item> it;
    for (uint32_t i = 0; i < d.n_objects; i++) {
      const rh_object& o = d.objects[i];
      if (o.kind != RH_OBJ_SPHERE) continue;
      Item x;
      x.obj = i;
      const double r = std::fabs(o.b[0]);
      double m = r;
      for (int k = 0; k < 3; k++) m = std::max(m, std::fabs(o.a[k]));
      if (!(m < 1e30)) return false;
      const double pad = 1e-7 * m + 1e-300;
      for (int k = 0; k < 3; k++) {
        x.c[k] = o.a[k];
        x.lo[k] = o.a[k] - r - pad;
        x.hi[k] = o.a[k] + r + pad;
      }
      it.push_back(x);
    }
    if (it.size() < kSphereTreeMin) return false;
    build(it, 0, it.size(), 0);
    return true;
  }
};

int build_wide(const rh_scene_desc& d, std::vector<WideNode>& wide, std::vector<DObject>& objs, uint32_t* max_depth,
               std::vector<uint32_t>& lin_objs, std::vector<uint32_t>& sphere_refs, uint32_t* sphere_root) {
  const double inf = std::numeric_limits<double>::infinity();
  objs.resize(d.n_objects);
  struct Pending { uint32_t node, wide_index, depth; };
  std::deque<Pending> fifo;
  auto empty_box = [&](double* b) { for (int k = 0; k < 3; k++) { b[k] = inf; b[3 + k] = -inf; } };
  std::vector<uint8_t> seen(d.n_nodes, 0);
  // node array the level-order pass below reads: the caller's nodes, then the sphere tree's
  SphereTree st;
  const bool sphere_tree = st.run(d);
  std::vector<rh_node> merged;
  const rh_node* all_nodes = d.nodes;
  if (sphere_tree) {
    merged.assign(d.nodes, d.nodes + d.n_nodes);
    for (rh_node nd : st.nodes) {
      if (!nd.is_leaf) { nd.left += d.n_nodes; nd.right += d.n_nodes; }
      merged.push_back(nd);
    }
    all_nodes = merged.data();
    sphere_refs = st.refs;
    *max_depth = std::max(*max_depth, st.depth);
  }
  *sphere_root = kEmpty;
  lin_objs.clear();
  for (uint32_t i = 0; i < d.n_objects; i++) {
    const rh_object& o = d.objects[i];
    DObject& t = objs[i];
    memset(&t, 0, sizeof t);
    memcpy(t.a, o.a, sizeof t.a);
    memcpy(t.b, o.b, sizeof t.b);
    memcpy(t.c, o.c, sizeof t.c);
    t.kind = o.kind;
    t.material = o.material;
    t.root = kEmpty;
    if (o.kind != RH_OBJ_PLANE && o.kind != RH_OBJ_SPHERE && o.kind != RH_OBJ_MESH)
      return rh::set_error(RH_ERR_ARG, "rh_scene_create: unknown object kind");
    if (o.material < 0 || (uint32_t)o.material >= d.n_materials)
      return rh::set_error(RH_ERR_ARG, "rh_scene_create: object material index out of range");
    t.is_emitter = d.materials[o.material].kind == RH_MAT_EMMIT;
    if (!(sphere_tree && o.kind == RH_OBJ_SPHERE)) lin_objs.push_back(i);
    if (o.kind == RH_OBJ_MESH && o.root != RH_NO_NODE) {
      if (o.root >= d.n_nodes) return rh::set_error(RH_ERR_ARG, "rh_scene_create: mesh root out of range");
      // the leaves of one mesh must occupy increasing triangle slots in left-to-right order:
      // the slot order carries the reference's tie rule (KDTree.hs:109-115)
      std::vector<std::pair<uint32_t, uint32_t>> dfs{{o.root, 0u}};
      uint32_t last_first = 0;
      bool any_leaf = false;
      while (!dfs.empty()) {
        auto [ni, depth] = dfs.back();
        dfs.pop_back();
        if (ni >= d.n_nodes || seen[ni]) return rh::set_error(RH_ERR_ARG, "rh_scene_create: node index out of range or shared");
        seen[ni] = 1;
        *max_depth = std::max(*max_depth, depth);
        const rh_node& nd = d.nodes[ni];
        if (nd.is_leaf) {
          if ((uint64_t)nd.left + nd.right > d.n_tris) return rh::set_error(RH_ERR_ARG, "rh_scene_create: leaf range out of bounds");
          if (nd.right > kCountMask) return rh::set_error(RH_ERR_ARG, "rh_scene_create: leaf too large");
          if (any_leaf && nd.left < last_first)
            return rh::set_error(RH_ERR_ARG, "rh_scene_create: leaves must store their triangles in left-to-right leaf order");
          last_first = nd.left;
          any_leaf = true;
        } else {
          if (nd.right != RH_NO_NODE) dfs.push_back({nd.right, depth + 1});
          if (nd.left != RH_NO_NODE) dfs.push_back({nd.left, depth + 1});
        }
      }
      if (*max_depth + 4 > (uint32_t)kStack) return rh::set_error(RH_ERR_ARG, "rh_scene_create: tree deeper than 100 levels");
      // synthetic super-root: slot 0 = the root itself (its box is tested like any other, KDTree.hs:96-103)
      t.root = (uint32_t)wide.size();
      WideNode w{};
      empty_box(w.box);
      empty_box(w.box + 6);
      w.child[0] = w.child[1] = kEmpty;
      wide.push_back(w);
      fifo.push_back({o.root, t.root, 0});
    }
  }
  if (sphere_tree) {  // super-root of the sphere tree, after the meshes' super-roots
    *sphere_root = (uint32_t)wide.size();
    WideNode w{};
    empty_box(w.box);
    empty_box(w.box + 6);
    w.child[0] = w.child[1] = kEmpty;
    w.refine = kSphereTreeFlag | 3u;
    wide.push_back(w);
    fifo.push_back({d.n_nodes, *sphere_root, 0});
  }
  // level order over all meshes: fill each wide node's two child slots, queue inner children
  // `fifo` entries mean: node `node` is the (only) real child of wide record `wide_index` slot 0 when depth==0,
  // otherwise the record `wide_index` IS the inner node `node`.
  std::deque<Pending> work;
  auto child_ref = [&](uint32_t ni, WideNode& w, int slot, uint32_t depth) {
    double* box = w.box + 6 * slot;
    if (ni == RH_NO_NODE) {
      empty_box(box);
      w.child[slot] = kEmpty;
      return;
    }
    const rh_node& nd = all_nodes[ni];
    memcpy(box, nd.lo, 3 * sizeof(double));
    memcpy(box + 3, nd.hi, 3 * sizeof(double));
    if (nd.is_leaf) {
      w.child[slot] = kLeafBit | (ni >= d.n_nodes ? kSphereLeafBit : 0u) | nd.right;
      w.first[slot] = nd.left;
    } else {
      work.push_back({ni, 0, depth + 1});  // wide_index assigned when popped
      w.child[slot] = 0xFFFFFFFEu;         // patched below
    }
  };
  // First the super-roots (already in `wide`), then breadth-first.
  struct Patch { uint32_t wide_index; int slot; };
  std::deque<Patch> patches;
  for (const Pending& p : fifo) {
    size_t before = work.size();
    child_ref(p.node, wide[p.wide_index], 0, 0);
    if (work.size() > before) patches.push_back({p.wide_index, 0});
  }
  while (!work.empty()) {
    Pending p = work.front();
    work.pop_front();
    Patch pa = patches.front();
    patches.pop_front();
    const uint32_t wi = (uint32_t)wide.size();
    if (wi >= 0x7FFFFFF0u) return rh::set_error(RH_ERR_ARG, "rh_scene_create: too many nodes");
    wide[pa.wide_index].child[pa.slot] = wi;
    wide.push_back(WideNode{});
    const rh_node& nd = all_nodes[p.node];
    WideNode w{};
    // boxes of the sphere tree are not boxes the reference tests: the exact walk passes them all (refine bits)
    if (p.node >= d.n_nodes) w.refine = kSphereTreeFlag | 3u;
    size_t before = work.size();
    child_ref(nd.left, w, 0, p.depth);
    if (work.size() > before) patches.push_back({wi, 0});
    before = work.size();
    child_ref(nd.right, w, 1, p.depth);
    if (work.size() > before) patches.push_back({wi, 1});
    wide[wi] = w;
  }
  return RH_OK;
}

// Allocator that leaves trivially constructible elements uninitialised: `std::vector<T, NoInit<T>> v(n)` does not spend a
// single-threaded pass zeroing gigabytes that the next (multi-threaded) loop overwrites.
template <class T>
struct NoInit : std::allocator<T> {
  template <class U> struct rebind { using other = NoInit<U>; };
  template <class U, class... A> void construct(U* p, A&&... a) {
    if constexpr (sizeof...(A) == 0) ::new ((void*)p) U;
    else ::new ((void*)p) U(std::forward<A>(a)...);
  }
};
using TriVec = std::vector<rh_tri, NoInit<rh_tri>>;
using ShadeVec = std::vector<rh_tri_shade, NoInit<rh_tri_shade>>;

// f(begin, end, thread) over [0, n) on up to 32 host threads (one call when n is small).  f must not throw.
template <class F>
void parallel_for(size_t n, size_t min_per_thread, F f) {
  const unsigned hw = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
  const unsigned nt = (unsigned)std::max<size_t>(1, std::min<size_t>(hw, n / std::max<size_t>(1, min_per_thread)));
  if (nt <= 1) {
    f((size_t)0, n, 0u);
    return;
  }
  std::vector<std::thread> pool;
  const size_t per = (n + nt - 1) / nt;
  try {
    for (unsigned t = 1; t < nt; t++) pool.emplace_back([=]() { f(std::min(n, t * per), std::min(n, (t + 1) * per), t); });
  } catch (...) {  // (could not start a thread: the caller's thread does the rest)
    const size_t done = pool.size() + 1;
    f((size_t)0, per, 0u);
    for (size_t t = done; t < nt; t++) f(std::min(n, t * per), std::min(n, (t + 1) * per), (unsigned)t);
    for (std::thread& th : pool) th.join();
    return;
  }
  f((size_t)0, std::min(n, per), 0u);
  for (std::thread& th : pool) th.join();
}

// Bounding box of one triangle record, padded for p0 + e != p exactly.
struct TriBox {
  static void tri_box(const rh_tri& t, double* lo, double* hi) {
    for (int k = 0; k < 3; k++) {
      const double a = t.p0[k], b = t.p0[k] + t.e1[k], c = t.p0[k] + t.e2[k];
      const double pad = 4e-16 * (std::fabs(a) + std::fabs(t.e1[k]) + std::fabs(t.e2[k]));
      lo[k] = std::min(a, std::min(b, c)) - pad;
      hi[k] = std::max(a, std::max(b, c)) + pad;
    }
  }
};

// Cull tree of the float path.  The reference's tree (midpoint of the box on a cycling axis, KDTree.hs:79-90) decides
// nothing but which triangles a ray gets to test, and every triangle a ray can hit lies inside its reference leaf's box
// and all of that leaf's ancestors (the boxes are built from the triangles' own vertices).  So the float path may cull
// with ANY bounding hierarchy over the same triangles: the accepted hits are the same set, the winner is picked by the
// same key (t, reference leaf order, list position — carried in the triangle records), and the caveat is the one the
// conservative float boxes already have (a hit within an ulp of a reference box face, DESIGN.md 3).  This builds a
// binned surface-area-heuristic tree with at most kSubLeaf triangles per leaf; the exact walk keeps the reference's
// own tree and boxes and reaches the permuted triangle records through an index.
struct SahTree {
  struct Ref { uint32_t slot; float lo[3], hi[3], c[3]; };
  // One subtree in its own arrays (LOCAL child indices and leaf slots), so that the two halves of a large range can be
  // built by two threads and spliced in left-to-right order: the result is the array a sequential build writes.
  struct Sub {
    std::vector<rh_node> nodes;   // leaves: left = first slot in `order`, right = count
    std::vector<uint32_t> order;  // new slot -> reference slot
    uint32_t max_depth = 0;
  };
  const rh_tri* tris;               // reference (leaf) order
  std::vector<rh_node> nodes;       // all trees built so far; leaves: left = first NEW slot, right = count
  std::vector<uint32_t> order;      // new slot -> reference slot
  uint32_t max_depth = 0;
  std::vector<Ref> refs;
  std::atomic<bool> failed{false};

  explicit SahTree(const rh_tri* t) : tris(t) {}

  static float area(const float* lo, const float* hi) {
    const float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
    return x * y + y * z + z * x;
  }

  static uint32_t append(Sub& out, const Sub& in) {
    const uint32_t node_off = (uint32_t)out.nodes.size(), slot_off = (uint32_t)out.order.size();
    for (rh_node nd : in.nodes) {
      if (nd.is_leaf) nd.left += slot_off;
      else {
        nd.left += node_off;
        nd.right += node_off;
      }
      out.nodes.push_back(nd);
    }
    out.order.insert(out.order.end(), in.order.begin(), in.order.end());
    out.max_depth = std::max(out.max_depth, in.max_depth);
    return node_off;
  }

  uint32_t build(size_t b, size_t e, uint32_t depth, Sub& out, int fork_levels) {
    out.max_depth = std::max(out.max_depth, depth);
    const float inf = std::numeric_limits<float>::infinity();
    constexpr int kBins = 16;
    // Bounds, then the bins of all three axes in one pass over the range.  The large ranges near the root are cut into
    // pieces for several threads; min / max and the counts merge exactly, so the tree does not depend on the thread count.
    struct Bounds { float lo[3], hi[3], clo[3], chi[3]; };
    struct Bins { float blo[3][kBins][3], bhi[3][kBins][3]; uint32_t cnt[3][kBins]; };
    auto bounds_of = [&](size_t kb, size_t ke, Bounds& o) {
      for (int k = 0; k < 3; k++) { o.lo[k] = o.clo[k] = inf; o.hi[k] = o.chi[k] = -inf; }
      for (size_t i = kb; i < ke; i++)
        for (int k = 0; k < 3; k++) {
          o.lo[k] = std::min(o.lo[k], refs[i].lo[k]);
          o.hi[k] = std::max(o.hi[k], refs[i].hi[k]);
          o.clo[k] = std::min(o.clo[k], refs[i].c[k]);
          o.chi[k] = std::max(o.chi[k], refs[i].c[k]);
        }
    };
    const size_t n = e - b;
    const bool wide_range = fork_levels > 0 && n >= (1u << 20);
    const unsigned pieces = wide_range ? std::max(1u, std::min(32u, std::thread::hardware_concurrency())) : 1u;
    Bounds bd;
    if (pieces > 1) {
      std::vector<Bounds> part(pieces);
      for (Bounds& q : part) bounds_of(0, 0, q);
      parallel_for(n, 1u << 16, [&](size_t kb, size_t ke, unsigned t) { bounds_of(b + kb, b + ke, part[t % pieces]); });
      bounds_of(0, 0, bd);
      for (const Bounds& q : part)
        for (int k = 0; k < 3; k++) {
          bd.lo[k] = std::min(bd.lo[k], q.lo[k]);
          bd.hi[k] = std::max(bd.hi[k], q.hi[k]);
          bd.clo[k] = std::min(bd.clo[k], q.clo[k]);
          bd.chi[k] = std::max(bd.chi[k], q.chi[k]);
        }
    } else {
      bounds_of(b, e, bd);
    }
    const float *lo = bd.lo, *hi = bd.hi, *clo = bd.clo, *chi = bd.chi;
    rh_node nd{};
    for (int k = 0; k < 3; k++) { nd.lo[k] = lo[k]; nd.hi[k] = hi[k]; }
    const uint32_t self = (uint32_t)out.nodes.size();
    out.nodes.push_back(nd);
    if (n <= kSubLeaf) {
      out.nodes[self].is_leaf = 1;
      out.nodes[self].left = (uint32_t)out.order.size();
      out.nodes[self].right = (uint32_t)n;
      for (size_t i = b; i < e; i++) out.order.push_back(refs[i].slot);
      return self;
    }
    // binned SAH over the three axes; deep or degenerate ranges fall back to the object median of the widest axis
    int best_axis = -1, best_bin = 0;
    float best_cost = inf;
    if (depth < 48) {
      float scale[3];
      for (int axis = 0; axis < 3; axis++) scale[axis] = (chi[axis] - clo[axis] > 0) ? (float)kBins / (chi[axis] - clo[axis]) : 0.f;
      auto clear_bins = [&](Bins& q) {
        for (int a = 0; a < 3; a++)
          for (int i = 0; i < kBins; i++) {
            q.cnt[a][i] = 0;
            for (int k = 0; k < 3; k++) { q.blo[a][i][k] = inf; q.bhi[a][i][k] = -inf; }
          }
      };
      auto bin_range = [&](size_t kb, size_t ke, Bins& q) {
        for (size_t i = kb; i < ke; i++)
          for (int axis = 0; axis < 3; axis++) {
            if (!(scale[axis] > 0)) continue;
            int bi = (int)((refs[i].c[axis] - clo[axis]) * scale[axis]);
            bi = bi < 0 ? 0 : (bi >= kBins ? kBins - 1 : bi);
            q.cnt[axis][bi]++;
            for (int k = 0; k < 3; k++) {
              q.blo[axis][bi][k] = std::min(q.blo[axis][bi][k], refs[i].lo[k]);
              q.bhi[axis][bi][k] = std::max(q.bhi[axis][bi][k], refs[i].hi[k]);
            }
          }
      };
      Bins bins_store;  // (1.3 KB on the stack per level)
      Bins* bins = &bins_store;
      clear_bins(*bins);
      if (pieces > 1) {
        std::vector<Bins> part(pieces);
        for (Bins& q : part) clear_bins(q);
        parallel_for(n, 1u << 16, [&](size_t kb, size_t ke, unsigned t) { bin_range(b + kb, b + ke, part[t % pieces]); });
        for (const Bins& q : part)
          for (int a = 0; a < 3; a++)
            for (int i = 0; i < kBins; i++) {
              bins->cnt[a][i] += q.cnt[a][i];
              for (int k = 0; k < 3; k++) {
                bins->blo[a][i][k] = std::min(bins->blo[a][i][k], q.blo[a][i][k]);
                bins->bhi[a][i][k] = std::max(bins->bhi[a][i][k], q.bhi[a][i][k]);
              }
            }
      } else {
        bin_range(b, e, *bins);
      }
      for (int axis = 0; axis < 3; axis++) {
        if (!(scale[axis] > 0)) continue;
        const auto& blo = bins->blo[axis];
        const auto& bhi = bins->bhi[axis];
        const uint32_t* cnt = bins->cnt[axis];
        float rarea[kBins];
        uint32_t rcnt[kBins];
        float alo[3] = {inf, inf, inf}, ahi[3] = {-inf, -inf, -inf};
        uint32_t c = 0;
        for (int i = kBins - 1; i > 0; i--) {
          for (int k = 0; k < 3; k++) { alo[k] = std::min(alo[k], blo[i][k]); ahi[k] = std::max(ahi[k], bhi[i][k]); }
          c += cnt[i];
          rarea[i] = c ? area(alo, ahi) : 0.f;
          rcnt[i] = c;
        }
        for (int k = 0; k < 3; k++) { alo[k] = inf; ahi[k] = -inf; }
        c = 0;
        for (int i = 1; i < kBins; i++) {
          for (int k = 0; k < 3; k++) { alo[k] = std::min(alo[k], blo[i - 1][k]); ahi[k] = std::max(ahi[k], bhi[i - 1][k]); }
          c += cnt[i - 1];
          if (!c || !rcnt[i]) continue;
          const float cost = area(alo, ahi) * (float)c + rarea[i] * (float)rcnt[i];
          if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = i; }
        }
      }
    }
    size_t mid;
    if (best_axis >= 0) {
      const int axis = best_axis;
      const float ext = chi[axis] - clo[axis], scale = (float)kBins / ext, c0 = clo[axis];
      const int bb = best_bin;
      mid = std::partition(refs.begin() + b, refs.begin() + e, [=](const Ref& r) {
              int bi = (int)((r.c[axis] - c0) * scale);
              bi = bi < 0 ? 0 : (bi >= kBins ? kBins - 1 : bi);
              return bi < bb;
            }) - refs.begin();
    } else {
      int axis = 0;
      for (int k = 1; k < 3; k++)
        if (chi[k] - clo[k] > chi[axis] - clo[axis]) axis = k;
      mid = b + n / 2;
      std::nth_element(refs.begin() + b, refs.begin() + mid, refs.begin() + e,
                       [axis](const Ref& x, const Ref& y) { return x.c[axis] < y.c[axis] || (x.c[axis] == y.c[axis] && x.slot < y.slot); });
    }
    if (mid == b || mid == e) mid = b + n / 2;
    uint32_t l, r;
    if (fork_levels > 0 && n >= (1u << 15) && !failed.load(std::memory_order_relaxed)) {
      Sub L, R;  // the two halves touch disjoint ranges of `refs`
      std::thread th([&]() {
        try {
          build(b, mid, depth + 1, L, fork_levels - 1);
        } catch (...) {
          failed = true;  // (no exception may leave a thread; the caller reports out-of-memory)
        }
      });
      try {
        build(mid, e, depth + 1, R, fork_levels - 1);
      } catch (...) {
        failed = true;
      }
      th.join();
      if (failed) return self;
      l = append(out, L);
      r = append(out, R);
    } else {
      l = build(b, mid, depth + 1, out, 0);
      r = build(mid, e, depth + 1, out, 0);
    }
    out.nodes[self].left = l;
    out.nodes[self].right = r;
    return self;
  }

  // Builds the tree of the triangles in the given reference slots; returns the root node index (RH_NO_NODE if none).
  uint32_t run(const std::vector<uint32_t>& slots) {
    if (slots.empty()) return RH_NO_NODE;
    const uint32_t count = (uint32_t)slots.size();
    refs.resize(count);
    parallel_for(count, 1u << 16, [&](size_t kb, size_t ke, unsigned) {
      for (size_t k = kb; k < ke; k++) {
        Ref& r = refs[k];
        r.slot = slots[k];
        double lo[3], hi[3];
        TriBox::tri_box(tris[slots[k]], lo, hi);
        for (int a = 0; a < 3; a++) {  // float is enough to choose splits; the stored boxes are recomputed in double
          r.lo[a] = (float)lo[a];
          r.hi[a] = (float)hi[a];
          r.c[a] = 0.5f * (r.lo[a] + r.hi[a]);
        }
      }
    });
    const unsigned n_threads = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    int fork_levels = 0;
    while ((1u << fork_levels) < n_threads) fork_levels++;
    Sub sub;
    build(0, count, 0, sub, count >= (1u << 16) ? fork_levels + 1 : 0);
    if (failed) throw std::bad_alloc();
    // splice into the arrays of all trees
    const uint32_t node_off = (uint32_t)nodes.size(), slot_off = (uint32_t)order.size();
    for (rh_node nd : sub.nodes) {
      if (nd.is_leaf) nd.left += slot_off;
      else {
        nd.left += node_off;
        nd.right += node_off;
      }
      nodes.push_back(nd);
    }
    order.insert(order.end(), sub.order.begin(), sub.order.end());
    max_depth = std::max(max_depth, sub.max_depth);
    return node_off;
  }

  // Exact (double, padded) boxes of all nodes from the permuted triangles, bottom-up.
  void refit(const TriVec& new_tris) {
    const double inf = std::numeric_limits<double>::infinity();
    parallel_for(nodes.size(), 1u << 16, [&](size_t ib, size_t ie, unsigned) {  // the leaves (independent of each other)
      for (size_t i = ib; i < ie; i++) {
        rh_node& nd = nodes[i];
        if (!nd.is_leaf) continue;
        for (int k = 0; k < 3; k++) { nd.lo[k] = inf; nd.hi[k] = -inf; }
        for (uint32_t t = 0; t < nd.right; t++) {
          double lo[3], hi[3];
          TriBox::tri_box(new_tris[nd.left + t], lo, hi);
          for (int k = 0; k < 3; k++) { nd.lo[k] = std::min(nd.lo[k], lo[k]); nd.hi[k] = std::max(nd.hi[k], hi[k]); }
        }
      }
    });
    for (size_t i = nodes.size(); i-- > 0;) {  // children always follow their parent in `nodes`
      rh_node& nd = nodes[i];
      if (nd.is_leaf) continue;
      for (int k = 0; k < 3; k++) { nd.lo[k] = inf; nd.hi[k] = -inf; }
      for (uint32_t c : {nd.left, nd.right})
        for (int k = 0; k < 3; k++) { nd.lo[k] = std::min(nd.lo[k], nodes[c].lo[k]); nd.hi[k] = std::max(nd.hi[k], nodes[c].hi[k]); }
    }
  }
};

template <class T>
int upload(DevBuf& b, const T* src, size_t n) {
  int rc = b.reserve(std::max<size_t>(n * sizeof(T), 256));
  if (rc) return rc;
  if (n) RH_CUDA(cudaMemcpy(b.p, src, n * sizeof(T), cudaMemcpyHostToDevice));
  return RH_OK;
}

// rh_scene_create's checks of the material and light tables (rh_scene_update makes the same ones).
int check_tables(const rh_material* mats, uint32_t n_materials, const rh_texture* textures, uint32_t n_textures, uint64_t n_texels,
                 const rh_light* lights, uint32_t n_lights, const std::string& w) {
  for (uint32_t i = 0; i < n_materials; i++) {
    const rh_material& m = mats[i];
    if (m.kind < RH_MAT_MIRROR || m.kind > RH_MAT_SHOWUV) return rh::set_error(RH_ERR_ARG, w + ": unknown material kind");
    if ((m.kind == RH_MAT_DIFFUSE || m.kind == RH_MAT_PLASTIC)) {
      if (m.cmap_kind < RH_CMAP_FLAT || m.cmap_kind > RH_CMAP_TEXTURE) return rh::set_error(RH_ERR_ARG, w + ": unknown colour-map kind");
      if (m.cmap_kind == RH_CMAP_TEXTURE) {
        if (m.texture < 0 || (uint32_t)m.texture >= n_textures) return rh::set_error(RH_ERR_ARG, w + ": texture index out of range");
        const rh_texture& t = textures[m.texture];
        if (t.w <= 0 || t.h <= 0 || t.offset + (uint64_t)t.w * t.h > n_texels)
          return rh::set_error(RH_ERR_ARG, w + ": texture outside the texel array");
      }
    }
  }
  for (uint32_t i = 0; i < n_lights; i++) {
    const rh_light& L = lights[i];
    if (L.kind != RH_LIGHT_DIRECTIONAL && L.kind != RH_LIGHT_POINT && L.kind != RH_LIGHT_SPHERE)
      return rh::set_error(RH_ERR_ARG, w + ": unknown light kind");
    if (L.kind == RH_LIGHT_SPHERE && !(std::isfinite(L.radius) && L.radius >= 0))
      return rh::set_error(RH_ERR_ARG, w + ": lights[" + std::to_string(i) + "]: a sphere light's radius must be finite and >= 0");
  }
  return RH_OK;
}

// RAYHS_B200_SETUP=host: rh_scene_create's host builders of the light tables (light_maps.cpp) read the cull tree and the
// triangle records on the host.
struct HostGeometry {
  const std::vector<WideNode>* cull;
  const TriVec* tris;
};

int derive_tables(Device* D, const rh_scene& G, const rh_material* mats, uint32_t n_materials, const rh_light* lights,
                  uint32_t n_lights, const HostGeometry* host, const rh_scene* old, rh_scene* T, rh_update_info* info,
                  const std::string& w);

int scene_create_on(Device* D, const rh_scene_desc* d, rh_scene** out) {
  if (!d || !out) return rh::set_error(RH_ERR_ARG, "rh_scene_create: null argument");
  if (d->n_materials > 0x7fff) return rh::set_error(RH_ERR_ARG, "rh_scene_create: more than 32767 materials");
  if ((d->n_nodes && !d->nodes) || (d->n_tris && (!d->tris || !d->tri_shade)) || (d->n_objects && !d->objects) ||
      (d->n_materials && !d->materials) || (d->n_lights && !d->lights))
    return rh::set_error(RH_ERR_ARG, "rh_scene_create: null array with non-zero count");
  if (int rc = check_tables(d->materials, d->n_materials, d->textures, d->n_textures, d->n_texels, d->lights, d->n_lights, "rh_scene_create"))
    return rc;
  using clk = std::chrono::steady_clock;
  auto ms_since = [](clk::time_point t) { return std::chrono::duration<double, std::milli>(clk::now() - t).count(); };
  const clk::time_point t_begin = clk::now();
  static const bool debug_setup = getenv("RAYHS_B200_DEBUG") && strchr(getenv("RAYHS_B200_DEBUG"), 's');
  clk::time_point t_stage = t_begin;
  auto stage = [&](const char* what) {
    if (debug_setup) fprintf(stderr, "rayhs_b200: scene_create %-28s %8.1f ms\n", what, ms_since(t_stage));
    t_stage = clk::now();
  };
  std::vector<WideNode> wide;
  std::vector<DObject> objs;
  uint32_t depth = 0;
  TriVec dtris;
  ShadeVec dshade;
  std::vector<uint32_t> lin_objs, sphere_refs;
  uint32_t sphere_root = kEmpty;
  std::vector<WideNode> wide_cull;      // the float path's own tree (same super-root indices as `wide`)
  uint32_t cull_depth = 0;              // its depth (the reference tree's is `depth`)
  std::vector<uint32_t> exact_index;    // reference slot -> slot in the permuted triangle arrays
  try {
    // the reference tree's wide records (exact walk) are built on their own thread beside the cull tree
    int rc = RH_OK, rc_ref = RH_OK;
    std::string ref_error;
    bool ref_threw = false;
    std::thread ref_thread([&]() {
      try {
        rc_ref = build_wide(*d, wide, objs, &depth, lin_objs, sphere_refs, &sphere_root);
        if (rc_ref) ref_error = rh::g_err;  // (the message is thread-local)
      } catch (...) {
        ref_threw = true;
      }
    });
    struct Joiner { std::thread& t; ~Joiner() { if (t.joinable()) t.join(); } } ref_join{ref_thread};
    // order key of the tie rule: the first slot of a triangle's reference leaf (leaves are numbered left to right by it)
    std::vector<uint32_t> leaf_key(d->n_tris, 0);
    for (uint32_t ni = 0; ni < d->n_nodes; ni++)
      if (d->nodes[ni].is_leaf)
        for (uint32_t k = 0; k < d->nodes[ni].right; k++) leaf_key[d->nodes[ni].left + k] = d->nodes[ni].left;
    stage("leaf keys");
    {
      SahTree sah(d->tris);
      std::vector<rh_object> objects2(d->objects, d->objects + d->n_objects);
      for (uint32_t i = 0; i < d->n_objects; i++) {
        if (objects2[i].kind != RH_OBJ_MESH || objects2[i].root == RH_NO_NODE) continue;
        std::vector<uint32_t> slots, dfs{objects2[i].root};
        while (!dfs.empty()) {  // the mesh's triangles, in reference order
          const rh_node& nd = d->nodes[dfs.back()];
          dfs.pop_back();
          if (nd.is_leaf) {
            for (uint32_t k = 0; k < nd.right; k++) slots.push_back(nd.left + k);
          } else {
            if (nd.right != RH_NO_NODE) dfs.push_back(nd.right);
            if (nd.left != RH_NO_NODE) dfs.push_back(nd.left);
          }
        }
        objects2[i].root = sah.run(slots);
      }
      stage("cull tree (binned SAH)");
      ref_thread.join();
      if (ref_threw) throw std::bad_alloc();
      if (rc_ref) return rh::set_error(rc_ref, ref_error);
      stage("reference tree -> wide nodes (rest)");
      // permute the records into the cull tree's leaf order
      TriVec ptris(sah.order.size());
      ShadeVec pshade(sah.order.size());
      exact_index.assign(d->n_tris, 0);
      parallel_for(sah.order.size(), 1u << 16, [&](size_t kb, size_t ke, unsigned) {  // (the caller's records are copied once)
        for (size_t k = kb; k < ke; k++) {
          const uint32_t from = sah.order[k];
          ptris[k] = d->tris[from];
          ptris[k].pad_ = leaf_key[from];
          pshade[k] = d->tri_shade[from];
          exact_index[from] = (uint32_t)k;
        }
      });
      stage("permutation");
      sah.refit(ptris);
      stage("refit");
      dtris.swap(ptris);
      dshade.swap(pshade);
      rh_scene_desc d2 = *d;
      d2.objects = objects2.data();
      d2.nodes = sah.nodes.data();
      d2.n_nodes = (uint32_t)sah.nodes.size();
      d2.n_tris = (uint32_t)dtris.size();
      std::vector<DObject> objs2;
      std::vector<uint32_t> lin2, refs2;
      uint32_t depth2 = 0, sroot2 = kEmpty;
      rc = build_wide(d2, wide_cull, objs2, &depth2, lin2, refs2, &sroot2);
      if (rc) return rc;
      stage("cull tree -> wide nodes");
      for (size_t i = 0; i < objs.size(); i++)
        if (objs[i].root != objs2[i].root) return rh::set_error(RH_ERR_STATE, "rh_scene_create: cull tree roots out of step");
      if (sroot2 != sphere_root) return rh::set_error(RH_ERR_STATE, "rh_scene_create: sphere tree roots out of step");
      cull_depth = depth2;
    }
    if (std::max(depth, cull_depth) + 4 > (uint32_t)kStack)
      return rh::set_error(RH_ERR_ARG, "rh_scene_create: tree too deep for the traversal stack");
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, "rh_scene_create: out of host memory");
  }
  const std::vector<WideNode>& cull = wide_cull.empty() ? wide : wide_cull;
  RH_CUDA(cudaSetDevice(D->dev));
  auto S = std::make_unique<rh_scene>();
  S->device = D;
  S->max_tree_depth = std::max(depth, cull_depth);
  int rc;
  // conservative float copy of the boxes: lower bounds rounded down, upper bounds rounded up
  // ... stored relative to the middle of all boxes, so that a scene far from the coordinate origin keeps float's full
  // resolution (one correctly rounded double subtraction per coordinate, then one extra float ulp outward for it)
  std::vector<WideNode32> wide32(cull.size());
  float abs_max = 0.f;
  double center[3] = {0, 0, 0};
  {
    const double inf = std::numeric_limits<double>::infinity();
    double blo[3] = {inf, inf, inf}, bhi[3] = {-inf, -inf, -inf};
    for (const WideNode& w : cull)
      for (int c = 0; c < 2; c++)
        if (w.child[c] != kEmpty)
          for (int k = 0; k < 3; k++) {
            const double lo = w.box[6 * c + k], hi = w.box[6 * c + 3 + k];
            if (!(std::fabs(lo) < 1e30) || !(std::fabs(hi) < 1e30))
              return rh::set_error(RH_ERR_ARG, "rh_scene_create: box coordinate is not finite or exceeds 1e30");
            blo[k] = std::min(blo[k], lo);
            bhi[k] = std::max(bhi[k], hi);
          }
    for (int k = 0; k < 3; k++)
      if (blo[k] <= bhi[k]) center[k] = 0.5 * (blo[k] + bhi[k]);
  }
  const float finf = std::numeric_limits<float>::infinity();
  {
    const unsigned hw = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    std::vector<float> abs_max_of(hw + 1, 0.f);
    std::atomic<bool> bad_leaf{false};
    parallel_for(cull.size(), 1u << 15, [&](size_t ib, size_t ie, unsigned t) {
      float amax = 0.f;
      for (size_t i = ib; i < ie; i++) {
        const WideNode& w = cull[i];
        WideNode32& n = wide32[i];
        for (int c = 0; c < 2; c++) {
          for (int k = 0; k < 3; k++) {
            const double lo = w.box[6 * c + k] - center[k], hi = w.box[6 * c + 3 + k] - center[k];
            float flo = (float)lo, fhi = (float)hi;
            if ((double)flo > lo) flo = std::nextafterf(flo, -finf);
            if ((double)fhi < hi) fhi = std::nextafterf(fhi, finf);
            if (std::isfinite(flo)) flo = std::nextafterf(flo, -finf);
            if (std::isfinite(fhi)) fhi = std::nextafterf(fhi, finf);
            n.box[6 * c + k] = flo;
            n.box[6 * c + 3 + k] = fhi;
            if (w.child[c] != kEmpty) amax = std::max(amax, std::max(std::fabs(flo), std::fabs(fhi)));
          }
          // leaf references of the cull tree carry their slot range (see kLeafCountShift): a stacked subtree is one word
          uint32_t ch = w.child[c];
          if (ch != kEmpty && (ch & kLeafBit)) {
            const uint32_t count = ch & kCountMask;
            if (count == 0 || count > kLeafMaxCount || w.first[c] > kLeafFirstMask) {
              bad_leaf = true;
              continue;
            }
            ch = (ch & (kLeafBit | kSphereLeafBit)) | ((count - 1) << kLeafCountShift) | w.first[c];
          }
          n.child[c] = ch;
        }
        n.pad_[0] = n.pad_[1] = 0;
      }
      abs_max_of[std::min<unsigned>(t, hw)] = amax;
    });
    if (bad_leaf) return rh::set_error(RH_ERR_ARG, "rh_scene_create: more than 134 M triangle slots, or a cull-tree leaf out of range");
    for (float a : abs_max_of) abs_max = std::max(abs_max, a);
  }
  stage("float boxes");
  S->ms_trees = ms_since(t_begin);
  clk::time_point t_mark = clk::now();
  if ((rc = upload(S->wide, wide.data(), wide.size()))) return rc;
  if ((rc = upload(S->wide32, wide32.data(), wide32.size()))) return rc;
  if ((rc = upload(S->tris, dtris.data(), dtris.size()))) return rc;
  if ((rc = upload(S->shade, dshade.data(), dshade.size()))) return rc;
  if ((rc = upload(S->textures, d->textures, d->n_textures))) return rc;
  if ((rc = upload(S->texels, d->texels, (size_t)d->n_texels * 3))) return rc;
  if ((rc = upload(S->lin_objs, lin_objs.data(), lin_objs.size()))) return rc;
  if ((rc = upload(S->sphere_refs, sphere_refs.data(), sphere_refs.size()))) return rc;
  if ((rc = upload(S->exact_index, exact_index.data(), exact_index.size()))) return rc;
  SceneView& v = S->view;
  v.wide = (const WideNode*)S->wide.p;
  v.wide32 = (const WideNode32*)S->wide32.p;
  v.abs_max = abs_max;
  for (int k = 0; k < 3; k++) v.center[k] = center[k];
  v.tris = (const rh_tri*)S->tris.p;
  v.shade = (const rh_tri_shade*)S->shade.p;
  v.textures = (const rh_texture*)S->textures.p;
  v.texels = (const double*)S->texels.p;
  v.n_wide = (uint32_t)cull.size();
  v.n_tris = (uint32_t)dtris.size();  // triangle slots on the device (the meshes' triangles, in cull-tree leaf order)
  v.n_objects = d->n_objects;
  v.n_textures = d->n_textures;
  v.lin_objs = (const uint32_t*)S->lin_objs.p;
  v.sphere_refs = (const uint32_t*)S->sphere_refs.p;
  v.exact_index = exact_index.empty() ? nullptr : (const uint32_t*)S->exact_index.p;
  v.n_lin = (uint32_t)lin_objs.size();
  v.sphere_root = sphere_root;
  v.n_smem_nodes = std::min<uint32_t>(v.n_wide, kSmemNodes);
  S->ms_upload = ms_since(t_mark);
  // what derive_tables reads, now and on every rh_scene_update
  try {
    S->objs_host.swap(objs);
    S->lin_objs_host.swap(lin_objs);
    S->sphere_root = sphere_root;
    S->ref_depth = depth;
    S->cull_depth = cull_depth;
    S->textures_host.assign(d->textures, d->textures + d->n_textures);
    S->n_texels = d->n_texels;
    S->slot_begin.assign((size_t)d->n_objects + 1, 0);
    std::vector<uint32_t> dfs;
    for (uint32_t i = 0; i < d->n_objects; i++) {
      S->slot_begin[i] = S->mesh_slots.size();
      if (S->objs_host[i].kind != RH_OBJ_MESH || S->objs_host[i].root == kEmpty) continue;
      dfs.assign(1, S->objs_host[i].root);  // the mesh's triangles: leaves of its cull tree
      while (!dfs.empty()) {
        const WideNode& w = cull[dfs.back()];
        dfs.pop_back();
        for (int c = 0; c < 2; c++) {
          if (w.child[c] == kEmpty) continue;
          if (w.child[c] & kLeafBit)
            for (uint32_t k = 0; k < (w.child[c] & kCountMask); k++) S->mesh_slots.push_back(w.first[c] + k);
          else dfs.push_back(w.child[c]);
        }
      }
    }
    S->slot_begin[d->n_objects] = S->mesh_slots.size();
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, "rh_scene_create: out of host memory");
  }
  const char* env_setup = getenv("RAYHS_B200_SETUP");
  const HostGeometry on_host{&cull, &dtris};
  if ((rc = derive_tables(D, *S, d->materials, d->n_materials, d->lights, d->n_lights,
                          env_setup && strcmp(env_setup, "host") == 0 ? &on_host : nullptr, nullptr, S.get(), nullptr, "rh_scene_create")))
    return rc;
  *out = S.release();
  return RH_OK;
}

// Device buffers of one table build that do not outlive it.
struct ScratchBufs {
  std::vector<DevBuf> bufs;
  ~ScratchBufs() {
    for (DevBuf& b : bufs) b.release();
  }
};

// Everything rh_scene_create derives from the material and light tables: the object records (is_emitter), the occluder
// tables and what depends on them (shadow_fast, refill_possible, deep_entries), has_transparent, tables_in_smem, and the
// light-space tables of the shadow kernels.  G is the scene whose geometry the tables are for.  They go into T's buffers,
// view and host copies: T is G in rh_scene_create, a fresh scene in rh_scene_update, which swaps them in on success.
// old (rh_scene_update with an unchanged occluder set): earlier device-built tables of G whose cube maps and lit-triangle
// bits are carried over where the light they belong to did not move; else every table is built anew.  host: build the
// light tables with the host builders (rh_scene_create only); null: on the device.
int derive_tables(Device* D, const rh_scene& G, const rh_material* mats, uint32_t n_materials, const rh_light* lights,
                  uint32_t n_lights, const HostGeometry* host, const rh_scene* old, rh_scene* T, rh_update_info* info,
                  const std::string& w) {
  using clk = std::chrono::steady_clock;
  const clk::time_point t_begin = clk::now();
  RH_CUDA(cudaSetDevice(D->dev));
  int rc;
  std::vector<DObject> objs;
  std::vector<OccPlane> occ_planes;
  std::vector<OccSphere> occ_spheres;
  std::vector<uint32_t> occ_meshes, occ_objs;  // occluder meshes: super-root, object index
  try {
    objs = G.objs_host;
    for (DObject& o : objs) o.is_emitter = mats[o.material].kind == RH_MAT_EMMIT;
    T->materials_host.assign(mats, mats + n_materials);
    T->lights_host.assign(lights, lights + n_lights);
    // occluder tables (isOccluder, RayHs.hs:81-82: everything but Emmit objects)
    for (uint32_t i : G.lin_objs_host) {
      const DObject& o = objs[i];
      if (o.is_emitter) continue;
      if (o.kind == RH_OBJ_PLANE) {
        OccPlane q;
        memcpy(q.p, o.a, sizeof q.p);
        memcpy(q.n, o.b, sizeof q.n);
        occ_planes.push_back(q);
      } else if (o.kind == RH_OBJ_SPHERE) {
        OccSphere q;
        memcpy(q.c, o.a, sizeof q.c);
        q.r = o.b[0];
        occ_spheres.push_back(q);
      } else if (o.root != kEmpty) {
        occ_meshes.push_back(o.root);
        occ_objs.push_back(i);
      }
    }
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, w + ": out of host memory");
  }
  if ((rc = upload(T->objects, objs.data(), objs.size()))) return rc;
  if ((rc = upload(T->materials, mats, n_materials))) return rc;
  if ((rc = upload(T->lights, lights, n_lights))) return rc;
  if ((rc = upload(T->occ_planes, occ_planes.data(), occ_planes.size()))) return rc;
  if ((rc = upload(T->occ_spheres, occ_spheres.data(), occ_spheres.size()))) return rc;
  if ((rc = upload(T->occ_meshes, occ_meshes.data(), occ_meshes.size()))) return rc;
  SceneView& v = T->view;
  v.objects = (const DObject*)T->objects.p;
  v.materials = (const rh_material*)T->materials.p;
  v.lights = (const rh_light*)T->lights.p;
  v.n_materials = n_materials;
  v.n_lights = n_lights;
  v.occ_planes = (const OccPlane*)T->occ_planes.p;
  v.occ_spheres = (const OccSphere*)T->occ_spheres.p;
  v.occ_meshes = (const uint32_t*)T->occ_meshes.p;
  v.n_occ_planes = (uint32_t)occ_planes.size();
  v.n_occ_spheres = (uint32_t)occ_spheres.size();
  v.n_occ_meshes = (uint32_t)occ_meshes.size();
  v.shadow_fast = occ_planes.size() <= (size_t)kOccPlanes && occ_spheres.size() <= (size_t)kOccSpheres &&
                  occ_meshes.size() <= (size_t)kOccMeshes && n_lights <= (uint32_t)kFastLights;
  v.tables_in_smem = (objs.size() <= (size_t)kSmemObjects && n_materials <= (uint32_t)kSmemObjects && n_lights <= (uint32_t)kSmemLights);
  T->has_transparent = false;
  for (uint32_t i = 0; i < n_materials; i++) T->has_transparent |= mats[i].kind == RH_MAT_TRANSPARENT;
  T->has_sphere_lights = false;
  for (uint32_t i = 0; i < n_lights; i++) T->has_sphere_lights |= lights[i].kind == RH_LIGHT_SPHERE;
  {
    // Deep-stack scratch (entries beyond the shared-memory short stack, and the exact walk's whole stack): a walk
    // stacks at most one entry per level of its tree; the per-lane-refill shadow kernel also stacks the other roots.
    const uint32_t n_roots = (uint32_t)occ_meshes.size() + (G.sphere_root != kEmpty ? 1u : 0u);
    T->refill_possible = n_roots <= 64;
    const uint32_t float_need = G.cull_depth + (T->refill_possible ? n_roots : 1u) + 4;
    T->deep_entries = std::max<uint32_t>(G.ref_depth + 4, float_need > (uint32_t)kShortStack ? float_need - kShortStack : 1u);
  }
  // Light-space tables of the shadow kernels (light_maps.cpp): cube maps of the nearest possible occluder distance, one
  // per (point light, occluder mesh), and lit-triangle flags per (triangle, point or directional light).  Only the
  // shared-memory-table shadow kernels read them.  Both hold for one light point, so a sphere light has neither, and
  // neither the map budget nor the lit-query limit counts it: the other lights get the tables of the scene without it.
  v.light_maps = nullptr;
  v.lit_flags = nullptr;
  v.light_map_index = nullptr;
  v.light_map_res = 0;
  T->n_light_maps = 0;
  T->tables_res = 0;
  T->map_index_host.clear();
  T->mesh_lit.clear();
  T->tables_on_device = host == nullptr;
  const rh_tri* d_tris = (const rh_tri*)G.tris.p;
  auto mesh_slots = [&](size_t m) { return G.mesh_slots.data() + G.slot_begin[occ_objs[m]]; };
  auto mesh_n_slots = [&](size_t m) { return G.slot_begin[occ_objs[m] + 1] - G.slot_begin[occ_objs[m]]; };
  {
    uint32_t n_point = 0, n_sphere = 0, sphere_bits = 0;  // (sphere_bits: of the light indices that have lit bits)
    for (uint32_t li = 0; li < n_lights; li++) {
      n_point += lights[li].kind == RH_LIGHT_POINT;
      n_sphere += lights[li].kind == RH_LIGHT_SPHERE;
      if (lights[li].kind == RH_LIGHT_SPHERE && li < 12) sphere_bits |= 1u << li;
    }
    const uint32_t n_table_lights = n_lights - n_sphere;
    const size_t n_pairs = (size_t)n_point * occ_meshes.size();
    if (v.shadow_fast && !occ_meshes.empty() && n_lights) {
      int R = kLightMapRes;
      while (R > 64 && std::max<size_t>(n_pairs, 1) * 6 * (size_t)R * R * sizeof(float) > kLightMapBudget) R /= 2;
      const size_t cells = (size_t)6 * R * R;
      try {
        std::vector<uint32_t> index((size_t)n_lights * kOccMeshes, kEmpty);
        uint32_t n_maps = 0;
        // The tables are built on the GPU (setup_kernels.cu: the triangle records and the cull tree are already in
        // HBM); RAYHS_B200_SETUP=host keeps the host builders of light_maps.cpp — same geometry code (light_geom.h),
        // same tables bit for bit (tests/test_round2_gpu.py).
        if (!host) {
          // Maps of a light that did not move (same kind and position, at any index) are copied from the old tables
          // into their place in the new numbering, with their old verdict; so are lit bits of unchanged light indices.
          const bool reuse_maps = old && old->tables_on_device && old->tables_res == (uint32_t)R;
          const std::vector<rh::MapStep> steps =
              rh::plan_maps(reuse_maps ? old->map_index_host : std::vector<uint32_t>(),
                            old ? rh::match_point_lights(old->lights_host.data(), (uint32_t)old->lights_host.size(), lights, n_lights)
                                : std::vector<int32_t>(n_lights, -1),
                            lights, n_lights, (uint32_t)occ_meshes.size());
          ScratchBufs scratch;
          scratch.bufs.resize(occ_meshes.size() + 1);
          DevBuf& words = scratch.bufs.back();
          std::vector<uint8_t> want(occ_meshes.size(), 0);
          if ((rc = words.reserve(64))) return rc;
          RH_CUDA(cudaMemsetAsync(words.p, 0, 64, D->stream));
          if (n_pairs && (rc = T->light_maps.reserve(n_pairs * cells * sizeof(float)))) return rc;
          for (size_t m = 0; m < occ_meshes.size(); m++) {
            const size_t n_slots = mesh_n_slots(m);
            if (!n_slots) continue;
            if ((rc = upload(scratch.bufs[m], mesh_slots(m), n_slots))) return rc;
            const uint32_t* d_slots = (const uint32_t*)scratch.bufs[m].p;
            // the cube maps first: a mesh none of whose maps is worth having is a triangle soup around its lights, where
            // nearly every triangle is shadowed by another one — the lit-triangle queries (long hulls through the whole
            // soup, ~0.25 us each on the GPU) are not made either
            uint32_t useful_maps = 0;
            for (uint32_t j = 0; j < n_point; j++) {
              const rh::MapStep& st = steps[m * n_point + j];
              float* dst = (float*)T->light_maps.p + (size_t)n_maps * cells;
              int useful = 0;
              if (st.raster) {
                double empty = 0;
                RH_CUDA((cudaError_t)device_light_map(lights[st.light].vec, d_tris, d_slots, n_slots, R, dst, kLightMapMinEmpty,
                                                      (unsigned long long*)words.p, &useful, &empty, D->stream));
                if (info) info->maps_rasterised++;
              } else if (st.old_map != kEmpty) {
                RH_CUDA(cudaMemcpyAsync(dst, (const float*)old->light_maps.p + (size_t)st.old_map * cells, cells * sizeof(float),
                                        cudaMemcpyDeviceToDevice, D->stream));
                useful = 1;
                if (info) info->maps_kept++;
              }
              if (useful) {
                index[(size_t)st.light * kOccMeshes + m] = n_maps++;
                useful_maps++;
              }
            }
            want[m] = n_slots * (size_t)n_table_lights <= kLitMaxQueriesDevice && (n_point == 0 || useful_maps > 0);
          }
          // lit triangles: the old bits of every light index whose light kept its kind and position stay, as long as
          // every mesh that had bits still has them (a mesh that gains them is queried for every light)
          const uint32_t all = n_lights >= 12 ? 0x0fffu : (1u << n_lights) - 1;
          bool reuse_lit = old && old->tables_on_device && old->tables_res && old->lit_flags.p && old->mesh_lit.size() == occ_meshes.size();
          for (size_t m = 0; reuse_lit && m < occ_meshes.size(); m++) reuse_lit = !(old->mesh_lit[m] && !want[m]);
          const uint32_t changed =
              reuse_lit ? rh::lit_changed_mask(old->lights_host.data(), (uint32_t)old->lights_host.size(), lights, n_lights) : all;
          for (size_t m = 0; m < occ_meshes.size(); m++) {
            if (!want[m]) continue;
            if (!T->lit_flags.p) {
              const size_t lit_bytes = ((G.view.n_tris + 1) / 2) * 4;  // (whole 32-bit words: the kernel sets bits with atomicOr)
              if ((rc = T->lit_flags.reserve(std::max<size_t>(lit_bytes, 256)))) return rc;
              if (reuse_lit)
                RH_CUDA(cudaMemcpyAsync(T->lit_flags.p, old->lit_flags.p, T->lit_flags.bytes, cudaMemcpyDeviceToDevice, D->stream));
              else
                RH_CUDA(cudaMemsetAsync(T->lit_flags.p, 0, T->lit_flags.bytes, D->stream));
            }
            const uint32_t mask = reuse_lit && old->mesh_lit[m] ? changed : all;
            RH_CUDA((cudaError_t)device_lit_flags(d_tris, (const WideNode32*)G.wide32.p, G.view.center, occ_meshes[m],
                                                  (const uint32_t*)scratch.bufs[m].p, (uint32_t)mesh_n_slots(m),
                                                  (const rh_light*)T->lights.p, n_lights, mask, sphere_bits, (uint32_t)m,
                                                  (uint16_t*)T->lit_flags.p, (unsigned long long*)words.p + 2, D->stream));
            if (info) info->lit_queries += (uint64_t)mesh_n_slots(m) * (uint64_t)__builtin_popcount(mask & all & ~sphere_bits);
          }
          unsigned long long flagged = 0;
          RH_CUDA(cudaMemcpyAsync(&flagged, (unsigned long long*)words.p + 2, 8, cudaMemcpyDeviceToHost, D->stream));
          RH_CUDA(cudaStreamSynchronize(D->stream));
          if (flagged) v.lit_flags = (const uint16_t*)T->lit_flags.p;
          else T->lit_flags.release();
          if (n_maps) {
            if ((rc = upload(T->light_map_index, index.data(), index.size()))) return rc;
            v.light_maps = (const float*)T->light_maps.p;
            v.light_map_index = (const uint32_t*)T->light_map_index.p;
            v.light_map_res = (uint32_t)R;
          } else {
            T->light_maps.release();
          }
          T->mesh_lit = want;
        } else {
          const std::vector<WideNode>& cull = *host->cull;
          const TriVec& dtris = *host->tris;
          std::vector<float> maps, one(cells);
          std::vector<uint16_t> lit;
          size_t n_lit = 0;
          for (size_t m = 0; m < occ_meshes.size(); m++) {
            const std::vector<uint32_t> slots(mesh_slots(m), mesh_slots(m) + mesh_n_slots(m));
          // lit triangles: per triangle and light, can another triangle of this mesh shadow it at all?  The queries
          // run on their own threads while this one builds the mesh's cube maps.
          const bool want_lit = slots.size() * (size_t)n_table_lights <= kLitMaxQueries;
          if (want_lit && lit.empty()) lit.assign(dtris.size(), 0);
          size_t lit_found = 0;
          bool lit_failed = false;
          auto lit_job = [&, m]() {
            // one query per (triangle, light), independent of each other: a few host threads share the triangles
            std::atomic<size_t> next{0}, flagged{0};
            std::atomic<bool> failed{false};
            auto work = [&]() {
              std::vector<uint32_t> walk;
              size_t mine = 0;
              try {
              for (;;) {
                const size_t begin = next.fetch_add(256);
                if (begin >= slots.size()) break;
                for (size_t at = begin; at < std::min(begin + 256, slots.size()); at++) {
                  const uint32_t s0 = slots[at];
                  uint32_t bits = 0;
                  for (uint32_t li = 0; li < n_lights && li < 12; li++) {
                    if ((sphere_bits >> li) & 1u) continue;
                    rh::LitQuery q;
                    if (!rh::lit_query_make(dtris[s0], lights[li].vec, lights[li].kind == RH_LIGHT_DIRECTIONAL, &q)) continue;
                    bool blocked = false;
                    walk.assign(1, occ_meshes[m]);
                    while (!walk.empty() && !blocked) {
                      const WideNode& w = cull[walk.back()];
                      walk.pop_back();
                      for (int c = 0; c < 2 && !blocked; c++) {
                        if (w.child[c] == kEmpty || rh::lit_query_box_outside(q, w.box + 6 * c, w.box + 6 * c + 3)) continue;
                        if (w.child[c] & kLeafBit) {
                          for (uint32_t k = 0; k < (w.child[c] & kCountMask) && !blocked; k++)
                            blocked = (w.first[c] + k != s0) && rh::lit_query_tri_meets(q, dtris[w.first[c] + k]);
                        } else {
                          walk.push_back(w.child[c]);
                        }
                      }
                    }
                    if (!blocked) bits |= 1u << li;
                  }
                  lit[s0] = (uint16_t)(bits | ((uint32_t)m << 12));
                  mine += bits != 0;
                }
              }
              } catch (const std::bad_alloc&) {
                failed = true;  // (no exception may leave a thread)
              }
              flagged += mine;
            };
            const unsigned n_threads = slots.size() < 4096 ? 1u : std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
            if (n_threads == 1) {
              work();
            } else {
              try {
                std::vector<std::thread> pool;
                for (unsigned t = 0; t < n_threads; t++) pool.emplace_back(work);
                for (std::thread& t : pool) t.join();
              } catch (...) {
                failed = true;
              }
            }
            lit_failed = failed.load();
            lit_found = flagged.load();
          };
          std::thread lit_thread;
          bool maps_failed = false;
          uint32_t point_lights = 0, useful_maps = 0;
          try {
            for (uint32_t li = 0; li < n_lights; li++) {
              if (lights[li].kind != RH_LIGHT_POINT) continue;
              point_lights++;
              double empty = 0;
              if (!rh::build_light_map(lights[li].vec, dtris.data(), slots.data(), slots.size(), R, one.data(), kLightMapMinEmpty, &empty))
                continue;
              index[(size_t)li * kOccMeshes + m] = n_maps++;
              useful_maps++;
              maps.insert(maps.end(), one.begin(), one.end());
            }
          } catch (...) {
            maps_failed = true;
          }
          // (same rule as the GPU builder: no lit-triangle queries for a mesh that is a soup around its lights)
          if (want_lit && !maps_failed && (point_lights == 0 || useful_maps > 0)) lit_thread = std::thread(lit_job);
          if (lit_thread.joinable()) lit_thread.join();
          if (lit_failed || maps_failed) throw std::bad_alloc();
          n_lit += lit_found;
          }
          if (n_lit) {
            if ((rc = upload(T->lit_flags, lit.data(), lit.size()))) return rc;
            v.lit_flags = (const uint16_t*)T->lit_flags.p;
          }
          if (n_maps) {
            if ((rc = upload(T->light_maps, maps.data(), maps.size()))) return rc;
            if ((rc = upload(T->light_map_index, index.data(), index.size()))) return rc;
            v.light_maps = (const float*)T->light_maps.p;
            v.light_map_index = (const uint32_t*)T->light_map_index.p;
            v.light_map_res = (uint32_t)R;
          }
        }
        for (uint32_t x : index)
          if (x != kEmpty) T->n_light_maps = std::max(T->n_light_maps, x + 1);
        T->tables_res = (uint32_t)R;
        T->map_index_host.swap(index);
      } catch (const std::bad_alloc&) {
        return rh::set_error(RH_ERR_OOM, w + ": out of host memory");
      }
    }
  }
  T->objs_host.swap(objs);
  T->ms_light_tables = std::chrono::duration<double, std::milli>(clk::now() - t_begin).count();
  return RH_OK;
}

void scene_destroy(rh_scene* s) {
  if (!s) return;
  if (s->device && s->device->dev >= 0) cudaSetDevice(s->device->dev);
  for (DevBuf* b : {&s->wide, &s->wide32, &s->tris, &s->shade, &s->objects, &s->materials, &s->lights, &s->textures, &s->texels,
                    &s->lin_objs, &s->sphere_refs, &s->occ_planes, &s->occ_spheres, &s->occ_meshes, &s->exact_index, &s->light_maps,
                    &s->light_map_index, &s->lit_flags})
    b->release();
  delete s;
}

// ------------------------------------------------------------------ scene updates (DESIGN.md "Scene updates")
// The fields derive_tables fills: a prepared update is swapped in with them, and the old tables leave with the scratch
// scene.
void swap_tables(rh_scene& a, rh_scene& b) {
  for (auto f : {&rh_scene::objects, &rh_scene::materials, &rh_scene::lights, &rh_scene::occ_planes, &rh_scene::occ_spheres,
                 &rh_scene::occ_meshes, &rh_scene::light_maps, &rh_scene::light_map_index, &rh_scene::lit_flags})
    std::swap(a.*f, b.*f);
  std::swap(a.deep_entries, b.deep_entries);
  std::swap(a.refill_possible, b.refill_possible);
  std::swap(a.has_transparent, b.has_transparent);
  std::swap(a.has_sphere_lights, b.has_sphere_lights);
  std::swap(a.n_light_maps, b.n_light_maps);
  std::swap(a.ms_light_tables, b.ms_light_tables);
  std::swap(a.objs_host, b.objs_host);
  std::swap(a.materials_host, b.materials_host);
  std::swap(a.lights_host, b.lights_host);
  std::swap(a.tables_res, b.tables_res);
  std::swap(a.map_index_host, b.map_index_host);
  std::swap(a.mesh_lit, b.mesh_lit);
  std::swap(a.tables_on_device, b.tables_on_device);
  SceneView &x = a.view, &y = b.view;
  std::swap(x.objects, y.objects);
  std::swap(x.materials, y.materials);
  std::swap(x.lights, y.lights);
  std::swap(x.occ_planes, y.occ_planes);
  std::swap(x.occ_spheres, y.occ_spheres);
  std::swap(x.occ_meshes, y.occ_meshes);
  std::swap(x.light_maps, y.light_maps);
  std::swap(x.light_map_index, y.light_map_index);
  std::swap(x.lit_flags, y.lit_flags);
  for (auto f : {&SceneView::n_materials, &SceneView::n_lights, &SceneView::n_occ_planes, &SceneView::n_occ_spheres,
                 &SceneView::n_occ_meshes, &SceneView::shadow_fast, &SceneView::tables_in_smem, &SceneView::light_map_res})
    std::swap(x.*f, y.*f);
}

// Validates an update of S and builds its new tables into a fresh scene *out (null when nothing changed); S is not
// touched.  *cls: the update's class (scene_update.h).
int scene_update_prepare(rh_scene* S, const rh_material* materials, uint32_t n_materials, const rh_light* lights, uint32_t n_lights,
                         rh_update_info* info, const std::string& w, int* cls, std::unique_ptr<rh_scene>* out) {
  out->reset();
  *cls = rh::kUpdateNone;
  if (info) memset(info, 0, sizeof *info);
  if (n_materials != S->materials_host.size())
    return rh::set_error(RH_ERR_ARG, w + ": n_materials (" + std::to_string(n_materials) + ") differs from the scene's material count (" +
                                         std::to_string(S->materials_host.size()) + ")");
  const rh_material* mats = materials ? materials : S->materials_host.data();
  if (!lights) {
    lights = S->lights_host.data();
    n_lights = (uint32_t)S->lights_host.size();
  }
  int rc = check_tables(mats, n_materials, S->textures_host.data(), (uint32_t)S->textures_host.size(), S->n_texels, lights, n_lights, w);
  if (rc) return rc;
  std::vector<int32_t> object_material;
  try {
    for (const DObject& o : S->objs_host) object_material.push_back(o.material);
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, w + ": out of host memory");
  }
  *cls = rh::classify_update(S->materials_host.data(), mats, n_materials, S->lights_host.data(), (uint32_t)S->lights_host.size(), lights,
                             n_lights, object_material);
  if (*cls == rh::kUpdateNone) return RH_OK;
  auto N = std::make_unique<rh_scene>();
  N->device = S->device;
  if (*cls == rh::kUpdateColours) {
    // the kernels read these two tables on every call; nothing is derived from the fields that changed
    if (info) info->colours_only = 1;
    try {
      N->materials_host.assign(mats, mats + n_materials);
      N->lights_host.assign(lights, lights + n_lights);
    } catch (const std::bad_alloc&) {
      return rh::set_error(RH_ERR_OOM, w + ": out of host memory");
    }
    RH_CUDA(cudaSetDevice(S->device->dev));
    if ((rc = upload(N->materials, mats, n_materials)) || (rc = upload(N->lights, lights, n_lights))) {
      scene_destroy(N.release());
      return rc;
    }
  } else {
    if (info) info->occluders_rebuilt = *cls == rh::kUpdateEmitters;
    rc = derive_tables(S->device, *S, mats, n_materials, lights, n_lights, nullptr, *cls == rh::kUpdateTables ? S : nullptr, N.get(),
                       info, w);
    if (rc) {
      scene_destroy(N.release());
      return rc;
    }
  }
  *out = std::move(N);
  return RH_OK;
}

// Swaps a prepared update in and releases the old tables.  Frames after a change of the light tables or the occluders
// cast other rays, so the scene's learned state (shadow schedule, queue factor, row costs) starts over as a fresh scene's.
void scene_update_commit(rh_scene* S, std::unique_ptr<rh_scene> N, int cls) {
  if (!N) return;
  if (cls == rh::kUpdateColours) {
    std::swap(S->materials, N->materials);
    std::swap(S->lights, N->lights);
    std::swap(S->materials_host, N->materials_host);
    std::swap(S->lights_host, N->lights_host);
    S->view.materials = (const rh_material*)S->materials.p;
    S->view.lights = (const rh_light*)S->lights.p;
  } else {
    swap_tables(*S, *N);
    S->shadow_mode = 0;
    S->tune_frames = S->tune_small_frames = 0;
    S->tune_ns_per_pair[0] = S->tune_ns_per_pair[1] = 0;
    S->cost_key.clear();
    S->row_cost.clear();
    S->queue_factor = S->views_queue_factor = 2;
    S->stream_compute_bound = false;
  }
  S->generation++;
  scene_destroy(N.release());
}

// ------------------------------------------------------------------ camera (Projection.hs:22-46, Mat.hs:83-93)
struct HV { double x, y, z; };
HV hsub(HV a, HV b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
HV hcross(HV a, HV b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
HV hnormalize(HV v) {
  double s = 1 / std::sqrt(v.x * v.x + v.y * v.y + v.z * v.z);
  return {s * v.x, s * v.y, s * v.z};
}

CameraParams make_camera(const rh_camera& c, int width, int height) {
  CameraParams p{};
  const double w = (double)width, h = (double)height;
  HV pos{c.position[0], c.position[1], c.position[2]}, tgt{c.target[0], c.target[1], c.target[2]}, tup{c.up[0], c.up[1], c.up[2]};
  HV forward = hnormalize(hsub(tgt, pos));      // Mat.hs:89-93
  HV right = hnormalize(hcross(tup, forward));
  HV up = hcross(forward, right);
  // fromColumns right up forward (Mat.hs:83-87), row-major
  p.m[0] = right.x; p.m[1] = up.x; p.m[2] = forward.x;
  p.m[3] = right.y; p.m[4] = up.y; p.m[5] = forward.y;
  p.m[6] = right.z; p.m[7] = up.z; p.m[8] = forward.z;
  p.pos[0] = pos.x; p.pos[1] = pos.y; p.pos[2] = pos.z;
  p.w = w;
  p.h = h;
  p.half_w = w / 2;
  p.half_h = h / 2;
  const double aspect = w / h;  // aspectSize, Projection.hs:41-46
  if (aspect > 1) { p.apw = w; p.aph = w / aspect; }
  else { p.apw = aspect * h; p.aph = h; }
  p.f = 0.5 * h / (std::tan(0.5) * c.fovy);  // Projection.hs:35 — `tan 0.5 * fovy` (SURVEY App. A-C1)
  // a lens of radius 0 casts the perspective rays bit for bit (rh_camera), so the kernels take the pinhole path for it
  p.projection = (c.projection == RH_PROJ_THIN_LENS && c.proj_width == 0) ? RH_PROJ_PERSPECTIVE : c.projection;
  if (p.projection == RH_PROJ_THIN_LENS) {
    p.lens_r = c.proj_width;
    p.focus = c.proj_height;
  }
  return p;
}

// A camera's argument checks: "" when its projection is known and, for RH_PROJ_THIN_LENS, its R, F and fovy are valid,
// else what is wrong
std::string camera_error(const rh_camera& c) {
  if (c.projection != RH_PROJ_ORTHOGRAPHIC && c.projection != RH_PROJ_PERSPECTIVE && c.projection != RH_PROJ_THIN_LENS)
    return "unknown projection";
  if (c.projection != RH_PROJ_THIN_LENS) return "";
  if (!std::isfinite(c.proj_width) || !(c.proj_width >= 0)) return "thin-lens aperture radius proj_width must be finite and >= 0";
  if (!std::isfinite(c.proj_height) || !(c.proj_height > 0)) return "thin-lens focus distance proj_height must be finite and > 0";
  if (!std::isfinite(c.fovy) || !(c.fovy > 0)) return "thin-lens fovy must be finite and > 0";
  return "";
}

// ------------------------------------------------------------------ render
// One validated frame for run_frame: a render (rh_render, one shard of rh_multi_render) or the ray frame of
// rh_trace_rays.
struct Frame {
  rh_render_opts o{};        // shard_count and band_height resolved
  CameraParams cam{};        // (renders)
  uint8_t* out = nullptr;    // RGB8 rows, or (trace) the colours as double[n_rays][3]; null with RH_FLAG_PEER_FRAMES
  int32_t* ids_out = nullptr;
  size_t out_bytes = 0, ids_bytes = 0;
  int rows_local = 0;
  size_t off_elem = 0;       // bytes per pass-0 item of o.offsets
  uint64_t rays_primary = 0;
  // rh_trace_rays: pass 0 reads n_rays caller-built rays (the last row may be partial), the colours leave unquantised,
  // and the scene's learned state (shadow-schedule tuning, queue factor, row costs) is neither used nor changed
  bool trace = false;
  uint64_t n_rays = 0;
  // RH_OFFSETS_SPLITMIX64: the stream's samples per pixel and the first of them this frame traces
  uint32_t stream_spp = 0, stream_base = 0;
  // rh_render_adaptive: pass 0 traces o.spp samples of each entry of a list of pixels (n_rays items; the frame's rows are
  // rows of the list, the last one may be partial), the sink stages the entries' new sums (ad), and the scene's learned
  // state is used but not changed
  bool pixel_list = false;
  PixelList list{};
  AdaptiveParams ad{};
  // rh_render_accumulate: the sink adds the samples to the accumulator's sums (read sum_in, write sum_out) and writes
  // RGB8 to `out` and the linear colours to `linear`, either of them optional
  bool accumulate = false;
  AccumParams acc{};
  double* linear = nullptr;
  size_t linear_bytes = 0;
  // rh_render_light_groups: the shadow kernels also add each group's terms, and a sink beside the resolve writes the
  // group images to group_out (device, or host through a chunk of scratch); RGB8 is optional
  uint32_t n_groups = 0;
  uint32_t group_mask[kMaxGroups] = {};
  double* group_out = nullptr;
  // rh_render_views: the local rows are [view][view_rows]; pass 0 takes each view's camera from cams (device) and, with
  // view_seeds (device), its SplitMix64 seed; the sink decides padding rows per view and writes RGB8 (optional) and the
  // linear colours (`linear`, optional).  Device offsets are read from the start of the array for every view.
  bool views = false;
  uint32_t view_rows = 0;
  const CameraParams* cams = nullptr;
  const unsigned long long* view_seeds = nullptr;
  // host data the kernels read, copied to the device at the start of each attempt (rh_render_views: the camera table,
  // the seeds and host per-pixel offsets)
  struct Upload { void* dst; const void* src; size_t bytes; };
  std::vector<Upload> uploads;
  const char* who = "rh_render";  // the entry point, in run_frame's messages
  // renders (not traces, list frames, light-group or views frames) tune the scene's shadow schedule and record its queue
  // factor and row costs
  bool learns() const { return !trace && !pixel_list && !n_groups && !views; }
};

// rh_render's argument checks (`who` names the entry point in the messages).  rgb_out may be null: each entry point
// decides which of its outputs it needs.
int render_frame(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, uint8_t* rgb_out,
                 int32_t* hit_ids_out, Frame* f, const char* who = "rh_render") {
  const std::string w(who);
  if (!scene || !camera || !o) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  const bool peer_frames = (o->flags & RH_FLAG_PEER_FRAMES) != 0;
  if (peer_frames && (!o->peer_frames || o->n_peer_frames <= 0 || o->n_peer_frames > kMaxPeers))
    return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_PEER_FRAMES needs 1..16 peer frame pointers");
  if (peer_frames && (o->flags & RH_FLAG_HIT_IDS))
    return rh::set_error(RH_ERR_ARG, w + ": hit ids are not exchanged; render them without RH_FLAG_PEER_FRAMES");
  if (scene->device != D) return rh::set_error(RH_ERR_ARG, w + ": scene lives on another device context");
  const int W = o->width, H = o->height, spp = o->spp;
  if (W <= 0 || H <= 0 || spp <= 0 || o->max_depth < 0 || o->max_depth > kMaxDepth)
    return rh::set_error(RH_ERR_ARG, w + ": bad width/height/spp/max_depth");
  const std::string cam_err = camera_error(*camera);
  if (!cam_err.empty()) return rh::set_error(RH_ERR_ARG, w + ": " + cam_err);
  const int G = o->shard_count <= 0 ? 1 : o->shard_count;
  if (o->shard_index < 0 || o->shard_index >= G) return rh::set_error(RH_ERR_ARG, w + ": shard_index out of range");
  const int bh = o->band_height > 0 ? o->band_height : rh_default_band_height(H, G);
  const int mode = o->offset_mode;
  if (mode < RH_OFFSETS_NONE || mode > RH_OFFSETS_SPLITMIX64) return rh::set_error(RH_ERR_ARG, w + ": bad offset_mode");
  if (mode != RH_OFFSETS_NONE && !o->offsets) return rh::set_error(RH_ERR_ARG, w + ": offsets is null");
  if (mode == RH_OFFSETS_TILED_F64 && o->offset_tile <= 0) return rh::set_error(RH_ERR_ARG, w + ": offset_tile must be > 0");
  if ((uint64_t)W * spp > 0x7fffffffu) return rh::set_error(RH_ERR_ARG, w + ": row too large");
  if ((o->flags & RH_FLAG_HIT_IDS) && !hit_ids_out) return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_HIT_IDS without hit_ids_out");
  if (mode == RH_OFFSETS_SPLITMIX64 && (o->flags & RH_FLAG_DEVICE_OFFSETS))
    return rh::set_error(RH_ERR_ARG, w + ": RH_OFFSETS_SPLITMIX64 takes a host pointer to the seed");
  f->who = who;
  f->o = *o;
  f->o.shard_count = G;
  f->o.band_height = bh;
  f->cam = make_camera(*camera, W, H);
  f->out = rgb_out;
  f->ids_out = hit_ids_out;
  f->stream_spp = (uint32_t)spp;
  f->stream_base = 0;
  f->rows_local = rh_shard_rows(H, G, bh);
  f->out_bytes = (size_t)f->rows_local * W * 3;
  f->ids_bytes = (size_t)f->rows_local * W * spp * sizeof(int2);
  f->off_elem = (mode == RH_OFFSETS_F32) ? sizeof(float) * 2 : sizeof(double) * 2;
  for (int lr = 0; lr < f->rows_local; lr++)  // padding rows of the last band trace nothing
    if (((long long)(lr / bh) * G + o->shard_index) * bh + lr % bh < H) f->rays_primary += (uint64_t)W * spp;
  return RH_OK;
}

// Shadow-walk schedule of a frame: forced by flags, else the scene's measured choice, else — on frames large enough to
// time — one of the scene's timing frames: the first is pooled and not compared (first use of freshly allocated queues),
// the second pooled, the third per-lane refill; the two kernels' times per walked (hit, light) pair are compared.  Small
// frames never take part: they run pooled, unprofiled, and after kTuneGiveUp of them the scene stays pooled.  A trace
// or a list frame uses the scene's decided schedule and takes no part in the tuning.
constexpr int kTuneGiveUp = 8;
struct ShadowChoice {
  bool use_refill = false;
  bool untuned = false;  // the schedule is neither forced nor decided: the frame counts towards the tuning
  bool tuning = false;   // ... and is one of the timing frames
  bool profile = false;  // every launch is timed on its own
};

ShadowChoice choose_shadow(const rh_scene* scene, const Frame& f) {
  const int32_t flags = f.o.flags;
  const bool refill_ok = scene->refill_possible && scene->view.n_lights <= (uint32_t)kMaskLights;
  if (f.learns() && !refill_ok && scene->shadow_mode == 0) scene->shadow_mode = 1;
  const bool forced = (flags & (RH_FLAG_SHADOW_POOLED | RH_FLAG_SHADOW_SPLIT)) != 0;
  const bool decided = scene->shadow_mode != 0;
  ShadowChoice c;
  c.untuned = f.learns() && !forced && !decided && !(flags & RH_FLAG_COUNT);
  c.tuning = c.untuned && (uint64_t)f.rows_local * f.o.width * f.o.spp >= (1ull << 21);
  if (flags & RH_FLAG_SHADOW_SPLIT) c.use_refill = refill_ok;
  else if (flags & RH_FLAG_SHADOW_POOLED) c.use_refill = false;
  else if (decided) c.use_refill = scene->shadow_mode == 2;
  else if (c.tuning) c.use_refill = scene->tune_frames == 2;
  c.profile = (flags & RH_FLAG_PROFILE) != 0 || c.tuning;
  return c;
}

struct Span { cudaEvent_t a, b; int kind; };  // a timed launch: 0 trace, 1 shadow kernels, 2 resolve / store

// Copies the host sample offsets of the frame's local rows [first_row, first_row + n_rows) to `slot` in work-item order:
// one copy per run of image rows that are contiguous inside one band, none for padding rows.  A trace frame's last row
// may be partial.  Adds the bytes copied to *bytes.
int upload_offset_rows(const Frame& f, size_t row_samples, int first_row, int n_rows, char* slot, cudaStream_t stream, size_t* bytes) {
  const rh_render_opts& o = f.o;
  const int bh = o.band_height;
  int lr = first_row;
  while (lr < first_row + n_rows) {
    const int lb = lr / bh, rib = lr % bh;
    const int run = std::min(bh - rib, first_row + n_rows - lr);
    const long long grow = ((long long)lb * o.shard_count + o.shard_index) * bh + rib;
    const long long rows_ok = std::max<long long>(0, std::min<long long>(run, (long long)o.height - grow));
    if (rows_ok > 0) {
      const size_t src_row = (o.flags & RH_FLAG_SHARD_OFFSETS) ? (size_t)lr : (size_t)grow;
      size_t n = (size_t)rows_ok * row_samples * f.off_elem;
      if (f.trace) n = std::min(n, ((size_t)f.n_rays - src_row * row_samples) * f.off_elem);  // (a partial last row)
      RH_CUDA(cudaMemcpyAsync(slot + (size_t)(lr - first_row) * row_samples * f.off_elem,
                              (const char*)o.offsets + src_row * row_samples * f.off_elem, n, cudaMemcpyHostToDevice, stream));
      *bytes += n;
    }
    lr += run;
  }
  return RH_OK;
}

// The chunk parameters that follow from the frame alone and are the same for every chunk of it, whichever kernels
// (run_frame's or rh_render_features's) take them.
ChunkParams frame_chunk_params(const Frame& f) {
  const rh_render_opts& o = f.o;
  ChunkParams P{};
  P.spp = o.spp;
  P.width = o.width;
  P.height = o.height;
  P.shard_index = o.shard_index;
  P.shard_count = o.shard_count;
  P.band_height = o.band_height;
  P.offset_mode = o.offset_mode;
  P.offset_tile = o.offset_tile;
  if (o.offset_mode == RH_OFFSETS_SPLITMIX64) memcpy(&P.offset_seed, o.offsets, sizeof P.offset_seed);
  P.stream_spp = f.stream_spp;
  P.stream_base = f.stream_base;
  if (o.flags & RH_FLAG_PEER_FRAMES) {
    P.n_peers = (uint32_t)o.n_peer_frames;
    for (int g = 0; g < o.n_peer_frames; g++) P.peer[g] = (uint8_t*)o.peer_frames[g];
  }
  P.list = f.list;
  P.cams = f.cams;
  P.view_seeds = f.view_seeds;
  P.view_rows = f.view_rows;
  return P;
}

// One frame on one device: its plan and buffers, and what the enqueued chunks recorded.
struct FrameRun {
  Device* D;
  const rh_scene* scene;
  const Frame& f;
  ShadowChoice sh;
  rh::ChunkPlan plan;
  size_t row_samples = 0, chunk_samples = 0;  // chunk_samples: the largest chunk's
  int n_chunks = 0, n_passes = 0, n_lanes = 1;
  bool counting = false, host_offsets = false, pipelined = false;
  uint8_t* d_rgb = nullptr;
  int2* d_ids = nullptr;
  double* d_linear = nullptr;
  // light-group frames: where the group sink writes (the caller's device buffer, else the lane's chunk of scratch), and
  // the doubles between two group images there
  bool group_out_dev = false;
  size_t group_out_stride = 0;
  const void* d_offsets = nullptr;
  int off_index = kOffIndexLocal;
  int ring = 2;                  // slots of the offset upload ring
  size_t cap = 0, walk_cap = 0;  // queue capacities in entries
  // recorded by the enqueue, per attempt
  uint32_t launches = 0;
  size_t upload_bytes = 0, ev_used = 0;
  std::vector<Span> spans;
  std::vector<cudaEvent_t> chunk_ev, copy_ev;  // streamed offsets: per chunk its kernels' begin and end, its upload's end

  cudaEvent_t prof_event(cudaStream_t stream) {
    if (ev_used == D->prof_events.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      D->prof_events.push_back(e);
    }
    cudaEvent_t e = D->prof_events[ev_used++];
    cudaEventRecord(e, stream);
    return e;
  }
  const ChunkCtl* ctl() const { return (const ChunkCtl*)D->pinned; }
  const FrameCounters* counters() const { return (const FrameCounters*)((const char*)D->pinned + (size_t)n_chunks * sizeof(ChunkCtl)); }

  // Queue capacity in entries, a whole number of slabs: factor x the chunk's samples, plus one partly filled slab per
  // warp that can be producing (each warp leaves its last slab of a queue open).
  int reserve_queues(uint32_t factor) {
    const size_t producers = std::min<size_t>((size_t)D->max_threads / 32, (chunk_samples + kSlab - 1) / kSlab + 1);
    cap = std::min<size_t>((size_t)factor * chunk_samples + 2 * producers * kSlab, 0x7fffff00u);
    cap = (cap + kSlab - 1) / kSlab * kSlab;
    const size_t n_slabs_cap = cap / kSlab;
    walk_cap = std::max<size_t>((cap / 2 + kSlab - 1) / kSlab * kSlab, 2 * producers * kSlab);
    const size_t deep_bytes = (size_t)scene->deep_entries * D->max_threads * sizeof(uint2);
    int rc;
    for (int l = 0; l < n_lanes; l++) {
      Device::Scratch& sc = D->lane[l];
      for (int k = 0; k < 2; k++) {
        if ((rc = sc.rayq[k].reserve(cap * 4 * sizeof(double2)))) return rc;
        if ((rc = sc.rayq_fill[k].reserve(n_slabs_cap * sizeof(uint32_t)))) return rc;
      }
      // hit queue (every shaded hit of a pass) and walk queue (the hits that need a tree walk: half as many entries)
      if ((rc = sc.hitq.reserve(cap * 5 * sizeof(double2)))) return rc;
      if ((rc = sc.hitq_words.reserve((2 * cap + n_slabs_cap) * sizeof(uint32_t)))) return rc;  // sample ids, lit flags, slab fills
      if ((rc = sc.shq.reserve(walk_cap * 5 * sizeof(double2)))) return rc;
      if ((rc = sc.shq_words.reserve((3 * walk_cap + walk_cap / kSlab) * sizeof(uint32_t)))) return rc;  // sample ids, walk masks, settled masks, slab fills
      if ((rc = sc.deep.reserve(deep_bytes))) return rc;
      if (pipelined && (rc = sc.deep_shadow.reserve(deep_bytes))) return rc;  // (kernels of both streams run side by side)
    }
    return RH_OK;
  }

  // Enqueues the chunk processed i-th: its offset upload (streamed offsets), its passes and its resolve.
  int enqueue_chunk(int i) {
    const rh_render_opts& o = f.o;
    const int ck = plan.order[i], first_row = plan.first_row[ck], n_rows = plan.rows[ck];
    const int ln = i % n_lanes;
    Device::Scratch& sc = D->lane[ln];
    const cudaStream_t lane_stream = ln ? D->stream2 : D->stream;
    double* group_out = group_out_dev ? f.group_out : (double*)sc.group_out.p;
    ChunkParams P = frame_chunk_params(f);
    P.first_row = first_row;
    P.n_rows = n_rows;
    P.n_samples = (uint32_t)((size_t)n_rows * row_samples);
    P.max_depth = o.max_depth;
    P.exact_boxes = (o.flags & RH_FLAG_EXACT_BOXES) ? 1 : 0;
    P.no_light_maps = (o.flags & RH_FLAG_NO_LIGHT_MAPS) ? 1 : 0;
    P.offset_index = off_index;
    P.offsets = d_offsets;
    P.accum = (double*)sc.accum.p;
    P.accum_stride = (uint32_t)chunk_samples;
    P.hit_ids = d_ids;
    P.rgb = d_rgb;
    P.ctl = (ChunkCtl*)D->ctl.p + ck;
    P.counters = (FrameCounters*)D->counters.p;
    P.q_hits.plane = (double2*)sc.hitq.p;
    P.q_hits.sample = (uint32_t*)sc.hitq_words.p;
    P.q_hits.walk = (uint32_t*)sc.hitq_words.p + cap;
    P.q_hits.settled = nullptr;
    P.q_hits.fill = (uint32_t*)sc.hitq_words.p + 2 * cap;
    P.q_hits.capacity = (uint32_t)cap;
    P.q_shadow.plane = (double2*)sc.shq.p;
    P.q_shadow.sample = (uint32_t*)sc.shq_words.p;
    P.q_shadow.walk = (uint32_t*)sc.shq_words.p + walk_cap;
    P.q_shadow.settled = (uint32_t*)sc.shq_words.p + 2 * walk_cap;
    P.q_shadow.fill = (uint32_t*)sc.shq_words.p + 3 * walk_cap;
    P.q_shadow.capacity = (uint32_t)walk_cap;
    P.deep_stack = (uint2*)sc.deep.p;
    P.deep_stride = (uint32_t)D->max_threads;

    if (host_offsets) {
      // upload this chunk's rows on the copy stream
      const int b = i % ring;
      char* slot = (char*)D->offsets.p + (size_t)b * chunk_samples * f.off_elem;
      if (i >= ring) RH_CUDA(cudaStreamWaitEvent(D->copy_stream, D->ev_done[b], 0));
      const int rc = upload_offset_rows(f, row_samples, first_row, n_rows, slot, D->copy_stream, &upload_bytes);
      if (rc) return rc;
      RH_CUDA(cudaEventRecord(D->ev_up[b], D->copy_stream));
      copy_ev.push_back(prof_event(D->copy_stream));  // (when each chunk's upload ended)
      RH_CUDA(cudaStreamWaitEvent(lane_stream, D->ev_up[b], 0));
      P.offsets = slot;
      chunk_ev.push_back(prof_event(lane_stream));  // after the wait: the span holds kernel time only
    }

    if ((o.flags & RH_FLAG_DEVICE_OFFSETS) && (o.flags & RH_FLAG_SHARD_OFFSETS) && d_offsets && !f.views)
      P.offsets = (const char*)d_offsets + (size_t)first_row * row_samples * f.off_elem;
    P.offset_base = (P.offset_index == kOffIndexLocal) ? 0ull : (unsigned long long)first_row * row_samples;
    if (f.trace || f.pixel_list) P.ray_items = (uint32_t)std::min<uint64_t>(P.n_samples, f.n_rays - (uint64_t)first_row * row_samples);
    for (int plane = 0; plane < 3; plane++)  // (three 1-D memsets: a 2-D one is limited to 2 GB of pitch)
      RH_CUDA(cudaMemsetAsync((double*)sc.accum.p + (size_t)plane * chunk_samples, 0, (size_t)P.n_samples * sizeof(double), lane_stream));
    if (f.n_groups) {
      P.groups = (double*)sc.groups.p;
      P.group_stride = (uint32_t)chunk_samples;
      P.n_groups = f.n_groups;
      memcpy(P.group_mask, f.group_mask, sizeof P.group_mask);
      // the 3 (n_groups + 1) planes follow each other: one memset up to the last plane's n_samples
      RH_CUDA(cudaMemsetAsync(P.groups, 0, ((size_t)(3 * f.n_groups + 2) * chunk_samples + P.n_samples) * sizeof(double), lane_stream));
    }
    const cudaStream_t shadow_stream = pipelined ? D->shadow_stream[ln] : lane_stream;
    for (int pass = 0; pass < n_passes; pass++) {
      P.pass = pass;
      P.q_in.plane = (double2*)sc.rayq[(pass + 1) & 1].p;
      P.q_in.fill = (uint32_t*)sc.rayq_fill[(pass + 1) & 1].p;
      P.q_in.capacity = (uint32_t)cap;
      P.q_out.plane = (double2*)sc.rayq[pass & 1].p;
      P.q_out.fill = (uint32_t*)sc.rayq_fill[pass & 1].p;
      P.q_out.capacity = (uint32_t)cap;  // (the last pass cannot emit: every ray in it has depth == maxDepth)
      cudaEvent_t a = nullptr;
      if (sh.profile) a = prof_event(lane_stream);
      P.deep_stack = (uint2*)sc.deep.p;
      P.hit_live_pass = (pipelined && pass > 0) ? pass - 1 : pass;
      if (pipelined && pass >= 2) RH_CUDA(cudaStreamWaitEvent(lane_stream, D->ev_classified[ln][pass - 2], 0));  // its slabs are free
      launch_trace(scene->view, f.cam, P, counting, D->n_sms, lane_stream);
      if (sh.profile) { cudaEvent_t b2 = prof_event(lane_stream); spans.push_back({a, b2, 0}); a = b2; }
      if (pipelined) {
        RH_CUDA(cudaEventRecord(D->ev_trace[ln][pass], lane_stream));
        RH_CUDA(cudaStreamWaitEvent(shadow_stream, D->ev_trace[ln][pass], 0));
        P.deep_stack = (uint2*)sc.deep_shadow.p;
      }
      const int n_shadow = launch_shadow(scene->view, P, counting, sh.use_refill, D->n_sms, shadow_stream,
                                         pipelined ? (void*)D->ev_classified[ln][pass] : nullptr, scene->has_sphere_lights);
      if (sh.profile) spans.push_back({a, prof_event(lane_stream), 1});
      launches += 2 + n_shadow;  // (trace, the one-thread kernel that closes its hit range, classify, walk)
    }
    if (pipelined) {  // the resolve kernel needs every pass's shadow terms
      RH_CUDA(cudaEventRecord(D->ev_shadows[ln], shadow_stream));
      RH_CUDA(cudaStreamWaitEvent(lane_stream, D->ev_shadows[ln], 0));
    }
    cudaEvent_t a = nullptr;
    if (sh.profile) a = prof_event(lane_stream);
    if (f.trace) {
      launch_store_colors(P, (double*)d_rgb, lane_stream);
    } else if (f.accumulate) {
      AccumParams A = f.acc;
      A.linear = d_linear;
      launch_accumulate_resolve(P, A, lane_stream);
    } else if (f.pixel_list) {
      launch_adaptive_fold(P, f.ad, lane_stream);
    } else if (f.views) {
      launch_views_resolve(P, d_linear, lane_stream);
    } else if (!f.n_groups) {
      launch_resolve(P, lane_stream);
    } else {
      if (d_rgb) {  // (a light-group frame without RGB8 output has no use for the resolve)
        launch_resolve(P, lane_stream);
        launches += 1;
      }
      launch_light_groups_resolve(P, group_out, group_out_stride, group_out_dev ? (size_t)first_row * o.width : 0, lane_stream);
    }
    if (sh.profile) spans.push_back({a, prof_event(lane_stream), 2});
    launches += 1;
    if (f.n_groups && !group_out_dev) {  // host output: the chunk's rows of every group image
      const size_t plane = (size_t)f.rows_local * o.width * 3, at = (size_t)first_row * o.width * 3;
      for (uint32_t g = 0; g <= f.n_groups; g++)
        RH_CUDA(cudaMemcpyAsync(f.group_out + g * plane + at, group_out + g * group_out_stride, (size_t)n_rows * o.width * 3 * sizeof(double),
                                cudaMemcpyDeviceToHost, lane_stream));
    }
    if (host_offsets) {
      RH_CUDA(cudaEventRecord(D->ev_done[i % ring], lane_stream));
      chunk_ev.push_back(prof_event(lane_stream));
    }
    return RH_OK;
  }

  void read_stats(rh_stats* stats, uint32_t factor) const;
  void print_timeline() const;
  void learn() const;
};

// RAYS_B200_DEBUG output of a counting frame (and, built with RH_WARP_TIMES, of the pooled walks' warp times).
void print_debug_counters(const FrameCounters* fc, bool counting) {
  if (counting && getenv("RAYHS_B200_DEBUG"))
    fprintf(stderr, "rayhs_b200: exact shadow walks %llu, most nodes visited by one shadow ray %llu; exact closest-hit walks %llu, "
            "most nodes visited by one closest-hit ray %llu\n", fc->exact_walks, fc->max_walk_nodes, fc->exact_closest,
            fc->max_closest_nodes);
  if (counting && getenv("RAYHS_B200_DEBUG"))
    for (int row = 0; row < 4; row++) {
      fprintf(stderr, "rayhs_b200: shadow walks of pass %d%s by log2(nodes + 1) [walks / nodes]:", row, row == 3 ? "+" : "");
      for (int b = 0; b < 20; b++)
        if (fc->walk_hist[row][b]) fprintf(stderr, " %d:%llu/%llu", b, fc->walk_hist[row][b], fc->walk_hist_nodes[row][b]);
      fprintf(stderr, "\n");
    }
#ifdef RH_WARP_TIMES
  if (getenv("RAYHS_B200_DEBUG"))
    for (int row = 0; row < 4; row++) {
      std::vector<int> b, e;
      unsigned long long tot_b = 0, tot_r = 0;
      int slow = -1, slow_end = 0;
      unsigned ref = 0;
      for (int i = 0; i < 4096; i++)
        if (fc->warp_end[row][i]) {
          if (b.empty()) ref = fc->warp_begin[row][i];
          b.push_back((int)(fc->warp_begin[row][i] - ref));
          e.push_back((int)(fc->warp_end[row][i] - ref));
          tot_b += fc->warp_batches[row][i];
          tot_r += fc->warp_rounds[row][i];
          if (slow < 0 || e.back() > slow_end) { slow = i; slow_end = e.back(); }
        }
      if (b.empty()) continue;
      std::sort(b.begin(), b.end());
      std::sort(e.begin(), e.end());
      const int t0 = b.front();
      fprintf(stderr, "rayhs_b200: pooled pass %d: %zu warps, %llu batches, %llu rounds; warp start (us after the first) p50 %.1f p99 %.1f max %.1f; "
              "warp end p1 %.1f p10 %.1f p50 %.1f p90 %.1f p99 %.1f max %.1f; slowest warp: %u batches %u rounds\n", row, b.size(), tot_b, tot_r,
              (b[b.size() / 2] - t0) / 1e3, (b[b.size() * 99 / 100] - t0) / 1e3, (b.back() - t0) / 1e3, (e[e.size() / 100] - t0) / 1e3,
              (e[e.size() / 10] - t0) / 1e3, (e[e.size() / 2] - t0) / 1e3, (e[e.size() * 9 / 10] - t0) / 1e3, (e[e.size() * 99 / 100] - t0) / 1e3,
              (e.back() - t0) / 1e3, fc->warp_batches[row][slow], fc->warp_rounds[row][slow]);
      std::vector<std::pair<int, int>> by_end;
      for (int i = 0; i < 4096; i++)
        if (fc->warp_end[row][i]) by_end.push_back({(int)(fc->warp_end[row][i] - ref) - t0, i});
      std::sort(by_end.rbegin(), by_end.rend());
      fprintf(stderr, "rayhs_b200:   slowest warps (block.warp end-us batches rounds pairs walk-us sum-of-longest-lane nodes tris):");
      for (size_t k = 0; k < 10 && k < by_end.size(); k++) {
        const int i = by_end[k].second;
        fprintf(stderr, " %d.%d %.0f %u %u %u %.0f %u %u |", i / 24, i % 24, by_end[k].first / 1e3, fc->warp_batches[row][i], fc->warp_rounds[row][i],
                fc->warp_pairs[row][i], fc->warp_walk_ns[row][i] / 1e3, fc->warp_max_nodes[row][i], fc->warp_max_tris[row][i]);
      }
      fprintf(stderr, "\n");
      {
        const int i = by_end[by_end.size() / 2].second;
        fprintf(stderr, "rayhs_b200:   median warp: %d.%d %.0f %u %u %u %.0f %u %u\n", i / 24, i % 24, by_end[by_end.size() / 2].first / 1e3,
                fc->warp_batches[row][i], fc->warp_rounds[row][i], fc->warp_pairs[row][i], fc->warp_walk_ns[row][i] / 1e3,
                fc->warp_max_nodes[row][i], fc->warp_max_tris[row][i]);
      }
    }
#endif
}

void FrameRun::read_stats(rh_stats* stats, uint32_t factor) const {
  memset(stats, 0, sizeof *stats);
  const FrameCounters* fc = counters();
  const uint64_t shadow_tasks = fc->shaded_hits;
  uint64_t queued_hits = 0;
  for (int ck = 0; ck < n_chunks; ck++)
    for (int p = 0; p < n_passes; p++) queued_hits += ctl()[ck].shadow_items[p];
  stats->rays_primary = f.rays_primary;
  stats->rays_reflect = fc->rays_reflect;
  stats->rays_probe = fc->rays_probe;
  stats->rays_exit = fc->rays_exit;
  stats->rays_shadow = shadow_tasks * scene->view.n_lights;  // one shadowIntersection per light (RayHs.hs:89-97)
  stats->box_tests = fc->k[0].box_tests;
  stats->tri_tests = fc->k[0].tri_tests;
  stats->prim_tests = fc->k[0].prim_tests;
  stats->shade_fetches = fc->k[0].shade_fetches;
  stats->texel_fetches = fc->k[0].texel_fetches;
  stats->node_visits = fc->k[0].node_visits;
  stats->node_visits_global = fc->k[0].global_node_visits;
  stats->shadow_node_visits_global = fc->k[1].global_node_visits;
  stats->tri_records = fc->k[0].tri_records;
  stats->shadow_tri_records = fc->k[1].tri_records;
  stats->shadow_box_tests = fc->k[1].box_tests;
  stats->shadow_tri_tests = fc->k[1].tri_tests;
  stats->shadow_prim_tests = fc->k[1].prim_tests;
  stats->shadow_node_visits = fc->k[1].node_visits;
  for (int ck = 0; ck < n_chunks; ck++)
    for (int p = 1; p < n_passes; p++) stats->queued_rays += ctl()[ck].ray_items[p];
  stats->shadow_tasks = shadow_tasks;
  stats->shadow_tasks_queued = queued_hits;
  stats->shadow_walk_pairs = fc->shadow_walk_pairs;
  stats->deep_stack_pushes = fc->deep_pushes;
  stats->rays_shadow_culled = fc->shadow_culled;
  print_debug_counters(fc, counting);
  stats->upload_bytes = upload_bytes;
  float ms = 0;
  cudaEventElapsedTime(&ms, D->ev_begin, D->ev_end);
  stats->ms_total = ms;
  for (const Span& s : spans) {
    float m = 0;
    cudaEventElapsedTime(&m, s.a, s.b);
    if (s.kind == 0) { stats->ms_trace += m; stats->trace_launches++; }
    else if (s.kind == 1) { stats->ms_shadow += m; stats->shadow_launches++; }
    else stats->ms_resolve += m;
  }
  stats->kernel_launches = launches;
  stats->chunks = (uint32_t)n_chunks;
  stats->negative_channels = (uint32_t)std::min<unsigned long long>(fc->negative_channels, 0xffffffffu);
  stats->queue_factor = factor;
  stats->shadow_split = sh.use_refill ? 1 : 0;
}

// RAYHS_B200_DEBUG=t: the timeline of a streamed frame.
void FrameRun::print_timeline() const {
  static const bool debug_timeline = getenv("RAYHS_B200_DEBUG") && strchr(getenv("RAYHS_B200_DEBUG"), 't');
  if (!debug_timeline || (int)copy_ev.size() != n_chunks || (int)chunk_ev.size() != 2 * n_chunks) return;
  float end_ms = 0;
  cudaEventElapsedTime(&end_ms, D->ev_begin, D->ev_end);
  fprintf(stderr, "rayhs_b200: streamed frame, %d chunks, %.2f ms; per chunk in processing order: rows, upload done, kernels begin, kernels end (ms)\n", n_chunks, end_ms);
  for (int i = 0; i < n_chunks; i++) {
    float up = 0, kb = 0, ke = 0;
    cudaEventElapsedTime(&up, D->ev_begin, copy_ev[i]);
    cudaEventElapsedTime(&kb, D->ev_begin, chunk_ev[2 * i]);
    cudaEventElapsedTime(&ke, D->ev_begin, chunk_ev[2 * i + 1]);
    fprintf(stderr, "rayhs_b200:   chunk %2d lane %d rows %4d  up %6.2f  begin %6.2f  end %6.2f\n", plan.order[i], i % n_lanes,
            plan.rows[plan.order[i]], up, kb, ke);
  }
}

// The scene's learned state after a render: the row costs and the compute-bound flag of a streamed frame with the
// default chunk plan, and the shadow-schedule tuning.
void FrameRun::learn() const {
  const rh_render_opts& o = f.o;
  if (host_offsets && o.chunk_samples <= 0 && (int)chunk_ev.size() == 2 * n_chunks && (int)copy_ev.size() == n_chunks) {
    scene->row_cost.assign(f.rows_local, 0.f);
    for (int i = 0; i < n_chunks; i++) {
      float ms = 0;
      cudaEventElapsedTime(&ms, chunk_ev[2 * i], chunk_ev[2 * i + 1]);
      const int ck = plan.order[i];
      for (int r = plan.first_row[ck]; r < plan.first_row[ck] + plan.rows[ck]; r++) scene->row_cost[r] = ms / (float)std::max(1, plan.rows[ck]);
    }
    // Did the last chunk's kernels have to wait for its upload, or the other way round?  Once the compute-bound plan is
    // in use it stays until BOTH lanes were waiting for data at the end of a frame.
    float lag = 0, lag2 = 0;
    cudaEventElapsedTime(&lag, copy_ev[n_chunks - 1], chunk_ev[2 * (n_chunks - 1)]);
    if (n_chunks >= 2) cudaEventElapsedTime(&lag2, copy_ev[n_chunks - 2], chunk_ev[2 * (n_chunks - 2)]);
    scene->stream_compute_bound = plan.ramped ? !(lag < 0.05f && lag2 < 0.05f) : lag > 0.5f;
    scene->cost_key = {o.width, o.height, o.spp, o.shard_count, o.shard_index, o.band_height};
  }
  if (sh.tuning) {
    // only frames with enough walks to time say anything (256 Ki pairs ~ 0.2 ms)
    const FrameCounters* fc = counters();
    double ms = 0;
    for (const Span& sp : spans) {
      float m = 0;
      cudaEventElapsedTime(&m, sp.a, sp.b);
      if (sp.kind == 1) ms += m;
    }
    if (fc->shadow_walk_pairs >= (1u << 18)) {
      if (scene->tune_frames >= 1) scene->tune_ns_per_pair[scene->tune_frames - 1] = ms * 1e6 / (double)fc->shadow_walk_pairs;
      if (++scene->tune_frames == 3) scene->shadow_mode = scene->tune_ns_per_pair[1] < scene->tune_ns_per_pair[0] ? 2 : 1;
    } else if (++scene->tune_small_frames >= kTuneGiveUp) {
      scene->shadow_mode = 1;
    }
  } else if (sh.untuned) {
    if (++scene->tune_small_frames >= kTuneGiveUp) scene->shadow_mode = 1;
  }
}

// Sets *d to where the kernels write an output: nowhere when the caller asked for none (user null), the caller's buffer
// when it is device memory, else `scratch`, which the caller copies back to `user` after the kernels.
template <class T>
int stage_output(DevBuf& scratch, T* user, size_t bytes, bool dev_out, T** d) {
  *d = user;
  if (!user || dev_out) return RH_OK;
  const int rc = scratch.reserve(bytes);
  if (rc) return rc;
  *d = (T*)scratch.p;
  return RH_OK;
}

// Runs a validated frame: chunk plan, scratch, the chunks' launches, and — when a chunk's queues overflowed — the whole
// frame again with twice the queue capacity.
int run_frame(Device* D, const rh_scene* scene, const Frame& f, rh_stats* stats) {
  const rh_render_opts& o = f.o;
  const int mode = o.offset_mode;
  const bool dev_out = (o.flags & RH_FLAG_DEVICE_OUT) != 0, dev_off = (o.flags & RH_FLAG_DEVICE_OFFSETS) != 0;
  const bool peer_frames = (o.flags & RH_FLAG_PEER_FRAMES) != 0, want_ids = (o.flags & RH_FLAG_HIT_IDS) != 0;
  RH_CUDA(cudaSetDevice(D->dev));
  FrameRun R{D, scene, f};
  R.sh = choose_shadow(scene, f);
  R.counting = (o.flags & RH_FLAG_COUNT) != 0;
  R.row_samples = (size_t)o.width * o.spp;
  // A Transparent hit inserts a probe pass per level (RayHs.hs:136-143): up to 2D + 1 passes.  Without a Transparent
  // material the rays of pass k all have depth k, and pass D emits nothing: D + 1 passes, no empty launches after them.
  R.n_passes = scene->has_transparent ? 2 * o.max_depth + 1 : o.max_depth + 1;
  R.host_offsets = (mode == RH_OFFSETS_F64 || mode == RH_OFFSETS_F32 || mode == kOffsetsRays) && !dev_off;
  // what the last streamed frame of this shape measured: kernel time per row, and whether the kernels or the upload
  // finished last
  const bool know_cost = f.learns() && (int)scene->row_cost.size() == f.rows_local &&
                         scene->cost_key == std::vector<int>{o.width, o.height, o.spp, o.shard_count, o.shard_index, o.band_height};
  // a light-group frame's chunks also hold 3 doubles per group and sample, and (host output) per group and pixel
  const size_t group_bytes = f.n_groups ? 3 * sizeof(double) * (f.n_groups + 1) : 0;
  R.group_out_dev = dev_out;
  R.plan = rh::plan_chunks(f.rows_local, R.row_samples, o.chunk_samples, D->total_mem, R.host_offsets,
                           know_cost ? scene->row_cost.data() : nullptr, scene->stream_compute_bound,
                           rh::kBytesPerSample + group_bytes * (dev_out ? 1 : 2));
  R.n_chunks = (int)R.plan.rows.size();
  R.chunk_samples = (size_t)*std::max_element(R.plan.rows.begin(), R.plan.rows.end()) * R.row_samples;
  const std::string w(f.who);
  if (R.chunk_samples > 0x7fffffffu) return rh::set_error(RH_ERR_ARG, w + ": chunk too large");

  int rc;
  if ((rc = stage_output(D->rgb, peer_frames ? nullptr : f.out, f.out_bytes, dev_out, &R.d_rgb)) ||
      (rc = stage_output(D->ids, want_ids ? (int2*)f.ids_out : nullptr, f.ids_bytes, dev_out, &R.d_ids)) ||
      (rc = stage_output(D->linear, f.linear, f.linear_bytes, dev_out, &R.d_linear)))
    return rc;
  // Two chunks in flight (two streams, two sets of queues) when the frame has several: the kernels are persistent and
  // fill the GPU, so a chunk's next kernel starts on the SMs the other chunk's kernel frees as its warps run out of
  // work — the tail of every launch is filled instead of idle.  One lane when every launch is timed on its own.
  R.n_lanes = (R.n_chunks >= 2 && !R.sh.profile && !R.counting) ? rh::kLanes : 1;
  // Passes pipelined over two streams per lane: trace(k + 1) needs only trace(k)'s ray queue, the shadow kernels of pass k
  // only its hits, so trace(0) trace(1) ... run on one stream and classify(0) walk(0) classify(1) ... on the other.  Every
  // kernel is persistent and fills the GPU; what the second stream buys is that the SMs a kernel's last warps leave idle
  // (a lone warp walks a tree at ~1 us per node: the tail of a small launch is most of it) start the other stream's
  // next kernel.  All adds to the accumulators are made by the shadow stream in pass order: same bits as one stream.
  // Single-chunk frames only: a frame of several chunks has two of them in flight, which fills the same gaps, and a ring
  // that holds two passes' hits at a time needs the queue capacity a triangle soup does not leave.
  R.pipelined = !R.sh.profile && !R.counting && R.n_passes >= 2 && R.n_chunks == 1;
  for (int l = 0; l < R.n_lanes; l++)
    if ((rc = D->lane[l].accum.reserve(R.chunk_samples * 3 * sizeof(double)))) return rc;
  if (f.n_groups) {
    const size_t chunk_px = R.chunk_samples / o.spp;
    R.group_out_stride = dev_out ? (size_t)f.rows_local * o.width * 3 : chunk_px * 3;
    for (int l = 0; l < R.n_lanes; l++) {
      if ((rc = D->lane[l].groups.reserve(R.chunk_samples * group_bytes))) return rc;
      if (!dev_out && (rc = D->lane[l].group_out.reserve(chunk_px * group_bytes))) return rc;
    }
  }
  const size_t ctl_bytes = (size_t)R.n_chunks * sizeof(ChunkCtl);
  if ((rc = D->ctl.reserve(ctl_bytes))) return rc;
  if ((rc = D->counters.reserve(sizeof(FrameCounters)))) return rc;
  if (D->pinned_bytes < ctl_bytes + sizeof(FrameCounters)) {
    if (D->pinned) cudaFreeHost(D->pinned);
    D->pinned = nullptr;
    D->pinned_bytes = 0;
    RH_CUDA(cudaMallocHost(&D->pinned, ctl_bytes + sizeof(FrameCounters)));
    D->pinned_bytes = ctl_bytes + sizeof(FrameCounters);
  }
  // sample offsets
  const size_t tile_bytes = (size_t)o.offset_tile * o.offset_tile * o.spp * f.off_elem;
  if (mode == RH_OFFSETS_TILED_F64) {
    if (dev_off) R.d_offsets = o.offsets;
    else {
      if ((rc = D->offsets.reserve(tile_bytes))) return rc;
      R.d_offsets = D->offsets.p;
    }
  } else if (mode != RH_OFFSETS_NONE && dev_off) {  // (RH_OFFSETS_SPLITMIX64 takes a host seed: frame_chunk_params's)
    R.d_offsets = o.offsets;
    R.off_index = (o.flags & RH_FLAG_SHARD_OFFSETS) ? kOffIndexLocal : kOffIndexGlobal;  // (compact: each chunk's slice is in work-item order)
  } else if (R.host_offsets) {
    // Upload ring: as many chunk-sized slots as 10 % of the device memory holds (all chunks, for the frames of
    // BASELINE.json), so that the copy stream can run ahead of the kernels instead of waiting for a slot.
    const size_t slot_bytes = R.chunk_samples * f.off_elem;
    R.ring = (int)std::max<size_t>(2, std::min<size_t>((size_t)R.n_chunks, (size_t)(0.1 * (double)D->total_mem) / slot_bytes));
    if ((rc = D->offsets.reserve((size_t)R.ring * slot_bytes))) return rc;
    while ((int)D->ev_up.size() < R.ring) {
      cudaEvent_t a, b;
      RH_CUDA(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
      RH_CUDA(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
      D->ev_up.push_back(a);
      D->ev_done.push_back(b);
    }
  }

  // queue capacity = factor * chunk samples; doubled when a chunk overflows (and remembered by the scene's renders; a
  // trace starts from 2, a list frame from the scene's factor).  A views frame starts from the larger of the scene's
  // factor and the one its own last views frame needed, halved while the lanes' queues would hold more entries than
  // factor 2 gives the largest chunk plan_chunks makes: a factor learned on small frames, whose per-warp slack is
  // large, must not size the queues of a batch many times their size (measured on dragon_full: 128² renders leave 32,
  // which asked a batch of 256 such views for 32 x 67 M queue entries and failed with RH_ERR_OOM).
  uint32_t factor = f.trace ? 2u : std::max(2u, scene->queue_factor);
  if (f.views) {
    factor = std::max(factor, scene->views_queue_factor);
    while (factor > 2 && (size_t)factor * R.chunk_samples * R.n_lanes > 2 * rh::max_chunk_samples(D->total_mem)) factor /= 2;
  }
  for (;;) {
    if ((rc = R.reserve_queues(factor))) return rc;
    R.launches = 0;
    R.upload_bytes = R.ev_used = 0;
    R.spans.clear();
    R.chunk_ev.clear();
    R.copy_ev.clear();
    RH_CUDA(cudaEventRecord(D->ev_begin, D->stream));
    RH_CUDA(cudaMemsetAsync(D->ctl.p, 0, ctl_bytes, D->stream));
    RH_CUDA(cudaMemsetAsync(D->counters.p, 0, sizeof(FrameCounters), D->stream));
    if (mode == RH_OFFSETS_TILED_F64 && !dev_off)
      RH_CUDA(cudaMemcpyAsync((void*)R.d_offsets, o.offsets, tile_bytes, cudaMemcpyHostToDevice, D->stream));
    for (const Frame::Upload& u : f.uploads) {
      RH_CUDA(cudaMemcpyAsync(u.dst, u.src, u.bytes, cudaMemcpyHostToDevice, D->stream));
      R.upload_bytes += u.bytes;
    }
    if (R.n_lanes > 1) {  // lane 1 starts after the control blocks are zeroed
      RH_CUDA(cudaEventRecord(D->ev_lane, D->stream));
      RH_CUDA(cudaStreamWaitEvent(D->stream2, D->ev_lane, 0));
    }
    for (int i = 0; i < R.n_chunks; i++)
      if ((rc = R.enqueue_chunk(i))) return rc;
    RH_CUDA(cudaGetLastError());
    if (R.n_lanes > 1) {  // join: everything below waits for lane 1 too
      RH_CUDA(cudaEventRecord(D->ev_lane, D->stream2));
      RH_CUDA(cudaStreamWaitEvent(D->stream, D->ev_lane, 0));
    }
    RH_CUDA(cudaMemcpyAsync(D->pinned, D->ctl.p, ctl_bytes, cudaMemcpyDeviceToHost, D->stream));
    RH_CUDA(cudaMemcpyAsync((char*)D->pinned + ctl_bytes, D->counters.p, sizeof(FrameCounters), cudaMemcpyDeviceToHost, D->stream));
    if (!dev_out && !peer_frames) {
      if (f.out) RH_CUDA(cudaMemcpyAsync(f.out, R.d_rgb, f.out_bytes, cudaMemcpyDeviceToHost, D->stream));
      if (want_ids) RH_CUDA(cudaMemcpyAsync(f.ids_out, R.d_ids, f.ids_bytes, cudaMemcpyDeviceToHost, D->stream));
      if (f.linear) RH_CUDA(cudaMemcpyAsync(f.linear, R.d_linear, f.linear_bytes, cudaMemcpyDeviceToHost, D->stream));
    }
    RH_CUDA(cudaEventRecord(D->ev_end, D->stream));
    RH_CUDA(cudaStreamSynchronize(D->stream));
    g_launches.fetch_add(R.launches, std::memory_order_relaxed);

    bool overflow = false;
    for (int ck = 0; ck < R.n_chunks; ck++) overflow |= R.ctl()[ck].overflow != 0;
    if (overflow) {
      if (R.cap >= 0x7fffff00u || factor >= (1u << 16))
        return rh::set_error(RH_ERR_OVERFLOW, w + ": ray queue overflow; lower " + (f.trace ? "chunk_rays" : "chunk_samples"));
      factor *= 2;
      if (f.learns()) scene->queue_factor = factor;
      if (f.views) scene->views_queue_factor = factor;
      continue;
    }
    if (stats) R.read_stats(stats, factor);
    R.print_timeline();
    if (f.learns()) R.learn();
    return RH_OK;
  }
}

int render_on(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, uint8_t* rgb_out,
              int32_t* hit_ids_out, rh_stats* stats) {
  // (rh_multi_render's shards store into the peer frames instead)
  if (!rgb_out && !(o && (o->flags & RH_FLAG_PEER_FRAMES))) return rh::set_error(RH_ERR_ARG, "rh_render: null argument");
  Frame f;
  const int rc = render_frame(D, scene, camera, o, rgb_out, hit_ids_out, &f);
  return rc ? rc : run_frame(D, scene, f, stats);
}

// A buffer an entry point takes with RH_FLAG_DEVICE_OUT: null when the call does not use it, and the alignment of the
// words its kernels move (1: none).
struct DeviceArg {
  const void* p;
  size_t align;
  const char* name;
};

// RH_FLAG_DEVICE_OUT's checks: every listed buffer aligned, then device (or managed) memory of D's GPU, which this
// makes the current one.
int check_device_outputs(Device* D, const std::string& who, std::initializer_list<DeviceArg> args) {
  for (const DeviceArg& a : args)
    if ((uintptr_t)a.p % a.align)
      return rh::set_error(RH_ERR_ARG, who + ": device " + a.name + " must be " + std::to_string(a.align) + "-byte aligned");
  RH_CUDA(cudaSetDevice(D->dev));
  for (const DeviceArg& a : args) {
    if (!a.p) continue;
    cudaPointerAttributes attr{};
    RH_CUDA(cudaPointerGetAttributes(&attr, a.p));
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
      return rh::set_error(RH_ERR_ARG, who + ": RH_FLAG_DEVICE_OUT with a pointer that is not device memory");
  }
  return RH_OK;
}

// ------------------------------------------------------------------ per-pixel state across calls (rh_accum, rh_adaptive)
// The checks the two kinds of state share; `noun` names the state in the messages, `reset` its reset entry point.
int shard_state_init(ShardState* S, Device* D, int width, int height, int shard_index, int shard_count, int band_height,
                     uint32_t stream_spp, const std::string& who) {
  const int G = shard_count <= 0 ? 1 : shard_count;
  if (width <= 0 || height <= 0) return rh::set_error(RH_ERR_ARG, who + ": bad width/height");
  if (shard_index < 0 || shard_index >= G) return rh::set_error(RH_ERR_ARG, who + ": shard_index out of range");
  S->device = D;
  S->context = D->context;
  S->dev = D->dev;
  S->width = width;
  S->height = height;
  S->shard_index = shard_index;
  S->shard_count = G;
  S->band_height = band_height > 0 ? band_height : rh_default_band_height(height, G);
  S->rows_local = rh_shard_rows(height, G, S->band_height);
  S->stream_spp = stream_spp;
  S->plane = (size_t)S->rows_local * width;
  return RH_OK;
}
int shard_state_context(const ShardState* S, Device* D, const std::string& w, const char* noun) {
  if (S->device != D || S->context != D->context) return rh::set_error(RH_ERR_ARG, w + ": " + noun + " lives on another device context");
  return RH_OK;
}
// The frame's size and shard are the state's; once the view is fixed, so are the scene, the camera bytes and max_depth.
int shard_state_matches(const ShardState* S, const Frame& f, bool fixed, const rh_scene* scene, const rh_camera* camera,
                        const std::string& w, const char* noun, const char* reset) {
  if (f.o.width != S->width || f.o.height != S->height || f.o.shard_index != S->shard_index ||
      f.o.shard_count != S->shard_count || f.o.band_height != S->band_height)
    return rh::set_error(RH_ERR_ARG, w + ": width, height, shard_index, shard_count or band_height differ from the " + noun + "'s");
  if (fixed && (scene != S->scene || memcmp(camera, &S->camera, sizeof S->camera) != 0 || f.o.max_depth != S->max_depth))
    return rh::set_error(RH_ERR_ARG, w + ": scene, camera or max_depth differ from the " + noun + "'s first call; " + reset + " it first");
  if (fixed && scene->generation != S->scene_generation)
    return rh::set_error(RH_ERR_ARG, w + ": the scene was updated since the " + noun + "'s first call; " + reset + " it first");
  return RH_OK;
}
void shard_state_fix_view(ShardState* S, const rh_scene* scene, const rh_camera* camera, int32_t max_depth) {
  S->scene = scene;
  S->scene_generation = scene->generation;
  S->camera = *camera;
  S->max_depth = max_depth;
}

// RH_OFFSETS_SPLITMIX64's window check: "" when samples [base, base + spp) lie inside a stream of stream_spp samples per
// pixel, else what is wrong
std::string stream_window_error(uint32_t base, uint32_t spp, uint32_t stream_spp) {
  if ((uint64_t)base + spp <= stream_spp) return "";
  return "RH_OFFSETS_SPLITMIX64 past the end of the stream (" + std::to_string(base) + " + spp " + std::to_string(spp) +
         " > stream_spp " + std::to_string(stream_spp) + ")";
}

// ------------------------------------------------------------------ progressive accumulation
// rh_render_accumulate's argument checks: rh_render's (render_frame), then those of the accumulator.
int accumulate_frame(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, rh_accum* acc,
                     uint8_t* rgb_out, double* linear_out, int32_t* hit_ids_out, Frame* f) {
  const std::string w = "rh_render_accumulate";
  if (!scene || !camera || !o || !acc) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  int rc = shard_state_context(acc, D, w, "accumulator");
  if (rc) return rc;
  if (o->flags & RH_FLAG_PEER_FRAMES) return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_PEER_FRAMES is not supported");
  f->accumulate = true;
  rc = render_frame(D, scene, camera, o, rgb_out, hit_ids_out, f, "rh_render_accumulate");
  if (rc) return rc;
  if ((rc = shard_state_matches(acc, *f, false, scene, camera, w, "accumulator", "rh_accum_reset"))) return rc;
  const uint32_t spp = (uint32_t)o->spp;
  if ((uint64_t)acc->n + spp > 0xffffffffu) return rh::set_error(RH_ERR_ARG, w + ": more than 2^32 - 1 samples per pixel");
  if (o->offset_mode == RH_OFFSETS_SPLITMIX64) {
    if (acc->stream_spp == 0)
      return rh::set_error(RH_ERR_ARG, w + ": RH_OFFSETS_SPLITMIX64 needs an accumulator created with stream_spp > 0");
    const std::string window = stream_window_error(acc->n, spp, acc->stream_spp);
    if (!window.empty()) return rh::set_error(RH_ERR_ARG, w + ": " + window);
  }
  if ((rc = shard_state_matches(acc, *f, acc->n > 0, scene, camera, w, "accumulator", "rh_accum_reset"))) return rc;
  const bool want_ids = (o->flags & RH_FLAG_HIT_IDS) != 0;
  if ((o->flags & RH_FLAG_DEVICE_OUT) &&
      (rc = check_device_outputs(D, w, {{rgb_out, 1, "rgb_out"}, {linear_out, 8, "linear_out"}, {want_ids ? hit_ids_out : nullptr, 1, "hit_ids_out"}})))
    return rc;
  const size_t half = 3 * acc->plane;
  f->stream_spp = acc->stream_spp;
  f->stream_base = acc->n;
  f->acc.sum_in = (const double*)acc->sums.p + (size_t)acc->cur * half;
  f->acc.sum_out = (double*)acc->sums.p + (size_t)(acc->cur ^ 1) * half;
  f->acc.plane = acc->plane;
  f->acc.n_before = acc->n;
  f->acc.n_total = acc->n + spp;
  f->linear = linear_out;
  f->linear_bytes = (size_t)f->rows_local * f->o.width * 3 * sizeof(double);
  return RH_OK;
}

int accumulate_on(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, rh_accum* acc,
                  uint8_t* rgb_out, double* linear_out, int32_t* hit_ids_out, rh_stats* stats) {
  Frame f;
  int rc = accumulate_frame(D, scene, camera, o, acc, rgb_out, linear_out, hit_ids_out, &f);
  if (rc || (rc = run_frame(D, scene, f, stats))) return rc;
  // the frame completed: its sums are the current ones
  if (acc->n == 0) shard_state_fix_view(acc, scene, camera, o->max_depth);
  acc->cur ^= 1;
  acc->n += (uint32_t)o->spp;
  return RH_OK;
}

int accum_create_on(Device* D, int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                    rh_accum** out) {
  if (!out) return rh::set_error(RH_ERR_ARG, "rh_accum_create: null out");
  *out = nullptr;
  auto A = std::make_unique<rh_accum>();
  int rc = shard_state_init(A.get(), D, width, height, shard_index, shard_count, band_height, stream_spp, "rh_accum_create");
  if (rc) return rc;
  RH_CUDA(cudaSetDevice(D->dev));
  rc = A->sums.reserve(2 * 3 * A->plane * sizeof(double));
  if (rc) return rc;
  *out = A.release();
  return RH_OK;
}

// ------------------------------------------------------------------ adaptive sampling
// rh_render_adaptive's list frames: a fixed number of list entries per frame row.  Small enough that chunk_samples can
// split a small image's list into several chunks, large enough that a 4K list has a few thousand rows.
constexpr int kListRowEntries = 1024;

// rh_render_adaptive's argument checks: rh_render's (render_frame), then those of the adaptive state.
int adaptive_frame(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o,
                   const rh_adaptive_opts* ao, rh_adaptive* ad, uint8_t* rgb_out, double* linear_out, Frame* f) {
  const std::string w = "rh_render_adaptive";
  if (!scene || !camera || !o || !ao || !ad) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  int rc = shard_state_context(ad, D, w, "adaptive state");
  if (rc) return rc;
  if (o->flags & (RH_FLAG_HIT_IDS | RH_FLAG_PEER_FRAMES | RH_FLAG_SHARD_OFFSETS | RH_FLAG_DEVICE_OFFSETS))
    return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_HIT_IDS, RH_FLAG_PEER_FRAMES, RH_FLAG_SHARD_OFFSETS and RH_FLAG_DEVICE_OFFSETS are not supported");
  if (o->offset_mode != RH_OFFSETS_SPLITMIX64) return rh::set_error(RH_ERR_ARG, w + ": offset_mode must be RH_OFFSETS_SPLITMIX64");
  if (!(ao->threshold >= 0)) return rh::set_error(RH_ERR_ARG, w + ": threshold must be >= 0");
  if (ao->min_spp < 2) return rh::set_error(RH_ERR_ARG, w + ": min_spp must be >= 2");
  if (ao->reserved_ != 0) return rh::set_error(RH_ERR_ARG, w + ": rh_adaptive_opts.reserved_ must be 0");
  f->pixel_list = true;
  if ((rc = render_frame(D, scene, camera, o, rgb_out, nullptr, f, "rh_render_adaptive"))) return rc;
  if ((rc = shard_state_matches(ad, *f, ad->fixed, scene, camera, w, "adaptive state", "rh_adaptive_reset"))) return rc;
  if ((o->flags & RH_FLAG_DEVICE_OUT) && (rc = check_device_outputs(D, w, {{rgb_out, 1, "rgb_out"}, {linear_out, 8, "linear_out"}})))
    return rc;
  f->ad = ad->A;
  f->ad.spp = (uint32_t)o->spp;
  f->ad.min_spp = ao->min_spp;
  f->ad.tt = ao->threshold * ao->threshold;
  f->stream_spp = ad->stream_spp;
  f->list = {f->ad.list, f->ad.counts, (uint32_t)ad->width, (uint32_t)ad->height, (uint32_t)ad->shard_index,
             (uint32_t)ad->shard_count, (uint32_t)ad->band_height};
  return RH_OK;
}

// Select (library stream), read n_active back, the list frame (run_frame), commit, output.  Until the commit the state
// is only read, so every failure before it leaves the state as it was.
int adaptive_on(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, const rh_adaptive_opts* ao,
                rh_adaptive* ad, uint8_t* rgb_out, double* linear_out, uint64_t* n_active_out, rh_stats* stats) {
  Frame f;
  int rc = adaptive_frame(D, scene, camera, o, ao, ad, rgb_out, linear_out, &f);
  if (rc) return rc;
  const bool dev_out = (o->flags & RH_FLAG_DEVICE_OUT) != 0, profile = (o->flags & RH_FLAG_PROFILE) != 0;
  AdaptiveParams A = f.ad;
  RH_CUDA(cudaSetDevice(D->dev));
  RH_CUDA(cudaEventRecord(ad->ev[0], D->stream));
  launch_adaptive_select(A, D->stream);
  RH_CUDA(cudaEventRecord(ad->ev[1], D->stream));
  uint32_t n_active = 0;
  RH_CUDA(cudaMemcpyAsync(&n_active, A.n_active, sizeof n_active, cudaMemcpyDeviceToHost, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  uint32_t launches = 3;

  // the list frame: its rows are rows of the list, unsharded; pass 0 reads the pixels through f.list
  rh_stats fs{};
  if (n_active) {
    const uint64_t rows = ((uint64_t)n_active + kListRowEntries - 1) / kListRowEntries;
    f.o.width = kListRowEntries;
    f.o.height = f.o.band_height = f.rows_local = (int)rows;
    f.o.shard_index = 0;
    f.o.shard_count = 1;
    f.out = nullptr;
    f.out_bytes = 0;
    f.n_rays = f.rays_primary = (uint64_t)n_active * A.spp;
    if ((rc = run_frame(D, scene, f, &fs))) return rc;
    RH_CUDA(cudaSetDevice(D->dev));
  }

  RH_CUDA(cudaEventRecord(ad->ev[2], D->stream));
  launch_adaptive_commit(A, n_active, D->stream);
  launches += n_active ? 1 : 0;
  const size_t px = ad->plane;
  unsigned long long negative = 0;
  if (rgb_out || linear_out) {
    if ((rc = stage_output(D->rgb, rgb_out, px * 3, dev_out, &A.rgb)) ||
        (rc = stage_output(D->linear, linear_out, px * 3 * sizeof(double), dev_out, &A.linear)))
      return rc;
    RH_CUDA(cudaMemsetAsync(A.negative, 0, sizeof(unsigned long long), D->stream));
    launch_adaptive_output(A, D->stream);
    launches += 1;
    if (!dev_out) {
      if (rgb_out) RH_CUDA(cudaMemcpyAsync(rgb_out, A.rgb, px * 3, cudaMemcpyDeviceToHost, D->stream));
      if (linear_out) RH_CUDA(cudaMemcpyAsync(linear_out, A.linear, px * 3 * sizeof(double), cudaMemcpyDeviceToHost, D->stream));
    }
    if (rgb_out) RH_CUDA(cudaMemcpyAsync(&negative, A.negative, sizeof negative, cudaMemcpyDeviceToHost, D->stream));
  }
  RH_CUDA(cudaEventRecord(ad->ev[3], D->stream));
  RH_CUDA(cudaGetLastError());
  RH_CUDA(cudaStreamSynchronize(D->stream));
  g_launches.fetch_add(launches, std::memory_order_relaxed);
  if (!ad->fixed) {
    shard_state_fix_view(ad, scene, camera, o->max_depth);
    ad->fixed = true;
  }
  if (n_active_out) *n_active_out = n_active;
  if (stats) {
    *stats = fs;  // (zero when nothing was traced)
    float ms = 0;
    cudaEventElapsedTime(&ms, ad->ev[0], ad->ev[3]);
    stats->ms_total = ms;
    if (profile) {
      float sel = 0, post = 0;
      cudaEventElapsedTime(&sel, ad->ev[0], ad->ev[1]);
      cudaEventElapsedTime(&post, ad->ev[2], ad->ev[3]);
      stats->ms_resolve += sel + post;
    }
    stats->kernel_launches += launches;
    stats->negative_channels = (uint32_t)std::min<unsigned long long>(negative, 0xffffffffu);
  }
  return RH_OK;
}

void adaptive_release(rh_adaptive* ad) {
  for (cudaEvent_t& e : ad->ev)
    if (e) cudaEventDestroy(e), e = nullptr;
  ad->state.release();
  ad->work.release();
  ad->scratch.release();
}

// State 52 bytes per pixel, list and staging 52, scratch one bit per pixel and a word per kSelectBlock pixels.
int adaptive_create_on(Device* D, int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                       rh_adaptive** out) {
  if (!out) return rh::set_error(RH_ERR_ARG, "rh_adaptive_create: null out");
  *out = nullptr;
  if (stream_spp < 1) return rh::set_error(RH_ERR_ARG, "rh_adaptive_create: stream_spp must be >= 1");
  std::unique_ptr<rh_adaptive, void (*)(rh_adaptive*)> ad(new rh_adaptive(), [](rh_adaptive* a) { adaptive_release(a); delete a; });
  int rc = shard_state_init(ad.get(), D, width, height, shard_index, shard_count, band_height, stream_spp, "rh_adaptive_create");
  if (rc) return rc;
  const size_t px = ad->plane;
  if (px >= 0xffffffffu) return rh::set_error(RH_ERR_ARG, "rh_adaptive_create: more than 2^32 - 2 pixels per shard");
  RH_CUDA(cudaSetDevice(D->dev));
  const size_t words = (px + 1) / 2 * 2;  // uint32 planes padded to 8 bytes
  const size_t n_blocks = (px + kSelectBlock - 1) / kSelectBlock;
  const size_t state_bytes = words * 4 + 6 * px * sizeof(double);
  if ((rc = ad->state.reserve(state_bytes))) return rc;
  if ((rc = ad->work.reserve(words * 4 + 6 * px * sizeof(double)))) return rc;
  if ((rc = ad->scratch.reserve(16 + (n_blocks + n_blocks * (kSelectBlock / 32)) * sizeof(uint32_t)))) return rc;
  for (cudaEvent_t& e : ad->ev) RH_CUDA(cudaEventCreate(&e));
  RH_CUDA(cudaMemsetAsync(ad->state.p, 0, state_bytes, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  AdaptiveParams& A = ad->A;
  A.counts = (uint32_t*)ad->state.p;
  A.sum = (double*)((char*)ad->state.p + words * 4);
  A.sumsq = A.sum + 3 * px;
  A.list = (uint32_t*)ad->work.p;
  A.stage = (double*)((char*)ad->work.p + words * 4);
  A.negative = (unsigned long long*)ad->scratch.p;
  A.n_active = (uint32_t*)((char*)ad->scratch.p + 8);
  A.block_counts = (uint32_t*)((char*)ad->scratch.p + 16);
  A.warp_masks = A.block_counts + n_blocks;
  A.plane = px;
  A.width = (uint32_t)width;
  A.height = (uint32_t)height;
  A.shard_index = (uint32_t)ad->shard_index;
  A.shard_count = (uint32_t)ad->shard_count;
  A.band_height = (uint32_t)ad->band_height;
  A.stream_spp = stream_spp;
  *out = ad.release();
  return RH_OK;
}

int adaptive_reset_on(rh_adaptive* ad) {
  RH_CUDA(cudaSetDevice(ad->dev));
  RH_CUDA(cudaMemset(ad->state.p, 0, (ad->plane + 1) / 2 * 2 * 4 + 6 * ad->plane * sizeof(double)));
  RH_CUDA(cudaDeviceSynchronize());  // (the library's streams do not wait for the legacy stream)
  ad->fixed = false;
  ad->scene = nullptr;
  return RH_OK;
}

// The state out: the counts as they are, S and Q from three planes to double[pixel][3] (host buffers through the
// device scratch of the linear colours).
int adaptive_state_on(Device* D, const rh_adaptive* ad, uint32_t* counts_out, double* sums_out, double* sumsq_out, int32_t flags) {
  const std::string w = "rh_adaptive_state";
  if (!ad) return rh::set_error(RH_ERR_ARG, w + ": null state");
  int rc = shard_state_context(ad, D, w, "adaptive state");
  if (rc) return rc;
  if (flags & ~RH_FLAG_DEVICE_OUT) return rh::set_error(RH_ERR_ARG, w + ": flags must be 0 or RH_FLAG_DEVICE_OUT");
  const bool dev = (flags & RH_FLAG_DEVICE_OUT) != 0;
  RH_CUDA(cudaSetDevice(D->dev));
  if (dev && (rc = check_device_outputs(D, w, {{counts_out, 1, "counts_out"}, {sums_out, 8, "sums_out"}, {sumsq_out, 8, "sumsq_out"}})))
    return rc;
  const size_t px = ad->plane, bytes = px * 3 * sizeof(double);
  if (counts_out)
    RH_CUDA(cudaMemcpyAsync(counts_out, ad->A.counts, px * sizeof(uint32_t), dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, D->stream));
  const double* planes[2] = {ad->A.sum, ad->A.sumsq};
  double* outs[2] = {sums_out, sumsq_out};
  for (int k = 0; k < 2; k++) {
    double* d;
    if ((rc = stage_output(D->linear, outs[k], bytes, dev, &d))) return rc;
    if (!d) continue;
    launch_adaptive_interleave(planes[k], px, d, D->stream);
    if (!dev) RH_CUDA(cudaMemcpyAsync(outs[k], d, bytes, cudaMemcpyDeviceToHost, D->stream));
  }
  RH_CUDA(cudaGetLastError());
  RH_CUDA(cudaStreamSynchronize(D->stream));
  return RH_OK;
}

// ------------------------------------------------------------------ batched ray queries
// Rays per launch: the kernels' claim units and ray indices stay far inside 32 bits.
constexpr uint64_t kQueryLaunch = 1ull << 24;
// Rays per chunk of host buffers: 2 Mi x (48 + 80) bytes = 256 MB of device scratch, whatever n is.
constexpr uint64_t kQueryChunk = 1ull << 21;
constexpr size_t kQueryCursorBytes = 256;  // (keeps the chunk buffers 256-byte aligned)

// rh_closest_intersection (light < 0) / rh_shadow_intersection (light >= 0).
int query_on(Device* D, const rh_scene* scene, int64_t light, const double* rays, uint64_t n, void* out, int32_t flags,
             const char* who) {
  const std::string w(who);
  if (!scene) return rh::set_error(RH_ERR_ARG, w + ": null scene");
  if (scene->device != D) return rh::set_error(RH_ERR_ARG, w + ": scene lives on another device context");
  if (flags & ~(RH_FLAG_DEVICE_OUT | RH_FLAG_EXACT_BOXES))
    return rh::set_error(RH_ERR_ARG, w + ": flags other than RH_FLAG_DEVICE_OUT and RH_FLAG_EXACT_BOXES");
  if (light >= 0 && (uint64_t)light >= scene->view.n_lights) return rh::set_error(RH_ERR_ARG, w + ": light index out of range");
  if (n == 0) return RH_OK;
  if (!rays || !out) return rh::set_error(RH_ERR_ARG, w + ": null buffer");
  const bool shadow = light >= 0, dev = (flags & RH_FLAG_DEVICE_OUT) != 0;
  const size_t out_bytes = shadow ? sizeof(uint8_t) : sizeof(rh_hit);
  int rc;
  // the kernels move rays and records in 16-byte words
  if (dev && (rc = check_device_outputs(D, w, {{rays, 16, "rays"}, {out, shadow ? 1u : 16u, shadow ? "occluded_out" : "hits_out"}})))
    return rc;
  RH_CUDA(cudaSetDevice(D->dev));
  Device::Scratch& sc = D->lane[0];  // the render's deep-stack scratch covers grid x block of the query kernels
  if ((rc = sc.deep.reserve((size_t)scene->deep_entries * D->max_threads * sizeof(uint2)))) return rc;
  const uint64_t chunk = dev ? kQueryLaunch : kQueryChunk;
  if ((rc = D->query.reserve(kQueryCursorBytes + (dev ? 0 : (size_t)chunk * (6 * sizeof(double) + out_bytes))))) return rc;
  char* d_rays = (char*)D->query.p + kQueryCursorBytes;
  char* d_out = d_rays + (size_t)chunk * 6 * sizeof(double);
  QueryParams Q{};
  Q.light = shadow ? (uint32_t)light : 0u;
  Q.exact_boxes = (flags & RH_FLAG_EXACT_BOXES) ? 1 : 0;
  Q.deep_stack = (uint2*)sc.deep.p;
  Q.deep_stride = (uint32_t)D->max_threads;
  Q.cursor = (uint32_t*)D->query.p;
  for (uint64_t first = 0; first < n; first += chunk) {
    const uint64_t m = std::min<uint64_t>(chunk, n - first);
    const double* src = rays + first * 6;
    char* dst = (char*)out + first * out_bytes;
    if (!dev) RH_CUDA(cudaMemcpyAsync(d_rays, src, (size_t)m * 6 * sizeof(double), cudaMemcpyHostToDevice, D->stream));
    Q.rays = dev ? src : (const double*)d_rays;
    Q.n = (uint32_t)m;
    if (shadow) Q.occluded = (uint8_t*)(dev ? dst : d_out);
    else Q.hits = (rh_hit*)(dev ? dst : d_out);
    RH_CUDA(cudaMemsetAsync(Q.cursor, 0, sizeof(uint32_t), D->stream));
    if (shadow) launch_query_shadow(scene->view, Q, D->n_sms, D->stream);
    else launch_query_closest(scene->view, Q, D->n_sms, D->stream);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    RH_CUDA(cudaGetLastError());
    if (!dev) RH_CUDA(cudaMemcpyAsync(dst, d_out, (size_t)m * out_bytes, cudaMemcpyDeviceToHost, D->stream));
  }
  RH_CUDA(cudaStreamSynchronize(D->stream));
  return RH_OK;
}

// ------------------------------------------------------------------ radiance queries
// rh_trace_rays runs the render's wavefront on a frame of one sample per ray: kTraceRowRays rays per row, as many rows
// as the rays need, unsharded.  Pass 0 reads the rays (kOffsetsRays) and the colours leave unquantised; everything in
// between — chunk plan, queues, overflow retry, pipelined passes, counts — is run_frame's.
constexpr int kTraceRowRays = 4096;

int trace_on(Device* D, const rh_scene* scene, const double* rays, uint64_t n, const rh_trace_opts* o, double* colors_out,
             int32_t* hit_ids_out, rh_stats* stats) {
  if (!scene || !o) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: null scene or opts");
  if (scene->device != D) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: scene lives on another device context");
  constexpr int32_t kFlags = RH_FLAG_DEVICE_OUT | RH_FLAG_HIT_IDS | RH_FLAG_EXACT_BOXES | RH_FLAG_SHADOW_POOLED |
                             RH_FLAG_SHADOW_SPLIT | RH_FLAG_NO_LIGHT_MAPS;
  if (o->flags & ~kFlags) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: unknown flag bits");
  if (o->max_depth < 0 || o->max_depth > kMaxDepth) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: max_depth outside 0..30");
  if (n == 0) {
    if (stats) memset(stats, 0, sizeof *stats);
    return RH_OK;
  }
  const bool want_ids = (o->flags & RH_FLAG_HIT_IDS) != 0, dev = (o->flags & RH_FLAG_DEVICE_OUT) != 0;
  if (!rays || !colors_out) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: null buffer");
  if (want_ids && !hit_ids_out) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: RH_FLAG_HIT_IDS without hit_ids_out");
  const uint64_t rows = (n + kTraceRowRays - 1) / kTraceRowRays;
  if (rows > 0x7fffffffu) return rh::set_error(RH_ERR_ARG, "rh_trace_rays: too many rays");
  // rays are read as 16-byte words; colours and ids are written as 8-byte words
  if (dev) {
    const int rc = check_device_outputs(D, "rh_trace_rays", {{rays, 16, "rays"}, {colors_out, 8, "colors_out"},
                                                             {want_ids ? hit_ids_out : nullptr, 8, "hit_ids_out"}});
    if (rc) return rc;
  }
  Frame f;
  f.who = "rh_trace_rays";
  f.o.width = kTraceRowRays;
  f.o.height = f.o.band_height = f.rows_local = (int)rows;
  f.o.max_depth = o->max_depth;
  f.o.spp = 1;
  f.o.offset_mode = kOffsetsRays;
  f.o.offsets = rays;
  f.o.shard_count = 1;
  f.o.chunk_samples = (int)std::min<uint64_t>(o->chunk_rays, 0x7fffffffu);
  f.o.flags = o->flags | (dev ? RH_FLAG_DEVICE_OFFSETS : 0);
  f.out = (uint8_t*)colors_out;
  f.ids_out = hit_ids_out;
  f.out_bytes = (size_t)n * 3 * sizeof(double);
  f.ids_bytes = (size_t)n * sizeof(int2);
  f.off_elem = sizeof(double) * 6;
  f.rays_primary = n;
  f.trace = true;
  f.n_rays = n;
  return run_frame(D, scene, f, stats);
}

// ------------------------------------------------------------------ feature buffers
// rh_render_features casts the render's camera rays (render_frame's checks and geometry, load_item's offsets) through
// feature_kernel, chunk after chunk of rows on the library stream.  Device outputs with device (or no) offsets are used
// in place, in chunks as large as one launch takes; host offsets and host outputs go through device scratch in smaller
// chunks, so that a 4K x 16-spp offset array (2.1 GB) is never staged at once.
constexpr uint64_t kFeatureLaunchSamples = 1ull << 30;  // camera samples per launch: item indices stay far inside 32 bits
constexpr uint64_t kFeatureChunkSamples = 1ull << 21;   // ... per chunk through scratch: 32 MB of F64 offsets, 16 MB of ids

int features_on(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, const rh_features* ft,
                int32_t* hit_ids_out, rh_stats* stats) {
  const std::string w = "rh_render_features";
  if (!scene || !camera || !o || !ft) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  if (o->flags & (RH_FLAG_PEER_FRAMES | RH_FLAG_COUNT | RH_FLAG_PROFILE))
    return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_PEER_FRAMES, RH_FLAG_COUNT and RH_FLAG_PROFILE are not supported");
  const bool want_ids = (o->flags & RH_FLAG_HIT_IDS) != 0;
  if (!ft->albedo && !ft->normal && !ft->depth && !ft->hits && !want_ids) return rh::set_error(RH_ERR_ARG, w + ": no output requested");
  if (o->offset_mode != RH_OFFSETS_SPLITMIX64 && (ft->stream_spp || ft->stream_base))
    return rh::set_error(RH_ERR_ARG, w + ": stream_spp and stream_base are for RH_OFFSETS_SPLITMIX64 only");
  Frame f;
  int rc = render_frame(D, scene, camera, o, nullptr, hit_ids_out, &f, "rh_render_features");
  if (rc) return rc;
  const uint32_t spp = (uint32_t)o->spp;
  if (ft->stream_spp) f.stream_spp = ft->stream_spp;
  f.stream_base = ft->stream_base;
  const std::string window = stream_window_error(f.stream_base, spp, f.stream_spp);
  if (!window.empty()) return rh::set_error(RH_ERR_ARG, w + ": " + window);
  const int mode = o->offset_mode;
  const bool dev = (o->flags & RH_FLAG_DEVICE_OUT) != 0, dev_off = (o->flags & RH_FLAG_DEVICE_OFFSETS) != 0;
  if (dev && (rc = check_device_outputs(D, w, {{ft->albedo, 8, "albedo"}, {ft->normal, 8, "normal"}, {ft->depth, 8, "depth"},
                                               {ft->hits, 8, "hits"}, {want_ids ? hit_ids_out : nullptr, 8, "hit_ids_out"}})))
    return rc;
  RH_CUDA(cudaSetDevice(D->dev));
  const bool host_offsets = (mode == RH_OFFSETS_F64 || mode == RH_OFFSETS_F32) && !dev_off;
  const size_t W = (size_t)o->width, row_samples = W * spp;
  const int rows = f.rows_local;
  const uint64_t per_chunk = (host_offsets || !dev) ? kFeatureChunkSamples : kFeatureLaunchSamples;
  const int chunk_rows = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)rows, per_chunk / row_samples));
  const size_t chunk_px = (size_t)chunk_rows * W, chunk_samples = chunk_px * spp;
  const size_t tile_bytes = mode == RH_OFFSETS_TILED_F64 && !dev_off ? (size_t)o->offset_tile * o->offset_tile * spp * f.off_elem : 0;

  // scratch: claim cursor, then (host buffers) the tile, one chunk of offsets and one chunk of each host output
  Device::Scratch& sc = D->lane[0];  // the render's deep-stack scratch covers grid x block of feature_kernel
  if ((rc = sc.deep.reserve((size_t)scene->deep_entries * D->max_threads * sizeof(uint2)))) return rc;
  size_t at = kQueryCursorBytes;
  auto carve = [&](bool need, size_t bytes) {
    const size_t here = at;
    if (need) at += (bytes + 255) / 256 * 256;
    return need ? here : 0;
  };
  const size_t s_tile = carve(tile_bytes > 0, tile_bytes), s_off = carve(host_offsets, chunk_samples * f.off_elem);
  const size_t s_albedo = carve(!dev && ft->albedo, chunk_px * 3 * sizeof(double)), s_normal = carve(!dev && ft->normal, chunk_px * 3 * sizeof(double));
  const size_t s_depth = carve(!dev && ft->depth, chunk_px * sizeof(double)), s_hits = carve(!dev && ft->hits, chunk_px * sizeof(uint32_t));
  const size_t s_ids = carve(!dev && want_ids, chunk_samples * sizeof(int2));
  if ((rc = D->query.reserve(at))) return rc;
  char* scratch = (char*)D->query.p;

  ChunkParams P = frame_chunk_params(f);
  QueryParams Q{};
  Q.exact_boxes = (o->flags & RH_FLAG_EXACT_BOXES) ? 1 : 0;
  Q.deep_stack = (uint2*)sc.deep.p;
  Q.deep_stride = (uint32_t)D->max_threads;
  Q.cursor = (uint32_t*)scratch;
  uint32_t launches = 0, chunks = 0;
  size_t uploaded = 0;
  RH_CUDA(cudaEventRecord(D->ev_begin, D->stream));
  if (tile_bytes) RH_CUDA(cudaMemcpyAsync(scratch + s_tile, o->offsets, tile_bytes, cudaMemcpyHostToDevice, D->stream));
  for (int r0 = 0; r0 < rows; r0 += chunk_rows) {
    const int n_rows = std::min(chunk_rows, rows - r0);
    const size_t px0 = (size_t)r0 * W, n_px = (size_t)n_rows * W;
    P.first_row = (uint32_t)r0;
    P.n_rows = (uint32_t)n_rows;
    P.n_samples = (uint32_t)(n_px * spp);
    P.offset_index = kOffIndexLocal;
    if (mode == RH_OFFSETS_TILED_F64) {
      P.offsets = dev_off ? o->offsets : scratch + s_tile;
    } else if (host_offsets) {
      if ((rc = upload_offset_rows(f, row_samples, r0, n_rows, scratch + s_off, D->stream, &uploaded))) return rc;
      P.offsets = scratch + s_off;
    } else if (mode == RH_OFFSETS_F64 || mode == RH_OFFSETS_F32) {  // device offsets: the shard's compact rows or the frame's
      if (o->flags & RH_FLAG_SHARD_OFFSETS) P.offsets = (const char*)o->offsets + px0 * spp * f.off_elem;
      else {
        P.offsets = o->offsets;
        P.offset_index = kOffIndexGlobal;
      }
    }
    auto out = [&](void* user, size_t px_bytes, size_t s) -> void* {
      return !user ? nullptr : dev ? (void*)((char*)user + px0 * px_bytes) : (void*)(scratch + s);
    };
    FeatureParams F{};
    F.albedo = (double*)out(ft->albedo, 3 * sizeof(double), s_albedo);
    F.normal = (double*)out(ft->normal, 3 * sizeof(double), s_normal);
    F.depth = (double*)out(ft->depth, sizeof(double), s_depth);
    F.hits = (uint32_t*)out(ft->hits, sizeof(uint32_t), s_hits);
    F.hit_ids = (int2*)out(want_ids ? hit_ids_out : nullptr, spp * sizeof(int2), s_ids);
    Q.n = (uint32_t)n_px;
    RH_CUDA(cudaMemsetAsync(Q.cursor, 0, sizeof(uint32_t), D->stream));
    launch_features(scene->view, f.cam, P, Q, F, D->n_sms, D->stream);
    RH_CUDA(cudaGetLastError());
    launches++;
    chunks++;
    if (!dev) {
      auto back = [&](void* user, size_t px_bytes, const void* src) -> int {
        if (user) RH_CUDA(cudaMemcpyAsync((char*)user + px0 * px_bytes, src, n_px * px_bytes, cudaMemcpyDeviceToHost, D->stream));
        return RH_OK;
      };
      if ((rc = back(ft->albedo, 3 * sizeof(double), F.albedo)) || (rc = back(ft->normal, 3 * sizeof(double), F.normal)) ||
          (rc = back(ft->depth, sizeof(double), F.depth)) || (rc = back(ft->hits, sizeof(uint32_t), F.hits)) ||
          (rc = back(want_ids ? hit_ids_out : nullptr, spp * sizeof(int2), F.hit_ids)))
        return rc;
    }
  }
  RH_CUDA(cudaEventRecord(D->ev_end, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  g_launches.fetch_add(launches, std::memory_order_relaxed);
  if (stats) {
    memset(stats, 0, sizeof *stats);
    stats->rays_primary = f.rays_primary;
    stats->chunks = chunks;
    stats->kernel_launches = launches;
    float ms = 0;
    cudaEventElapsedTime(&ms, D->ev_begin, D->ev_end);
    stats->ms_total = ms;
  }
  return RH_OK;
}

// ------------------------------------------------------------------ light groups
// rh_render_light_groups is a render (render_frame's checks, run_frame's plan, queues, overflow retry and passes) whose
// shadow kernels also add each group's terms beside the sample's, and whose chunks end with the group sink beside the
// resolve.  Like a list frame it uses the scene's learned state without changing it.
int light_groups_on(Device* D, const rh_scene* scene, const rh_camera* camera, const rh_render_opts* o, const rh_light_groups* lg,
                    uint8_t* rgb_out, int32_t* hit_ids_out, rh_stats* stats) {
  const std::string w = "rh_render_light_groups";
  if (!lg) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  if (o && (o->flags & (RH_FLAG_PEER_FRAMES | RH_FLAG_COUNT)))
    return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_PEER_FRAMES and RH_FLAG_COUNT are not supported");
  if (lg->n_groups < 1 || lg->n_groups > (uint32_t)kMaxGroups) return rh::set_error(RH_ERR_ARG, w + ": n_groups must be 1..16");
  if (lg->reserved_) return rh::set_error(RH_ERR_ARG, w + ": reserved_ must be 0");
  if (!lg->out) return rh::set_error(RH_ERR_ARG, w + ": out is null");
  Frame f;
  f.n_groups = lg->n_groups;
  int rc = render_frame(D, scene, camera, o, rgb_out, hit_ids_out, &f, "rh_render_light_groups");
  if (rc) return rc;
  const uint32_t n_lights = scene->view.n_lights;
  if (n_lights > (uint32_t)kMaskLights) return rh::set_error(RH_ERR_ARG, w + ": scenes with more than 32 lights are not supported");
  if (n_lights && !lg->group_of_light) return rh::set_error(RH_ERR_ARG, w + ": group_of_light is null");
  for (uint32_t l = 0; l < n_lights; l++) {
    const uint32_t g = lg->group_of_light[l];
    if (g >= lg->n_groups)
      return rh::set_error(RH_ERR_ARG, w + ": group_of_light[" + std::to_string(l) + "] = " + std::to_string(g) + " is not below n_groups");
    f.group_mask[g] |= 1u << l;
  }
  f.group_out = lg->out;
  if ((o->flags & RH_FLAG_DEVICE_OUT) && (rc = check_device_outputs(D, w, {{lg->out, 8, "out"}}))) return rc;
  return run_frame(D, scene, f, stats);
}

// ------------------------------------------------------------------ camera batches
// rh_render_views is one render (render_frame's checks, run_frame's plan, queues, overflow retry and passes) of a tall
// frame whose local rows are [view][rows]: pass 0 builds each row's rays with its view's camera, and the chunks end with
// a sink that decides padding rows per view.  Like a list frame it uses the scene's learned state without changing it.
int views_on(Device* D, const rh_scene* scene, const rh_views* vw, const rh_render_opts* o, uint8_t* rgb_out, double* linear_out,
             int32_t* hit_ids_out, rh_stats* stats) {
  const std::string w = "rh_render_views";
  if (!vw || !o) return rh::set_error(RH_ERR_ARG, w + ": null argument");
  if (o->flags & (RH_FLAG_PEER_FRAMES | RH_FLAG_COUNT))
    return rh::set_error(RH_ERR_ARG, w + ": RH_FLAG_PEER_FRAMES and RH_FLAG_COUNT are not supported");
  if (vw->n_views < 1 || vw->n_views > kMaxViews) return rh::set_error(RH_ERR_ARG, w + ": n_views must be 1..65536");
  if (!vw->cameras) return rh::set_error(RH_ERR_ARG, w + ": cameras is null");
  if (vw->reserved_) return rh::set_error(RH_ERR_ARG, w + ": reserved_ must be 0");
  if (vw->seeds && o->offset_mode != RH_OFFSETS_SPLITMIX64)
    return rh::set_error(RH_ERR_ARG, w + ": seeds go with RH_OFFSETS_SPLITMIX64 only");
  if (!rgb_out && !linear_out) return rh::set_error(RH_ERR_ARG, w + ": rgb_out and linear_out are both null");
  const uint32_t V = vw->n_views;
  for (uint32_t v = 0; v < V; v++) {
    const std::string cam_err = camera_error(vw->cameras[v]);
    if (!cam_err.empty()) return rh::set_error(RH_ERR_ARG, w + ": cameras[" + std::to_string(v) + "]: " + cam_err);
  }
  Frame f;
  f.views = true;
  int rc = render_frame(D, scene, &vw->cameras[0], o, rgb_out, hit_ids_out, &f, "rh_render_views");
  if (rc) return rc;
  const int rows = f.rows_local, W = f.o.width;
  if ((uint64_t)V * rows > 0x7fffffffu) return rh::set_error(RH_ERR_ARG, w + ": n_views x shard rows must be below 2^31");
  if ((o->flags & RH_FLAG_DEVICE_OUT) &&
      (rc = check_device_outputs(D, w, {{rgb_out, 1, "rgb_out"}, {linear_out, 8, "linear_out"},
                                        {(o->flags & RH_FLAG_HIT_IDS) ? hit_ids_out : nullptr, 1, "hit_ids_out"}})))
    return rc;
  RH_CUDA(cudaSetDevice(D->dev));
  // the camera table and the seeds, behind one another in one buffer
  std::vector<CameraParams> cams(V);
  for (uint32_t v = 0; v < V; v++) cams[v] = make_camera(vw->cameras[v], W, f.o.height);
  const size_t cam_bytes = V * sizeof(CameraParams), seed_bytes = vw->seeds ? V * sizeof(uint64_t) : 0;
  if ((rc = D->views.reserve(cam_bytes + seed_bytes))) return rc;
  f.cams = (const CameraParams*)D->views.p;
  f.uploads.push_back({D->views.p, cams.data(), cam_bytes});
  if (vw->seeds) {
    f.view_seeds = (const unsigned long long*)((char*)D->views.p + cam_bytes);
    f.uploads.push_back({(char*)D->views.p + cam_bytes, vw->seeds, seed_bytes});
  }
  // host per-pixel offsets are the same for every view: staged once, then read as device offsets are
  const int mode = f.o.offset_mode;
  if ((mode == RH_OFFSETS_F64 || mode == RH_OFFSETS_F32) && !(f.o.flags & RH_FLAG_DEVICE_OFFSETS)) {
    const int off_rows = (f.o.flags & RH_FLAG_SHARD_OFFSETS) ? rows : f.o.height;
    const size_t bytes = (size_t)off_rows * W * f.o.spp * f.off_elem;
    if (D->offsets.reserve(bytes)) {
      cudaGetLastError();  // (clears the failed allocation)
      return rh::set_error(RH_ERR_OOM, w + ": the host offsets (" + std::to_string(bytes) + " bytes) do not fit in device memory");
    }
    f.uploads.push_back({D->offsets.p, f.o.offsets, bytes});
    f.o.offsets = D->offsets.p;
    f.o.flags |= RH_FLAG_DEVICE_OFFSETS;
  }
  f.view_rows = (uint32_t)rows;
  f.rows_local = (int)(V * rows);
  f.out_bytes *= V;
  f.ids_bytes *= V;
  f.rays_primary *= V;
  f.linear = linear_out;
  f.linear_bytes = (size_t)f.rows_local * W * 3 * sizeof(double);
  return run_frame(D, scene, f, stats);
}

}  // namespace

// ================================================================== C ABI
extern "C" {

const char* rh_last_error(void) { return rh::g_err.c_str(); }
int rh_abi_version(void) { return RH_ABI_VERSION; }
uint64_t rh_launch_count(void) { return g_launches.load(); }

int rh_init(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_dev) return rh::set_error(RH_ERR_STATE, "rh_init: already initialised");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return rh::set_error(RH_ERR_CUDA, std::string("rh_init: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback");
  if (device < 0) RH_CUDA(cudaGetDevice(&device));
  if (device >= n) return rh::set_error(RH_ERR_ARG, "rh_init: device index out of range");
  auto d = std::make_unique<Device>();
  int rc = d->open(device);
  if (rc) { d->close(); return rc; }
  g_dev = std::move(d);
  return RH_OK;
}

void rh_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_dev) g_dev->close();
  g_dev.reset();
}

int rh_scene_create(const rh_scene_desc* desc, rh_scene** out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_scene_create: call rh_init first");
  return scene_create_on(g_dev.get(), desc, out);
}
void rh_scene_destroy(rh_scene* scene) { scene_destroy(scene); }
int rh_scene_info(const rh_scene* scene, double* setup_ms3, int32_t* info4) {
  if (!scene) return rh::set_error(RH_ERR_ARG, "rh_scene_info: null scene");
  if (setup_ms3) {
    setup_ms3[0] = scene->ms_trees;
    setup_ms3[1] = scene->ms_light_tables;
    setup_ms3[2] = scene->ms_upload;
  }
  if (info4) {
    info4[0] = (int32_t)scene->view.tables_in_smem;
    info4[1] = (int32_t)scene->view.shadow_fast;
    info4[2] = (int32_t)scene->max_tree_depth;
    info4[3] = (int32_t)scene->deep_entries;
  }
  return RH_OK;
}

int rh_scene_light_tables(const rh_scene* scene, uint32_t* info4, float* maps_out, uint32_t* index_out, uint16_t* lit_out) {
  if (!scene) return rh::set_error(RH_ERR_ARG, "rh_scene_light_tables: null scene");
  const SceneView& v = scene->view;
  RH_CUDA(cudaSetDevice(scene->device->dev));
  if (info4) {
    info4[0] = scene->n_light_maps;
    info4[1] = v.light_map_res;
    info4[2] = v.lit_flags ? 1u : 0u;
    info4[3] = v.n_tris;
  }
  if (maps_out && scene->n_light_maps)
    RH_CUDA(cudaMemcpy(maps_out, v.light_maps, (size_t)scene->n_light_maps * 6 * v.light_map_res * v.light_map_res * sizeof(float),
                       cudaMemcpyDeviceToHost));
  if (index_out && v.light_map_index)
    RH_CUDA(cudaMemcpy(index_out, v.light_map_index, (size_t)v.n_lights * kOccMeshes * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (lit_out && v.lit_flags) RH_CUDA(cudaMemcpy(lit_out, v.lit_flags, (size_t)v.n_tris * sizeof(uint16_t), cudaMemcpyDeviceToHost));
  return RH_OK;
}

int rh_scene_update(rh_scene* scene, const rh_material* materials, uint32_t n_materials, const rh_light* lights, uint32_t n_lights,
                    rh_update_info* info) {
  const std::string w = "rh_scene_update";
  if (!scene) return rh::set_error(RH_ERR_ARG, w + ": null scene");
  int cls = 0;
  std::unique_ptr<rh_scene> N;
  int rc = scene_update_prepare(scene, materials, n_materials, lights, n_lights, info, w, &cls, &N);
  if (rc) return rc;
  scene_update_commit(scene, std::move(N), cls);
  return RH_OK;
}

int rh_cull_tree_build(const rh_tri* tris, uint32_t n_tris, uint32_t* order_out, rh_node* nodes_out, uint32_t* n_nodes_out,
                       uint32_t* depth_out) {
  if ((!tris && n_tris) || !order_out || !nodes_out || !n_nodes_out) return rh::set_error(RH_ERR_ARG, "rh_cull_tree_build: null argument");
  try {
    SahTree sah(tris);
    std::vector<uint32_t> slots(n_tris);
    for (uint32_t i = 0; i < n_tris; i++) slots[i] = i;
    sah.run(slots);
    TriVec permuted(sah.order.size());
    for (size_t k = 0; k < sah.order.size(); k++) permuted[k] = tris[sah.order[k]];
    sah.refit(permuted);
    if (sah.nodes.size() > 2 * (size_t)n_tris + 1) return rh::set_error(RH_ERR_STATE, "rh_cull_tree_build: more nodes than a binary tree has");
    memcpy(order_out, sah.order.data(), sah.order.size() * sizeof(uint32_t));
    memcpy(nodes_out, sah.nodes.data(), sah.nodes.size() * sizeof(rh_node));
    *n_nodes_out = (uint32_t)sah.nodes.size();
    if (depth_out) *depth_out = sah.max_depth;
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, "rh_cull_tree_build: out of host memory");
  }
  return RH_OK;
}

int rh_scene_record_bytes(const rh_scene* scene, uint64_t* bytes5) {
  if (!scene || !bytes5) return rh::set_error(RH_ERR_ARG, "rh_scene_record_bytes: null argument");
  bytes5[0] = scene->wide32.bytes;
  bytes5[1] = scene->tris.bytes;
  bytes5[2] = scene->shade.bytes;
  bytes5[3] = scene->texels.bytes;
  bytes5[4] = scene->light_maps.bytes + scene->lit_flags.bytes;
  return RH_OK;
}

int rh_render(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, uint8_t* rgb_out,
              int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render: call rh_init first");
  return render_on(g_dev.get(), scene, camera, opts, rgb_out, hit_ids_out, stats);
}

int rh_trace_rays(const rh_scene* scene, const double* rays, uint64_t n, const rh_trace_opts* opts, double* colors_out,
                  int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_trace_rays: call rh_init first");
  return trace_on(g_dev.get(), scene, rays, n, opts, colors_out, hit_ids_out, stats);
}

int rh_accum_create(int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                    rh_accum** out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_accum_create: call rh_init first");
  return accum_create_on(g_dev.get(), width, height, shard_index, shard_count, band_height, stream_spp, out);
}
int rh_accum_reset(rh_accum* acc) {
  if (!acc) return rh::set_error(RH_ERR_ARG, "rh_accum_reset: null accumulator");
  acc->n = 0;
  acc->scene = nullptr;
  return RH_OK;
}
void rh_accum_destroy(rh_accum* acc) {
  if (!acc) return;
  if (acc->dev >= 0) cudaSetDevice(acc->dev);  // (not through acc->device: that context may have been shut down)
  acc->sums.release();
  delete acc;
}
int rh_render_accumulate(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, rh_accum* acc,
                         uint8_t* rgb_out, double* linear_out, int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render_accumulate: call rh_init first");
  return accumulate_on(g_dev.get(), scene, camera, opts, acc, rgb_out, linear_out, hit_ids_out, stats);
}

int rh_adaptive_create(int width, int height, int shard_index, int shard_count, int band_height, uint32_t stream_spp,
                       rh_adaptive** out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_adaptive_create: call rh_init first");
  return adaptive_create_on(g_dev.get(), width, height, shard_index, shard_count, band_height, stream_spp, out);
}
int rh_adaptive_reset(rh_adaptive* ad) {
  if (!ad) return rh::set_error(RH_ERR_ARG, "rh_adaptive_reset: null state");
  return adaptive_reset_on(ad);
}
void rh_adaptive_destroy(rh_adaptive* ad) {
  if (!ad) return;
  if (ad->dev >= 0) cudaSetDevice(ad->dev);  // (not through ad->device: that context may have been shut down)
  adaptive_release(ad);
  delete ad;
}
int rh_render_adaptive(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, const rh_adaptive_opts* aopts,
                       rh_adaptive* ad, uint8_t* rgb_out, double* linear_out, uint64_t* n_active_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render_adaptive: call rh_init first");
  return adaptive_on(g_dev.get(), scene, camera, opts, aopts, ad, rgb_out, linear_out, n_active_out, stats);
}
int rh_adaptive_state(const rh_adaptive* ad, uint32_t* counts_out, double* sums_out, double* sumsq_out, int32_t flags) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_adaptive_state: call rh_init first");
  return adaptive_state_on(g_dev.get(), ad, counts_out, sums_out, sumsq_out, flags);
}

int rh_closest_intersection(const rh_scene* scene, const double* rays, uint64_t n, rh_hit* hits_out, int32_t flags) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_closest_intersection: call rh_init first");
  return query_on(g_dev.get(), scene, -1, rays, n, hits_out, flags, "rh_closest_intersection");
}
int rh_shadow_intersection(const rh_scene* scene, uint32_t light, const double* rays, uint64_t n, uint8_t* occluded_out,
                           int32_t flags) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_shadow_intersection: call rh_init first");
  return query_on(g_dev.get(), scene, light, rays, n, occluded_out, flags, "rh_shadow_intersection");
}

int rh_render_features(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts, const rh_features* features,
                       int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render_features: call rh_init first");
  return features_on(g_dev.get(), scene, camera, opts, features, hit_ids_out, stats);
}

int rh_render_light_groups(const rh_scene* scene, const rh_camera* camera, const rh_render_opts* opts,
                           const rh_light_groups* groups, uint8_t* rgb_out, int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render_light_groups: call rh_init first");
  return light_groups_on(g_dev.get(), scene, camera, opts, groups, rgb_out, hit_ids_out, stats);
}

int rh_render_views(const rh_scene* scene, const rh_views* views, const rh_render_opts* opts, uint8_t* rgb_out,
                    double* linear_out, int32_t* hit_ids_out, rh_stats* stats) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_render_views: call rh_init first");
  return views_on(g_dev.get(), scene, views, opts, rgb_out, linear_out, hit_ids_out, stats);
}

int rh_default_band_height(int height, int shard_count) {
  if (shard_count <= 1) return height > 0 ? height : 1;
  // interleave bands so that every shard sees every part of the frame (SURVEY 8e).  Narrow bands balance the shards (the
  // dragon covers the middle third of the bench frame; measured on 8 B200: 16 rows 6.64 ms, 4 rows 6.60, 1 row 6.52 per
  // frame); 4 rows keep a shard's offset upload at a few hundred copies per frame.
  int bh = 4;
  while (bh > 1 && height / (bh * shard_count) < 4) bh /= 2;
  return bh;
}
int rh_shard_rows(int height, int shard_count, int band_height) {
  if (height <= 0 || shard_count <= 0 || band_height <= 0) return 0;
  const int n_bands = (height + band_height - 1) / band_height;
  return ((n_bands + shard_count - 1) / shard_count) * band_height;
}

int rh_deinterleave_bands(const uint8_t* gathered_dev, uint8_t* out_dev, int width, int height, int shard_count,
                          int band_height) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_deinterleave_bands: call rh_init first");
  if (!gathered_dev || !out_dev || width <= 0 || height <= 0 || shard_count <= 0 || band_height <= 0)
    return rh::set_error(RH_ERR_ARG, "rh_deinterleave_bands: bad argument");
  RH_CUDA(cudaSetDevice(g_dev->dev));
  launch_deinterleave(gathered_dev, out_dev, width, height, shard_count, band_height, g_dev->stream);
  g_launches.fetch_add(1);
  RH_CUDA(cudaGetLastError());
  RH_CUDA(cudaStreamSynchronize(g_dev->stream));
  return RH_OK;
}

// ------------------------------------------------------------------ several GPUs from one process
}  // extern "C"

struct rh_multi_scene {
  std::vector<rh_scene*> replica;  // one per GPU of the multi context
};

namespace {
std::vector<std::unique_ptr<Device>> g_multi;  // rh_multi_init
DevBuf g_multi_frame;                            // the full frame on device 0
}  // namespace

extern "C" {

int rh_multi_init(int n_gpus) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_multi.empty()) return rh::set_error(RH_ERR_STATE, "rh_multi_init: already initialised");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return rh::set_error(RH_ERR_CUDA, std::string("rh_multi_init: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback");
  if (n_gpus <= 0 || n_gpus > n || n_gpus > kMaxPeers) return rh::set_error(RH_ERR_ARG, "rh_multi_init: n_gpus out of range");
  std::vector<std::unique_ptr<Device>> devs;
  for (int g = 0; g < n_gpus; g++) {
    auto d = std::make_unique<Device>();
    int rc = d->open(g);
    if (rc) {
      d->close();
      for (auto& x : devs) x->close();
      return rc;
    }
    if (g > 0) {  // stores into device 0's frame
      int can = 0;
      cudaDeviceCanAccessPeer(&can, g, 0);
      cudaError_t pe = can ? cudaDeviceEnablePeerAccess(0, 0) : cudaErrorPeerAccessUnsupported;
      if (pe == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); pe = cudaSuccess; }
      if (pe != cudaSuccess) {
        d->close();
        for (auto& x : devs) x->close();
        return rh::set_error(RH_ERR_CUDA, std::string("rh_multi_init: no peer access from a device to device 0: ") + cudaGetErrorString(pe));
      }
    }
    devs.push_back(std::move(d));
  }
  g_multi = std::move(devs);
  return RH_OK;
}

void rh_multi_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_multi.empty()) {
    cudaSetDevice(g_multi[0]->dev);
    g_multi_frame.release();
  }
  for (auto& d : g_multi) d->close();
  g_multi.clear();
}

int rh_multi_gpu_count(void) { return (int)g_multi.size(); }

int rh_multi_scene_create(const rh_scene_desc* desc, rh_multi_scene** out) {
  if (g_multi.empty()) return rh::set_error(RH_ERR_STATE, "rh_multi_scene_create: call rh_multi_init first");
  if (!out) return rh::set_error(RH_ERR_ARG, "rh_multi_scene_create: null argument");
  auto ms = std::make_unique<rh_multi_scene>();
  for (auto& d : g_multi) {
    rh_scene* s = nullptr;
    int rc = scene_create_on(d.get(), desc, &s);
    if (rc) {
      for (rh_scene* r : ms->replica) scene_destroy(r);
      return rc;
    }
    ms->replica.push_back(s);
  }
  *out = ms.release();
  return RH_OK;
}

void rh_multi_scene_destroy(rh_multi_scene* scene) {
  if (!scene) return;
  for (rh_scene* r : scene->replica) scene_destroy(r);
  delete scene;
}

int rh_multi_scene_update(rh_multi_scene* scene, const rh_material* materials, uint32_t n_materials, const rh_light* lights,
                          uint32_t n_lights, rh_update_info* info) {
  const std::string w = "rh_multi_scene_update";
  if (!scene || scene->replica.empty()) return rh::set_error(RH_ERR_ARG, w + ": null scene");
  // every replica is prepared before any is swapped: the update takes on all GPUs or on none
  std::vector<std::unique_ptr<rh_scene>> prepared(scene->replica.size());
  int cls = 0;
  for (size_t g = 0; g < scene->replica.size(); g++) {
    int rc = scene_update_prepare(scene->replica[g], materials, n_materials, lights, n_lights, g == 0 ? info : nullptr, w, &cls, &prepared[g]);
    if (rc) {
      for (auto& p : prepared)
        if (p) scene_destroy(p.release());
      return rc;
    }
  }
  for (size_t g = 0; g < scene->replica.size(); g++) scene_update_commit(scene->replica[g], std::move(prepared[g]), cls);
  return RH_OK;
}

int rh_multi_render(const rh_multi_scene* scene, const rh_camera* camera, const rh_render_opts* opts, uint8_t* rgb_out,
                    rh_stats* stats) {
  if (g_multi.empty()) return rh::set_error(RH_ERR_STATE, "rh_multi_render: call rh_multi_init first");
  if (!scene || !camera || !opts || !rgb_out) return rh::set_error(RH_ERR_ARG, "rh_multi_render: null argument");
  const int G = (int)g_multi.size();
  if ((int)scene->replica.size() != G) return rh::set_error(RH_ERR_ARG, "rh_multi_render: scene belongs to another multi context");
  if (opts->flags & (RH_FLAG_HIT_IDS | RH_FLAG_DEVICE_OUT | RH_FLAG_DEVICE_OFFSETS))
    return rh::set_error(RH_ERR_ARG, "rh_multi_render: hit ids and device pointers are not supported here");
  if (opts->width <= 0 || opts->height <= 0) return rh::set_error(RH_ERR_ARG, "rh_multi_render: bad width/height");
  const size_t bytes = (size_t)opts->width * opts->height * 3;
  RH_CUDA(cudaSetDevice(g_multi[0]->dev));
  int rc = g_multi_frame.reserve(bytes);
  if (rc) return rc;
  void* frame = g_multi_frame.p;
  std::vector<int> rcs(G, RH_OK);
  std::vector<std::string> errs(G);
  std::vector<rh_stats> st(G);
  std::vector<std::thread> threads;
  for (int g = 0; g < G; g++)
    threads.emplace_back([&, g]() {
      rh_render_opts o = *opts;
      o.shard_index = g;
      o.shard_count = G;
      o.flags |= RH_FLAG_PEER_FRAMES;
      o.n_peer_frames = 1;
      void* frames[1] = {frame};
      o.peer_frames = frames;
      rcs[g] = render_on(g_multi[g].get(), scene->replica[g], camera, &o, nullptr, nullptr, &st[g]);
      if (rcs[g]) errs[g] = rh_last_error();  // thread-local: carry it to the caller's thread
    });
  for (auto& t : threads) t.join();
  for (int g = 0; g < G; g++)
    if (rcs[g]) return rh::set_error(rcs[g], "rh_multi_render (GPU " + std::to_string(g) + "): " + errs[g]);
  RH_CUDA(cudaSetDevice(g_multi[0]->dev));
  RH_CUDA(cudaMemcpy(rgb_out, frame, bytes, cudaMemcpyDeviceToHost));  // every shard has synchronised its stream
  if (stats) {
    *stats = st[0];
    for (int g = 1; g < G; g++) {
      const rh_stats& s = st[g];
      stats->rays_primary += s.rays_primary; stats->rays_reflect += s.rays_reflect; stats->rays_probe += s.rays_probe;
      stats->rays_exit += s.rays_exit; stats->rays_shadow += s.rays_shadow; stats->rays_shadow_culled += s.rays_shadow_culled;
      stats->shadow_tasks += s.shadow_tasks; stats->queued_rays += s.queued_rays;
      stats->box_tests += s.box_tests; stats->tri_tests += s.tri_tests; stats->prim_tests += s.prim_tests;
      stats->shade_fetches += s.shade_fetches; stats->texel_fetches += s.texel_fetches; stats->node_visits += s.node_visits;
      stats->shadow_box_tests += s.shadow_box_tests; stats->shadow_tri_tests += s.shadow_tri_tests;
      stats->shadow_prim_tests += s.shadow_prim_tests; stats->shadow_node_visits += s.shadow_node_visits;
      stats->node_visits_global += s.node_visits_global; stats->shadow_node_visits_global += s.shadow_node_visits_global;
      stats->tri_records += s.tri_records; stats->shadow_tri_records += s.shadow_tri_records;
      stats->shadow_tasks_queued += s.shadow_tasks_queued; stats->shadow_walk_pairs += s.shadow_walk_pairs;
      stats->deep_stack_pushes += s.deep_stack_pushes;
      stats->upload_bytes += s.upload_bytes;
      stats->ms_total = std::max(stats->ms_total, s.ms_total);
      stats->ms_trace = std::max(stats->ms_trace, s.ms_trace);
      stats->ms_shadow = std::max(stats->ms_shadow, s.ms_shadow);
      stats->ms_resolve = std::max(stats->ms_resolve, s.ms_resolve);
      stats->kernel_launches += s.kernel_launches;
      stats->chunks += s.chunks;
      stats->negative_channels += s.negative_channels;
      stats->queue_factor = std::max(stats->queue_factor, s.queue_factor);
    }
  }
  return RH_OK;
}

int rh_peer_alloc(size_t bytes, void** dev_ptr_out, unsigned char handle_out[RH_PEER_HANDLE_BYTES]) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_peer_alloc: call rh_init first");
  if (!bytes || !dev_ptr_out || !handle_out) return rh::set_error(RH_ERR_ARG, "rh_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == RH_PEER_HANDLE_BYTES, "CUDA IPC handle size");
  RH_CUDA(cudaSetDevice(g_dev->dev));
  void* p = nullptr;
  RH_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return rh::set_error(RH_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
  }
  memcpy(handle_out, &h, sizeof h);
  *dev_ptr_out = p;
  return RH_OK;
}
int rh_peer_open(const unsigned char handle[RH_PEER_HANDLE_BYTES], void** dev_ptr_out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_peer_open: call rh_init first");
  if (!handle || !dev_ptr_out) return rh::set_error(RH_ERR_ARG, "rh_peer_open: bad argument");
  RH_CUDA(cudaSetDevice(g_dev->dev));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  RH_CUDA(cudaIpcOpenMemHandle(dev_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return RH_OK;
}
int rh_peer_close(void* dev_ptr) {
  if (!dev_ptr) return RH_OK;
  RH_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return RH_OK;
}
int rh_peer_free(void* dev_ptr) {
  if (!dev_ptr) return RH_OK;
  RH_CUDA(cudaFree(dev_ptr));
  return RH_OK;
}

int rh_bench_gather(uint64_t bytes, int iters, double* gbs_out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_bench_gather: call rh_init first");
  if (bytes < 128 || iters <= 0 || !gbs_out) return rh::set_error(RH_ERR_ARG, "rh_bench_gather: bad argument");
  Device* D = g_dev.get();
  RH_CUDA(cudaSetDevice(D->dev));
  void* buf = nullptr;
  double2* sink = nullptr;
  RH_CUDA(cudaMalloc(&buf, bytes));
  RH_CUDA(cudaMalloc(&sink, 64));
  RH_CUDA(cudaMemsetAsync(buf, 0, bytes, D->stream));
  const int block = 256, grid = D->n_sms * 8;
  const uint32_t loads = 64;
  launch_gather_bench((const double2*)buf, bytes / 128, loads, sink, grid, block, D->stream);  // warm-up
  RH_CUDA(cudaEventRecord(D->ev_begin, D->stream));
  for (int i = 0; i < iters; i++) launch_gather_bench((const double2*)buf, bytes / 128, loads, sink, grid, block, D->stream);
  RH_CUDA(cudaEventRecord(D->ev_end, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  g_launches.fetch_add(iters + 1);
  float ms = 0;
  cudaEventElapsedTime(&ms, D->ev_begin, D->ev_end);
  *gbs_out = (double)grid * block * loads * 128.0 * iters / (ms * 1e-3) / 1e9;
  cudaFree(buf);
  cudaFree(sink);
  RH_CUDA(cudaGetLastError());
  return RH_OK;
}

int rh_bench_stream(uint64_t bytes, int iters, double* gbs_out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_bench_stream: call rh_init first");
  if (bytes < 4096 || iters <= 0 || !gbs_out) return rh::set_error(RH_ERR_ARG, "rh_bench_stream: bad argument");
  Device* D = g_dev.get();
  RH_CUDA(cudaSetDevice(D->dev));
  void* buf = nullptr;
  double2* sink = nullptr;
  RH_CUDA(cudaMalloc(&buf, bytes));
  RH_CUDA(cudaMalloc(&sink, 64));
  RH_CUDA(cudaMemsetAsync(buf, 0, bytes, D->stream));
  const int block = 256, grid = D->n_sms * 8;
  const uint64_t n = bytes / 16;
  for (int i = 0; i < 2; i++) launch_stream_bench((const double2*)buf, n, sink, grid, block, D->stream);  // warm-up: fills L2
  RH_CUDA(cudaEventRecord(D->ev_begin, D->stream));
  for (int i = 0; i < iters; i++) launch_stream_bench((const double2*)buf, n, sink, grid, block, D->stream);
  RH_CUDA(cudaEventRecord(D->ev_end, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  g_launches.fetch_add(iters + 2);
  float ms = 0;
  cudaEventElapsedTime(&ms, D->ev_begin, D->ev_end);
  *gbs_out = (double)n * 16.0 * iters / (ms * 1e-3) / 1e9;
  cudaFree(buf);
  cudaFree(sink);
  RH_CUDA(cudaGetLastError());
  return RH_OK;
}

int rh_bench_dfma(int iters, double* tflops_out) {
  if (!g_dev) return rh::set_error(RH_ERR_STATE, "rh_bench_dfma: call rh_init first");
  if (iters <= 0 || !tflops_out) return rh::set_error(RH_ERR_ARG, "rh_bench_dfma: bad argument");
  Device* D = g_dev.get();
  RH_CUDA(cudaSetDevice(D->dev));
  double* sink = nullptr;
  RH_CUDA(cudaMalloc(&sink, 64));
  const int block = 256, grid = D->n_sms * 8;
  launch_dfma_bench(sink, iters, grid, block, D->stream);
  RH_CUDA(cudaEventRecord(D->ev_begin, D->stream));
  launch_dfma_bench(sink, iters, grid, block, D->stream);
  RH_CUDA(cudaEventRecord(D->ev_end, D->stream));
  RH_CUDA(cudaStreamSynchronize(D->stream));
  g_launches.fetch_add(2);
  float ms = 0;
  cudaEventElapsedTime(&ms, D->ev_begin, D->ev_end);
  *tflops_out = (double)grid * block * 8.0 * iters * 2.0 / (ms * 1e-3) / 1e12;
  cudaFree(sink);
  RH_CUDA(cudaGetLastError());
  return RH_OK;
}

}  // extern "C"
