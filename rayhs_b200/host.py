"""Host side above the C ABI, mirroring the reference's interface for the ray-casting path.

Names follow src/RayHs.hs: `Rendering` (41-45), `buildRendering` (47-50), `rayTrace` (161-166),
`distributedRayTrace` (190-195), and src/Image.hs: `Image` (21-23), `writePPM` (70-75).
The scene description layer (JSON.hs / Descriptors.hs / Mesh.hs OBJ loader / KDTree.hs build) is
the C++ front end inside librayhs_b200.so (frontend.cpp, host_build.cpp) because GHC is not in
this image; everything below `rayTrace` runs in the sm_100a kernels.  PyTorch is used only for
device buffers and the NCCL all-gather of the row bands (one process per GPU).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import capi
from .capi import check, lib

_initialised = False


def init(device: int = -1) -> None:
    """rh_init on `device` (-1: the current CUDA device).  Raises when no GPU is present."""
    global _initialised
    if not _initialised:
        check(lib().rh_init(int(device)))
        _initialised = True


def shutdown() -> None:
    global _initialised
    if _initialised:
        lib().rh_shutdown()
        _initialised = False


class Scene:
    """Scene.hs:8-10 after `buildScene` (Descriptors.hs:39-55): raw objects, the flattened
    tree arrays, and (lazily) the device copy."""

    def __init__(self, loaded: C.c_void_p):
        self._loaded = loaded
        self._flat = C.c_void_p()
        self._dev = C.c_void_p()
        L = lib()
        w, h, d = C.c_int32(), C.c_int32(), C.c_int32()
        L.rh_loaded_size(loaded, C.byref(w), C.byref(h), C.byref(d))
        self.width, self.height, self.max_depth = w.value, h.value, d.value
        self.camera = capi.rh_camera.from_buffer_copy(L.rh_loaded_camera(loaded).contents)

    # ---- construction (front end)
    @staticmethod
    def from_json(path: str, base_dir: str | None = None) -> "Scene":
        h = C.c_void_p()
        base = base_dir if base_dir is not None else ""
        check(lib().rh_load_json(path.encode(), base.encode(), C.byref(h)))
        return Scene(h)

    @staticmethod
    def from_pack(path: str) -> "Scene":
        h = C.c_void_p()
        check(lib().rh_load_pack(path.encode(), C.byref(h)))
        return Scene(h)

    @staticmethod
    def synthetic(n_tris: int, n_spheres: int, seed: int = 0x5EED) -> "Scene":
        h = C.c_void_p()
        check(lib().rh_make_synthetic(int(n_tris), int(n_spheres), int(seed), C.byref(h)))
        return Scene(h)

    def save_pack(self, path: str) -> None:
        check(lib().rh_save_pack(self._loaded, path.encode()))

    # ---- views
    @property
    def raw(self):
        """POINTER(rh_raw_scene): the scene before any tree build (what the oracle is fed)."""
        return lib().rh_loaded_raw(self._loaded)

    @property
    def flat(self):
        """POINTER(rh_scene_desc): KDTree.hs:68-90 build + flattening, on the host."""
        if not self._flat:
            check(lib().rh_flatten(self.raw, C.byref(self._flat)))
        return lib().rh_flat_desc(self._flat)

    @property
    def device(self) -> C.c_void_p:
        if not self._dev:
            init()
            check(lib().rh_scene_create(self.flat, C.byref(self._dev)))
        return self._dev

    def _info(self):
        ms, info = (C.c_double * 3)(), (C.c_int32 * 4)()
        check(lib().rh_scene_info(self.device, ms, info))
        return list(ms), list(info)

    def light_tables(self) -> dict:
        """The light-space tables rh_scene_create built (cube maps, their index, lit-triangle flags), copied back."""
        import numpy as np

        info = (C.c_uint32 * 4)()
        check(lib().rh_scene_light_tables(self.device, info, None, None, None))
        n_maps, res, has_lit, n_tris = (int(x) for x in info)
        maps = np.empty((n_maps, 6, res, res), dtype=np.float32)
        index = np.full((int(self.flat.contents.n_lights), 8), 0xFFFFFFFF, dtype=np.uint32)
        lit = np.zeros(n_tris, dtype=np.uint16)
        check(lib().rh_scene_light_tables(self.device, info, maps.ctypes.data if n_maps else None, index.ctypes.data if n_maps else None,
                                          lit.ctypes.data if has_lit else None))
        return {"maps": maps, "index": index, "lit": lit if has_lit else None, "res": res}

    @property
    def record_bytes(self) -> dict:
        """Bytes of the gathered records in HBM (cull-tree nodes, triangle / shading records, texels, light-space tables)."""
        b = (C.c_uint64 * 5)()
        check(lib().rh_scene_record_bytes(self.device, b))
        return dict(zip(("nodes", "tris", "shade", "texels", "light_tables"), (int(x) for x in b)))

    @property
    def tables_in_smem(self) -> bool:
        return bool(self._info()[1][0])

    def close(self) -> None:
        L = lib()
        if self._dev:
            L.rh_scene_destroy(self._dev)
            self._dev = C.c_void_p()
        if self._flat:
            L.rh_flat_destroy(self._flat)
            self._flat = C.c_void_p()
        if self._loaded:
            L.rh_loaded_destroy(self._loaded)
            self._loaded = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class Rendering:
    """RayHs.hs:41-45."""
    scene: Scene
    camera: capi.rh_camera
    width: int
    height: int
    maxDepth: int


def buildRendering(scene_json: str, base_dir: str | None = None, width: int | None = None, height: int | None = None) -> Rendering:
    """parseFile + buildRendering (RayHs.hs:197-200, 47-50).  `width`/`height` override the JSON values."""
    sc = Scene.from_json(scene_json, base_dir)
    return Rendering(sc, sc.camera, width or sc.width, height or sc.height, sc.max_depth)


def renderingFromScene(sc: Scene, width: int | None = None, height: int | None = None, maxDepth: int | None = None) -> Rendering:
    return Rendering(sc, sc.camera, width or sc.width, height or sc.height, sc.max_depth if maxDepth is None else maxDepth)


@dataclass
class Image:
    """Image.hs:21-23, already quantised by toIntC (Image.hs:54-55): uint8 [height, width, 3]."""
    width: int
    height: int
    pixels: np.ndarray
    stats: dict = field(default_factory=dict)
    hit_ids: np.ndarray | None = None


def sample_offsets(n_pixels: int, spp: int, seed: int = 24, dtype=np.float64) -> np.ndarray:
    """[n_pixels, spp, 2] offsets (x-0.5, y-0.5), x drawn before y, one stream, pixel-major
    (RayHs.hs:173-188; seed 24 as in RayHs.hs:239)."""
    out = np.empty((n_pixels, spp, 2), dtype=dtype)
    fn = lib().rh_sample_offsets_f64 if dtype == np.float64 else lib().rh_sample_offsets_f32
    fn(int(seed), int(n_pixels), int(spp), out.ctypes.data)
    return out


def _opts(job: Rendering, spp: int, mode: int, offsets_ptr, tile: int, shard_index: int, shard_count: int, band_height: int,
          chunk_samples: int, flags: int) -> capi.rh_render_opts:
    o = capi.rh_render_opts()
    o.width, o.height, o.max_depth, o.spp = job.width, job.height, job.maxDepth, spp
    o.offset_mode, o.offset_tile, o.offsets = mode, tile, offsets_ptr
    o.shard_index, o.shard_count, o.band_height = shard_index, shard_count, band_height
    o.chunk_samples, o.flags = chunk_samples, flags
    return o


def _offset_mode(offsets, tile: int):
    if offsets is None:
        return capi.RH_OFFSETS_NONE, None
    if tile:
        return capi.RH_OFFSETS_TILED_F64, offsets
    if hasattr(offsets, "dtype") and str(offsets.dtype).endswith("float32"):
        return capi.RH_OFFSETS_F32, offsets
    return capi.RH_OFFSETS_F64, offsets


def render(job: Rendering, spp: int = 1, offsets=None, offset_tile: int = 0, want_hit_ids: bool = False,
           shard_index: int = 0, shard_count: int = 1, band_height: int = 0, chunk_samples: int = 0,
           count: bool = False, profile: bool = False, exact_boxes: bool = False, out: np.ndarray | None = None,
           shadow: str | None = None, seed: int | None = None, light_maps: bool = True) -> Image:
    """One rh_render call with HOST buffers (numpy or pinned torch CPU tensors for `offsets`).
    `seed` (instead of `offsets`): the kernel regenerates sample_offsets(width*height, spp, seed) on the device.
    Returns the shard-compact RGB8 rows when shard_count > 1."""
    L = lib()
    mode, off = _offset_mode(offsets, offset_tile)
    off_ptr = None
    seed_box = None
    if seed is not None:
        if offsets is not None:
            raise ValueError("pass either offsets or seed")
        seed_box = C.c_uint64(seed)
        mode, off, off_ptr = capi.RH_OFFSETS_SPLITMIX64, None, C.addressof(seed_box)
    if off is not None:
        off_ptr = off.data_ptr() if hasattr(off, "data_ptr") else off.ctypes.data
        need = (offset_tile * offset_tile if offset_tile else job.width * job.height) * spp * 2
        have = off.numel() if hasattr(off, "numel") else off.size
        if have != need:
            raise ValueError(f"offsets has {have} values, expected {need}")
    bh = band_height or L.rh_default_band_height(job.height, shard_count)
    rows = L.rh_shard_rows(job.height, shard_count, bh)
    flags = ((capi.RH_FLAG_HIT_IDS if want_hit_ids else 0) | (capi.RH_FLAG_COUNT if count else 0)
             | (capi.RH_FLAG_PROFILE if profile else 0) | (capi.RH_FLAG_EXACT_BOXES if exact_boxes else 0) | _shadow_flag(shadow)
             | (0 if light_maps else capi.RH_FLAG_NO_LIGHT_MAPS))
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, chunk_samples, flags)
    rgb = out if out is not None else np.empty((rows, job.width, 3), dtype=np.uint8)
    ids = np.empty((rows, job.width, spp, 2), dtype=np.int32) if want_hit_ids else None
    st = capi.rh_stats()
    check(L.rh_render(job.scene.device, C.byref(job.camera), C.byref(o), rgb.ctypes.data,
                      ids.ctypes.data if ids is not None else None, C.byref(st)))
    return Image(job.width, rows, rgb, st.as_dict(), ids)


# ---- batched ray queries (RayHs.hs:67-71 closestIntersection, RayHs.hs:74-87 shadowIntersection)

# one rh_hit record (include/rayhs_b200.h)
HIT_DTYPE = np.dtype([("t", "<f8"), ("p", "<f8", 3), ("n", "<f8", 3), ("uv", "<f8", 2), ("object", "<i4"), ("tri", "<i4")])
assert HIT_DTYPE.itemsize == C.sizeof(capi.rh_hit)


@dataclass
class Hits:
    """closestIntersection of a batch of rays: views of one buffer of rh_hit records (`records`), numpy arrays or CUDA
    tensors like the rays.  t [n] (+inf on a miss), p [n, 3], n [n, 3] (mesh normals interpolated, not renormalised),
    uv [n, 2], object [n] (scene index, -1 on a miss), tri [n] (index in the mesh's triangles, -1 for planes, spheres
    and misses)."""
    t: object
    p: object
    n: object
    uv: object
    object: object
    tri: object
    records: object


def _query_rays(origins, directions):
    """Checks a batch of rays and packs it as the library's [n, 6] (origin, direction) float64 array: numpy arrays (host
    path) or CUDA tensors on the current device (device path).  Returns (rays, on_device)."""
    if isinstance(origins, np.ndarray) and isinstance(directions, np.ndarray):
        on_device = False
    elif all(type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False) for x in (origins, directions)):
        import torch

        on_device = True
        if origins.device != directions.device or origins.device.index != torch.cuda.current_device():
            raise ValueError("origins and directions must be CUDA tensors on the current device")
    else:
        raise ValueError("origins and directions must both be numpy arrays or both CUDA torch tensors")
    for name, a in (("origins", origins), ("directions", directions)):
        if str(a.dtype) not in ("float64", "torch.float64"):
            raise ValueError(f"{name} must be float64, got {a.dtype}")
        if a.ndim != 2 or a.shape[1] != 3:
            raise ValueError(f"{name} must have shape [n, 3], got {tuple(a.shape)}")
    if origins.shape[0] != directions.shape[0]:
        raise ValueError(f"origins has {origins.shape[0]} rays, directions {directions.shape[0]}")
    if on_device:
        import torch

        rays = torch.cat((origins, directions), dim=1).contiguous()
        torch.cuda.current_stream().synchronize()  # the library runs on its own stream
        return rays, True
    rays = np.empty((origins.shape[0], 6), dtype=np.float64)
    rays[:, :3], rays[:, 3:] = origins, directions
    return rays, False


def _ptr(a):
    return a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data


def closestIntersection(scene, origins, directions, exact_boxes: bool = False) -> Hits:
    """RayHs.hs:67-71 for every ray (origins[i], directions[i]): the closest hit over the scene's object list, as the
    reference computes it.  numpy arrays in, numpy arrays out; CUDA tensors in, CUDA tensors out (no host copy).
    `exact_boxes`: the reference's double slab test at every box (validation; same records)."""
    rays, on_device = _query_rays(origins, directions)
    n = rays.shape[0]
    flags = (capi.RH_FLAG_DEVICE_OUT if on_device else 0) | (capi.RH_FLAG_EXACT_BOXES if exact_boxes else 0)
    if on_device:
        import torch

        rec = torch.empty((n, HIT_DTYPE.itemsize), dtype=torch.uint8, device=rays.device)
        check(lib().rh_closest_intersection(scene.device, rays.data_ptr(), n, rec.data_ptr(), flags))
        f, i = rec.view(torch.float64), rec.view(torch.int32)
        return Hits(f[:, 0], f[:, 1:4], f[:, 4:7], f[:, 7:9], i[:, 18], i[:, 19], rec)
    rec = np.empty(n, dtype=HIT_DTYPE)
    check(lib().rh_closest_intersection(scene.device, rays.ctypes.data, n, rec.ctypes.data, flags))
    return Hits(rec["t"], rec["p"], rec["n"], rec["uv"], rec["object"], rec["tri"], rec)


def shadowIntersection(scene, light: int, origins, directions, exact_boxes: bool = False):
    """RayHs.hs:74-87 for every ray towards light `light` (index into the scene's lights): True where a non-emitter
    object has a hit in front of the light.  The caller builds the rays, as accumDiffuse does with `rayEps p ld`.
    Returns a bool numpy array or CUDA tensor, like the rays."""
    rays, on_device = _query_rays(origins, directions)
    n = rays.shape[0]
    flags = (capi.RH_FLAG_DEVICE_OUT if on_device else 0) | (capi.RH_FLAG_EXACT_BOXES if exact_boxes else 0)
    if on_device:
        import torch

        out = torch.empty(n, dtype=torch.uint8, device=rays.device)
    else:
        out = np.empty(n, dtype=np.uint8)
    check(lib().rh_shadow_intersection(scene.device, int(light), _ptr(rays), n, _ptr(out), flags))
    return out.view(torch.bool) if on_device else out.view(np.bool_)


# ---- radiance queries (RayHs.hs:149-154 traceRay)

@dataclass
class Radiance:
    """traceRay of a batch of rays: colors [n, 3] float64 (linear, not clamped, no toIntC), hit_ids [n, 2] int32
    (object, tri) of each ray's closest hit when asked for, numpy arrays or CUDA tensors like the rays, and the call's
    rh_stats as Image carries them."""
    colors: object
    stats: dict = field(default_factory=dict)
    hit_ids: object = None


def traceRay(scene, origins, directions, max_depth: int, *, want_hit_ids: bool = False, exact_boxes: bool = False,
             shadow: str | None = None, light_maps: bool = True, chunk_rays: int = 0) -> Radiance:
    """RayHs.hs:149-154 `traceRay sc 0 max_depth` for every ray (origins[i], directions[i]): the full Whitted radiance
    (shadows, reflection, refraction, textures), as the render computes it for a camera ray.  A ray that starts at depth
    d of a tree limited to maxD is traced with max_depth = maxD - d.  numpy arrays in, numpy arrays out; CUDA tensors
    in, CUDA tensors out.  `shadow` ('pooled' / 'split'), `exact_boxes` and `light_maps` as for render (same colours);
    `chunk_rays`: rays per wavefront chunk (0: the library's choice)."""
    rays, on_device = _query_rays(origins, directions)
    if not 0 <= int(chunk_rays) < 1 << 32:
        raise ValueError(f"chunk_rays must be in 0 .. 2^32 - 1, got {chunk_rays}")
    n = rays.shape[0]
    o = capi.rh_trace_opts()
    o.max_depth, o.chunk_rays = int(max_depth), int(chunk_rays)
    o.flags = ((capi.RH_FLAG_DEVICE_OUT if on_device else 0) | (capi.RH_FLAG_HIT_IDS if want_hit_ids else 0)
               | (capi.RH_FLAG_EXACT_BOXES if exact_boxes else 0) | _shadow_flag(shadow) | (0 if light_maps else capi.RH_FLAG_NO_LIGHT_MAPS))
    if on_device:
        import torch

        colors = torch.empty((n, 3), dtype=torch.float64, device=rays.device)
        ids = torch.empty((n, 2), dtype=torch.int32, device=rays.device) if want_hit_ids else None
    else:
        colors = np.empty((n, 3), dtype=np.float64)
        ids = np.empty((n, 2), dtype=np.int32) if want_hit_ids else None
    st = capi.rh_stats()
    check(lib().rh_trace_rays(scene.device, _ptr(rays), n, C.byref(o), _ptr(colors), _ptr(ids) if ids is not None else None,
                              C.byref(st)))
    return Radiance(colors, st.as_dict(), ids)


def scene_setup_ms(scene: Scene) -> dict:
    """Milliseconds rh_scene_create spent on its parts (host-side trees, light-space tables, uploads)."""
    ms, info = scene._info()
    return {"trees": ms[0], "light_tables": ms[1], "upload": ms[2], "deep_stack_entries_per_thread": info[3], "max_tree_depth": info[2]}


def _shadow_flag(shadow: str | None) -> int:
    """Shadow-walk schedule: None = the library's per-scene choice, 'pooled' / 'split' (per-lane refill) = forced
    (same image)."""
    if shadow is None:
        return 0
    return {"pooled": capi.RH_FLAG_SHADOW_POOLED, "split": capi.RH_FLAG_SHADOW_SPLIT}[shadow]


def render_device(job: Rendering, rgb_dev, spp: int = 1, offsets_dev=None, offset_tile: int = 0, shard_index: int = 0,
                  shard_count: int = 1, band_height: int = 0, chunk_samples: int = 0, count: bool = False,
                  profile: bool = False, shadow: str | None = None, seed: int | None = None, peer_frames=None,
                  light_maps: bool = True, shard_offsets: bool = False, hit_ids_dev=None) -> dict:
    """rh_render into a DEVICE framebuffer (torch CUDA uint8 tensor [rows, width, 3]).  `offsets_dev` is the
    full-frame [height*width, spp, 2] float64/float32 stream (or the [tile*tile, spp, 2] tile), either a CUDA
    tensor (already uploaded) or a pinned CPU tensor (uploaded chunk by chunk inside the call); with `shard_offsets`
    it holds only this shard's rows, shard-compact ([rows*width, spp, 2]).  `hit_ids_dev`: CUDA int32 tensor
    [rows*width*spp, 2] for the primary hit ids.  The call returns after the frame is complete."""
    import torch

    L = lib()
    mode, off = _offset_mode(offsets_dev, offset_tile)
    bh = band_height or L.rh_default_band_height(job.height, shard_count)
    rows = L.rh_shard_rows(job.height, shard_count, bh)
    if peer_frames is None and (tuple(rgb_dev.shape) != (rows, job.width, 3) or rgb_dev.dtype != torch.uint8 or not rgb_dev.is_cuda):
        raise ValueError("rgb_dev must be a CUDA uint8 tensor of shape [rows, width, 3]")
    flags = (capi.RH_FLAG_DEVICE_OUT | (capi.RH_FLAG_COUNT if count else 0) | (capi.RH_FLAG_PROFILE if profile else 0)
             | _shadow_flag(shadow) | (0 if light_maps else capi.RH_FLAG_NO_LIGHT_MAPS)
             | (capi.RH_FLAG_SHARD_OFFSETS if shard_offsets else 0) | (capi.RH_FLAG_HIT_IDS if hit_ids_dev is not None else 0))
    if off is not None and off.is_cuda:
        flags |= capi.RH_FLAG_DEVICE_OFFSETS
        torch.cuda.current_stream().synchronize()
    off_ptr = off.data_ptr() if off is not None else None
    seed_box = None
    if seed is not None:  # the kernel regenerates sample_offsets(width*height, spp, seed) on the device
        seed_box = C.c_uint64(seed)
        mode, off_ptr = capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed_box)
    ptrs = None
    if peer_frames is not None:  # fused exchange: rows go straight into every shard's full frame (PeerFrames.pointers)
        flags |= capi.RH_FLAG_PEER_FRAMES
        ptrs = (C.c_void_p * len(peer_frames))(*peer_frames)
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, chunk_samples, flags)
    if ptrs is not None:
        o.n_peer_frames, o.peer_frames = len(peer_frames), ptrs
    st = capi.rh_stats()
    check(L.rh_render(job.scene.device, C.byref(job.camera), C.byref(o), rgb_dev.data_ptr() if rgb_dev is not None else None,
                      hit_ids_dev.data_ptr() if hit_ids_dev is not None else None, C.byref(st)))
    return st.as_dict()


def render_multi(job: Rendering, n_gpus: int, spp: int = 1, offsets=None, seed: int | None = None, band_height: int = 0,
                 shadow: str | None = None) -> Image:
    """rh_multi_render: the whole frame on `n_gpus` GPUs of this process (one host thread per GPU, row bands interleaved,
    finished rows stored into one frame on GPU 0 over NVLink) — what a single-process host such as the Haskell
    front end calls.  The multi context and the replicated scene are created on first use."""
    L = lib()
    if L.rh_multi_gpu_count() == 0:
        check(L.rh_multi_init(int(n_gpus)))
    elif L.rh_multi_gpu_count() != n_gpus:
        raise ValueError(f"multi context already open on {L.rh_multi_gpu_count()} GPUs")
    sc = job.scene
    if getattr(sc, "_multi", None) is None:
        sc._multi = C.c_void_p()
        check(L.rh_multi_scene_create(sc.flat, C.byref(sc._multi)))
    mode, off = _offset_mode(offsets, 0)
    off_ptr = None
    seed_box = None
    if seed is not None:
        seed_box = C.c_uint64(seed)
        mode, off_ptr = capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed_box)
    elif off is not None:
        off_ptr = off.data_ptr() if hasattr(off, "data_ptr") else off.ctypes.data
    o = _opts(job, spp, mode, off_ptr, 0, 0, 1, band_height, 0, _shadow_flag(shadow))
    rgb = np.empty((job.height, job.width, 3), dtype=np.uint8)
    st = capi.rh_stats()
    check(L.rh_multi_render(sc._multi, C.byref(job.camera), C.byref(o), rgb.ctypes.data, C.byref(st)))
    return Image(job.width, job.height, rgb, st.as_dict(), None)


def multi_shutdown(scenes=()) -> None:
    L = lib()
    for sc in scenes:
        if getattr(sc, "_multi", None):
            L.rh_multi_scene_destroy(sc._multi)
            sc._multi = None
    L.rh_multi_shutdown()


class PeerFrames:
    """One full [height, width, 3] RGB8 frame per process of a torch.distributed job (one process per GPU), each mapped
    into every other process through CUDA IPC (rh_peer_alloc / rh_peer_open), so that rh_render's resolve kernel can
    store finished rows straight into all of them over NVLink (RH_FLAG_PEER_FRAMES) — the fused form of the
    all-gather + de-interleave exchange of SURVEY 8e.  `pointers` is ordered by rank; `frame` is this rank's own frame
    as a torch tensor.  After every rank's render call has returned, one barrier makes all frames complete."""

    def __init__(self, height: int, width: int):
        import torch
        import torch.distributed as dist

        L = lib()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self._own = C.c_void_p()
        handle = C.create_string_buffer(64)
        check(L.rh_peer_alloc(height * width * 3, C.byref(self._own), handle))
        handles = [None] * self.world
        dist.all_gather_object(handles, handle.raw)
        self._opened = {}
        self.pointers = []
        for r, h in enumerate(handles):
            if r == self.rank:
                self.pointers.append(self._own.value)
            else:
                p = C.c_void_p()
                check(L.rh_peer_open(h, C.byref(p)))
                self._opened[r] = p
                self.pointers.append(p.value)

        class _Cai:
            __cuda_array_interface__ = {"shape": (height, width, 3), "typestr": "|u1", "data": (self._own.value, False), "version": 3}

        self.frame = torch.as_tensor(_Cai(), device="cuda")

    def close(self):
        import torch.distributed as dist

        L = lib()
        self.frame = None
        for p in self._opened.values():
            L.rh_peer_close(p)
        self._opened = {}
        dist.barrier()  # nobody frees while a peer still has the allocation mapped
        if self._own:
            L.rh_peer_free(self._own)
            self._own = C.c_void_p()


def shard_global_rows(height: int, shard_index: int, shard_count: int, band_height: int) -> list[int]:
    """Image rows of one shard, in shard-compact order (SURVEY 8e): band b = row // band_height belongs to
    shard b % shard_count.  Padding rows of the last band are reported as -1."""
    rows = lib().rh_shard_rows(height, shard_count, band_height)
    out = []
    for lr in range(rows):
        g = ((lr // band_height) * shard_count + shard_index) * band_height + lr % band_height
        out.append(g if g < height else -1)
    return out


def assemble_bands(parts: list[np.ndarray], height: int, band_height: int) -> np.ndarray:
    """Host re-assembly of shard-compact band buffers (SURVEY 8e); the device path is rh_deinterleave_bands."""
    G = len(parts)
    width = parts[0].shape[1]
    out = np.empty((height, width, 3), dtype=np.uint8)
    for row in range(height):
        band, rib = divmod(row, band_height)
        out[row] = parts[band % G][(band // G) * band_height + rib]
    return out


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist
    except ImportError:
        pass
    return None


def _trace(job: Rendering, spp: int, offsets, offset_tile: int, **kw) -> Image:
    dist = _dist()
    if dist is None:
        return render(job, spp=spp, offsets=offsets, offset_tile=offset_tile, **kw)
    # one process per GPU: each rank renders its interleaved row bands, then one NCCL all-gather
    import torch

    L = lib()
    G, rank = dist.get_world_size(), dist.get_rank()
    bh = kw.pop("band_height", 0) or L.rh_default_band_height(job.height, G)
    rows = L.rh_shard_rows(job.height, G, bh)
    img = render(job, spp=spp, offsets=offsets, offset_tile=offset_tile, shard_index=rank, shard_count=G, band_height=bh, **kw)
    if dist.get_backend() == "nccl":
        mine = torch.from_numpy(img.pixels).cuda()
        gathered = torch.empty((G, rows, job.width, 3), dtype=torch.uint8, device=mine.device)
        dist.all_gather_into_tensor(gathered, mine)
        full = torch.empty((job.height, job.width, 3), dtype=torch.uint8, device=mine.device)
        torch.cuda.current_stream().synchronize()
        check(L.rh_deinterleave_bands(gathered.data_ptr(), full.data_ptr(), job.width, job.height, G, bh))
        pixels = full.cpu().numpy()
    else:  # gloo (CPU tests of the shard logic)
        mine = torch.from_numpy(img.pixels)
        parts = [torch.empty_like(mine) for _ in range(G)]
        dist.all_gather(parts, mine)
        pixels = assemble_bands([p.numpy() for p in parts], job.height, bh)
    return Image(job.width, job.height, pixels, img.stats, None)


def rayTrace(job: Rendering, **kw) -> Image:
    """RayHs.hs:161-166: one sample per pixel at the integer pixel coordinate (Image.hs:31-36)."""
    return _trace(job, 1, None, 0, **kw)


def distributedRayTrace(job: Rendering, spp: int = 64, seed: int = 24, offsets=None, offset_tile: int = 0, **kw) -> Image:
    """RayHs.hs:190-195 with the reference's hard-coded 64 samples (RayHs.hs:175) as the default."""
    if offsets is None:
        n = offset_tile * offset_tile if offset_tile else job.width * job.height
        offsets = sample_offsets(n, spp, seed)
    return _trace(job, spp, offsets, offset_tile, **kw)


def writePPM(path: str, image: Image) -> None:
    """Image.hs:70-75 — byte-identical P3 text."""
    px = np.ascontiguousarray(image.pixels, dtype=np.uint8)
    check(lib().rh_write_ppm(path.encode(), px.ctypes.data, image.width, image.height))


def main(argv: list[str] | None = None) -> int:
    """`rayhs [-oFILE | --output=FILE] scene.json` (RayHs.hs:204-234; getOpt RequireOrder, default out.ppm)."""
    import sys

    args = list(sys.argv[1:] if argv is None else argv)
    out_file = "out.ppm"
    while args and args[0].startswith("-") and args[0] != "-":
        a = args.pop(0)
        if a.startswith("--output"):
            out_file = a.split("=", 1)[1] if "=" in a else "out.ppm"
        elif a.startswith("-o"):
            out_file = a[2:] or "out.ppm"
        else:
            sys.stderr.write(f"unrecognized option `{a}'\nUsage: ray [OPTION...] files...\n")
            return 1
    if not args:
        sys.stderr.write("Please specify scene file\n")
        return 1
    scene_file = args[0]
    print(f"Reading scene {scene_file}")
    job = buildRendering(scene_file)
    print("Rendering...")
    image = rayTrace(job)
    writePPM(out_file, image)
    print(f"Writing output to {out_file}")
    return 0
