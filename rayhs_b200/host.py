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
        self._tables = None  # (materials, lights) ctypes arrays after update(): what raw and flat describe from then on
        self._raw_view = self._flat_view = None

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
        """POINTER(rh_raw_scene): the scene before any tree build (what the oracle is fed), with the tables of the last
        update()."""
        r = lib().rh_loaded_raw(self._loaded)
        if self._tables is None:
            return r
        self._raw_view = self._patched(capi.rh_raw_scene, r)
        return C.pointer(self._raw_view)

    @property
    def flat(self):
        """POINTER(rh_scene_desc): KDTree.hs:68-90 build + flattening, on the host, with the tables of the last update()."""
        if not self._flat:
            check(lib().rh_flatten(self.raw, C.byref(self._flat)))
        d = lib().rh_flat_desc(self._flat)
        if self._tables is None:
            return d
        self._flat_view = self._patched(capi.rh_scene_desc, d)
        return C.pointer(self._flat_view)

    def _patched(self, struct, ptr):
        """A copy of the library's description whose material and light tables are this Scene's (kept alive by it)."""
        mats, lights = self._tables
        c = struct.from_buffer_copy(ptr.contents)
        c.materials = C.cast(mats, C.POINTER(capi.rh_material))
        c.lights = C.cast(lights, C.POINTER(capi.rh_light)) if len(lights) else None
        c.n_lights = len(lights)
        return c

    @property
    def materials(self):
        """A copy of the current material table (ctypes array of rh_material)."""
        r = self.raw.contents
        return (capi.rh_material * r.n_materials).from_buffer_copy(
            C.string_at(r.materials, r.n_materials * C.sizeof(capi.rh_material)) if r.n_materials else b"")

    @property
    def lights(self):
        """A copy of the current light table (ctypes array of rh_light)."""
        r = self.raw.contents
        return (capi.rh_light * r.n_lights).from_buffer_copy(
            C.string_at(r.lights, r.n_lights * C.sizeof(capi.rh_light)) if r.n_lights else b"")

    def update(self, materials=None, lights=None) -> dict:
        """rh_scene_update: replaces the material table (same length) and / or the light table (any length; None keeps
        a table) of the device copy, of the multi-GPU replica render_multi made, and of raw / flat.  Before the device
        copy exists only the description changes.  Returns the library's rh_update_info as a dict."""
        def table(kind, rows):
            if isinstance(rows, C.Array) and rows._type_ is kind:
                return (kind * len(rows)).from_buffer_copy(rows)
            rows = list(rows)
            if not all(isinstance(x, kind) for x in rows):
                raise TypeError(f"expected {kind.__name__} entries")
            return (kind * len(rows))(*rows)

        cur_m, cur_l = self.materials, self.lights
        mats = cur_m if materials is None else table(capi.rh_material, materials)
        lts = cur_l if lights is None else table(capi.rh_light, lights)
        if len(mats) != len(cur_m):
            raise ValueError(f"{len(mats)} materials for a scene with {len(cur_m)}: objects keep their material indices")
        info = capi.rh_update_info()
        args = (None if materials is None else mats, len(mats), None if lights is None else (lts if len(lts) else (capi.rh_light * 1)()),
                len(lts))
        L = lib()
        if self._dev:
            check(L.rh_scene_update(self._dev, *args, C.byref(info)))
        if getattr(self, "_multi", None):
            check(L.rh_multi_scene_update(self._multi, *args, None if self._dev else C.byref(info)))
        self._tables = (mats, lts)
        return {n: int(getattr(info, n)) for n, _ in info._fields_}

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


def thinLens(camera: capi.rh_camera, aperture: float, focus_distance: float) -> capi.rh_camera:
    """A copy of `camera` as a thin-lens camera (RH_PROJ_THIN_LENS: depth of field): the same position, target, up and
    fovy, a circular lens of radius `aperture` (world units; 0 casts the perspective rays) and the plane at
    `focus_distance` along the view axis in focus.  Every render entry point takes it; see rh_camera in
    include/rayhs_b200.h for the rays."""
    c = capi.rh_camera.from_buffer_copy(camera)
    c.projection = capi.RH_PROJ_THIN_LENS
    c.proj_width, c.proj_height = float(aperture), float(focus_distance)
    return c


def sphereLight(position, color, radius: float) -> capi.rh_light:
    """A sphere light (RH_LIGHT_SPHERE: soft shadows): a point light at `position` whose falloff radius `radius` (finite,
    >= 0) is also the radius of the ball it emits from; each shaded point samples one point of the ball (see rh_light in
    include/rayhs_b200.h).  For Scene.update's light table, or to turn a scene's point lights into sphere lights."""
    L = capi.rh_light()
    L.kind = capi.RH_LIGHT_SPHERE
    L.vec[:] = [float(x) for x in position]
    L.color[:] = [float(x) for x in color]
    L.radius = float(radius)
    return L


@dataclass
class Image:
    """Image.hs:21-23, already quantised by toIntC (Image.hs:54-55): uint8 [height, width, 3].  `linear` (progressive
    calls that ask for it): float64 [height, width, 3], the averaged colour toIntC is applied to."""
    width: int
    height: int
    pixels: np.ndarray
    stats: dict = field(default_factory=dict)
    hit_ids: np.ndarray | None = None
    linear: np.ndarray | None = None


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


def _ptr(a):
    return a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data


def _offsets(job: Rendering, spp: int, offsets, seed: int | None, tile: int, shard_rows: int | None = None):
    """The sample source of one call: `offsets` (float64 / float32 values of the full frame, [width*height, spp, 2]; of
    a tile, [tile*tile, spp, 2]; or with `shard_rows` of this shard's rows only, [shard_rows*width, spp, 2]: numpy, a
    CPU tensor or a CUDA tensor), `seed` (the SplitMix64 stream the library regenerates) or neither (pixel centres).
    Returns (mode, pointer, keep, on_device): `keep` holds what the pointer refers to (the seed, or the dense copy of a
    strided view, which the library could not read) and must outlive the call; `on_device`: the offsets are CUDA."""
    if seed is not None:
        if offsets is not None:
            raise ValueError("pass either offsets or seed")
        box = C.c_uint64(seed)
        return capi.RH_OFFSETS_SPLITMIX64, C.addressof(box), box, False
    if offsets is None:
        return capi.RH_OFFSETS_NONE, None, None, False
    need = (tile * tile if tile else (job.height if shard_rows is None else shard_rows) * job.width) * spp * 2
    have = offsets.numel() if hasattr(offsets, "numel") else offsets.size
    if have != need:
        raise ValueError(f"offsets has {have} values, expected {need}")
    mode = (capi.RH_OFFSETS_TILED_F64 if tile else capi.RH_OFFSETS_F32 if str(offsets.dtype).endswith("float32")
            else capi.RH_OFFSETS_F64)
    off = offsets.contiguous() if hasattr(offsets, "contiguous") else np.ascontiguousarray(offsets)
    return mode, _ptr(off), off, bool(getattr(off, "is_cuda", False))


def _flags(*, want_hit_ids: bool = False, device: bool = False, count: bool = False, profile: bool = False,
           exact_boxes: bool = False, shadow: str | None = None, light_maps: bool = True) -> int:
    """RH_FLAG_* bits of the keyword arguments the entry points share.  `shadow`, the shadow-walk schedule: None = the
    library's per-scene choice, 'pooled' / 'split' (per-lane refill) = forced (same image)."""
    return ((capi.RH_FLAG_HIT_IDS if want_hit_ids else 0) | (capi.RH_FLAG_DEVICE_OUT if device else 0)
            | (capi.RH_FLAG_COUNT if count else 0) | (capi.RH_FLAG_PROFILE if profile else 0)
            | (capi.RH_FLAG_EXACT_BOXES if exact_boxes else 0) | (0 if light_maps else capi.RH_FLAG_NO_LIGHT_MAPS)
            | (0 if shadow is None else {"pooled": capi.RH_FLAG_SHADOW_POOLED, "split": capi.RH_FLAG_SHADOW_SPLIT}[shadow]))


def _shard_rows(job: Rendering, shard_count: int, band_height: int):
    """(band height, rows of one shard): `band_height` 0 is the library's choice."""
    L = lib()
    bh = band_height or L.rh_default_band_height(job.height, shard_count)
    return bh, L.rh_shard_rows(job.height, shard_count, bh)


def _alloc(device: bool):
    """empty(shape, dtype name) for a call's outputs: numpy arrays, or CUDA tensors with `device`.  On the device the
    current torch stream is synchronised first, since the library runs on its own stream."""
    if not device:
        return lambda shape, dtype: np.empty(shape, dtype=dtype)
    import torch

    torch.cuda.current_stream().synchronize()
    return lambda shape, dtype: torch.empty(shape, dtype=getattr(torch, dtype), device="cuda")


def render(job: Rendering, spp: int = 1, offsets=None, offset_tile: int = 0, want_hit_ids: bool = False,
           shard_index: int = 0, shard_count: int = 1, band_height: int = 0, chunk_samples: int = 0,
           count: bool = False, profile: bool = False, exact_boxes: bool = False, out: np.ndarray | None = None,
           shadow: str | None = None, seed: int | None = None, light_maps: bool = True) -> Image:
    """One rh_render call with HOST buffers (numpy or pinned torch CPU tensors for `offsets`).
    `seed` (instead of `offsets`): the kernel regenerates sample_offsets(width*height, spp, seed) on the device.
    Returns the shard-compact RGB8 rows when shard_count > 1."""
    mode, off_ptr, keep, on_device = _offsets(job, spp, offsets, seed, offset_tile)
    if on_device:
        raise ValueError("CUDA offsets go to render_device; render takes host offsets")
    bh, rows = _shard_rows(job, shard_count, band_height)
    flags = _flags(want_hit_ids=want_hit_ids, count=count, profile=profile, exact_boxes=exact_boxes, shadow=shadow,
                   light_maps=light_maps)
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, chunk_samples, flags)
    rgb = out if out is not None else np.empty((rows, job.width, 3), dtype=np.uint8)
    ids = np.empty((rows, job.width, spp, 2), dtype=np.int32) if want_hit_ids else None
    st = capi.rh_stats()
    check(lib().rh_render(job.scene.device, C.byref(job.camera), C.byref(o), rgb.ctypes.data,
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
    path) or CUDA tensors on the current device (device path; _alloc(True) synchronises the packing).  Returns (rays,
    on_device)."""
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

        return torch.cat((origins, directions), dim=1).contiguous(), True
    rays = np.empty((origins.shape[0], 6), dtype=np.float64)
    rays[:, :3], rays[:, 3:] = origins, directions
    return rays, False


def closestIntersection(scene, origins, directions, exact_boxes: bool = False) -> Hits:
    """RayHs.hs:67-71 for every ray (origins[i], directions[i]): the closest hit over the scene's object list, as the
    reference computes it.  numpy arrays in, numpy arrays out; CUDA tensors in, CUDA tensors out (no host copy).
    `exact_boxes`: the reference's double slab test at every box (validation; same records)."""
    rays, on_device = _query_rays(origins, directions)
    n = rays.shape[0]
    rec = _alloc(on_device)((n, HIT_DTYPE.itemsize), "uint8")
    check(lib().rh_closest_intersection(scene.device, _ptr(rays), n, _ptr(rec), _flags(device=on_device, exact_boxes=exact_boxes)))
    if on_device:
        import torch

        f, i = rec.view(torch.float64), rec.view(torch.int32)
        return Hits(f[:, 0], f[:, 1:4], f[:, 4:7], f[:, 7:9], i[:, 18], i[:, 19], rec)
    rec = rec.view(HIT_DTYPE).reshape(n)
    return Hits(rec["t"], rec["p"], rec["n"], rec["uv"], rec["object"], rec["tri"], rec)


def shadowIntersection(scene, light: int, origins, directions, exact_boxes: bool = False):
    """RayHs.hs:74-87 for every ray towards light `light` (index into the scene's lights): True where a non-emitter
    object has a hit in front of the light.  The caller builds the rays, as accumDiffuse does with `rayEps p ld`.
    Returns a bool numpy array or CUDA tensor, like the rays."""
    rays, on_device = _query_rays(origins, directions)
    n = rays.shape[0]
    out = _alloc(on_device)(n, "uint8")
    check(lib().rh_shadow_intersection(scene.device, int(light), _ptr(rays), n, _ptr(out), _flags(device=on_device, exact_boxes=exact_boxes)))
    if on_device:
        import torch

        return out.view(torch.bool)
    return out.view(np.bool_)


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
    o.flags = _flags(device=on_device, want_hit_ids=want_hit_ids, exact_boxes=exact_boxes, shadow=shadow, light_maps=light_maps)
    empty = _alloc(on_device)
    colors = empty((n, 3), "float64")
    ids = empty((n, 2), "int32") if want_hit_ids else None
    st = capi.rh_stats()
    check(lib().rh_trace_rays(scene.device, _ptr(rays), n, C.byref(o), _ptr(colors), _ptr(ids) if ids is not None else None,
                              C.byref(st)))
    return Radiance(colors, st.as_dict(), ids)


# ---- feature buffers (first hits of the camera rays, for denoisers and compositing)

@dataclass
class Features:
    """rh_render_features of one view: per pixel of the (shard-compact) rows, the mean over its samples of the albedo
    albedo [rows, w, 3] and of the normal normal [rows, w, 3] of each camera ray's closest hit (0 for a miss; normals are
    not renormalised), the mean t of the hitting samples depth [rows, w] (+inf without one), the number of hitting samples
    hits [rows, w] (uint32; int32 on the device), the hit ids [rows, w, spp, 2] when asked for, and the call's stats.
    numpy arrays, or CUDA tensors with device=True."""
    albedo: object
    normal: object
    depth: object
    hits: object
    hit_ids: object = None
    stats: dict = field(default_factory=dict)


def renderFeatures(job: Rendering, spp: int = 1, offsets=None, seed: int | None = None, offset_tile: int = 0, stream_spp: int = 0,
                   stream_base: int = 0, want_hit_ids: bool = False, shard_index: int = 0, shard_count: int = 1,
                   band_height: int = 0, exact_boxes: bool = False, device: bool = False) -> Features:
    """Feature buffers of the camera rays render(job, spp, offsets / seed, ...) casts.  `offsets`: full-frame
    [width*height, spp, 2] float64 / float32 (or the [tile*tile, spp, 2] tile with `offset_tile`), numpy, a CPU tensor
    or, with device=True, a CUDA tensor (a strided view is copied to a dense array first); `seed`: the SplitMix64 stream
    instead, samples stream_base .. stream_base + spp - 1 of a stream of `stream_spp` samples per pixel (0: spp), as an
    Accumulator holding stream_base samples draws them.  `device`: outputs are CUDA tensors."""
    if seed is None and (stream_spp or stream_base):
        raise ValueError("stream_spp and stream_base go with seed")
    mode, off_ptr, keep, dev_off = _offsets(job, spp, offsets, seed, offset_tile)
    if dev_off and not device:
        raise ValueError("CUDA offsets need device=True")
    flags = _flags(want_hit_ids=want_hit_ids, exact_boxes=exact_boxes, device=device) | (capi.RH_FLAG_DEVICE_OFFSETS if dev_off else 0)
    bh, rows = _shard_rows(job, shard_count, band_height)
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, 0, flags)
    shape = (rows, job.width)
    empty = _alloc(device)
    hits_dtype = "int32" if device else "uint32"  # (torch has no uint32 arithmetic to speak of)
    fe = Features(empty(shape + (3,), "float64"), empty(shape + (3,), "float64"), empty(shape, "float64"), empty(shape, hits_dtype),
                  empty(shape + (spp, 2), "int32") if want_hit_ids else None)
    ft = capi.rh_features()
    ft.albedo, ft.normal, ft.depth, ft.hits = (_ptr(a) for a in (fe.albedo, fe.normal, fe.depth, fe.hits))
    ft.stream_spp, ft.stream_base = int(stream_spp), int(stream_base)
    st = capi.rh_stats()
    check(lib().rh_render_features(job.scene.device, C.byref(job.camera), C.byref(o), C.byref(ft),
                                   _ptr(fe.hit_ids) if want_hit_ids else None, C.byref(st)))
    fe.stats = st.as_dict()
    return fe


# ---- light groups (one linear image per group of lights, for relighting in compositing)

@dataclass
class LightGroups:
    """rh_render_light_groups of one view: groups [G, rows, w, 3] float64, the linear image of each group of lights;
    rest [rows, w, 3], what no light adds (Diffuse's ambient term, Emmit, ShowNormal, ShowUV); image, the render's RGB8
    rows (None unless asked for); hit_ids [rows, w, spp, 2] when asked for; and the call's stats.  numpy arrays, or CUDA
    tensors for a call with device outputs."""
    groups: object
    rest: object
    image: object = None
    hit_ids: object = None
    stats: dict = field(default_factory=dict)

    def relight(self, scales):
        """sum over g of scales[g] * groups[g] (per channel, in group order), plus rest: the image with the colours of
        group g's lights multiplied by scales[g], up to rounding.  scales: [G, 3]."""
        on_device = getattr(self.groups, "is_cuda", False)
        if on_device:
            import torch

            s = torch.as_tensor(scales, dtype=torch.float64).to(self.groups.device)
        else:
            s = np.asarray(scales, dtype=np.float64)
        G = self.groups.shape[0]
        if tuple(s.shape) != (G, 3):
            raise ValueError(f"scales must have shape [{G}, 3], got {tuple(s.shape)}")
        out = s[0] * self.groups[0]
        for g in range(1, G):
            out = out + s[g] * self.groups[g]
        return out + self.rest


def renderLightGroups(job: Rendering, spp: int = 1, offsets=None, seed: int | None = None, groups=None, rgb: bool = True,
                      want_hit_ids: bool = False, shadow: str | None = None, exact_boxes: bool = False, light_maps: bool = True,
                      chunk_samples: int = 0, shard_index: int = 0, shard_count: int = 1, band_height: int = 0,
                      device: bool = False, profile: bool = False) -> LightGroups:
    """The light groups of the frame render(job, spp, offsets / seed, ...) renders.  `groups`: the group of each of the
    scene's lights (a sequence of ints, G = largest + 1 <= 16); None: one group per light.  `offsets`: full-frame
    [width*height, spp, 2] float64 / float32, numpy, a CPU tensor or a CUDA tensor; `seed`: the SplitMix64 stream
    instead.  CUDA offsets or device=True: the outputs are CUDA tensors.  `rgb`: also return the render's RGB8 rows."""
    n_lights = job.scene.raw.contents.n_lights
    if groups is None:
        groups = list(range(n_lights))
    groups = [int(g) for g in groups]
    if len(groups) != n_lights:
        raise ValueError(f"groups has {len(groups)} entries for a scene with {n_lights} lights")
    if any(not 0 <= g < 16 for g in groups):
        raise ValueError("group indices must be in 0 .. 15")
    G = max(groups, default=0) + 1
    mode, off_ptr, keep, dev_off = _offsets(job, spp, offsets, seed, 0)
    device = device or dev_off
    flags = (_flags(want_hit_ids=want_hit_ids, exact_boxes=exact_boxes, shadow=shadow, light_maps=light_maps, profile=profile,
                    device=device) | (capi.RH_FLAG_DEVICE_OFFSETS if dev_off else 0))
    bh, rows = _shard_rows(job, shard_count, band_height)
    o = _opts(job, spp, mode, off_ptr, 0, shard_index, shard_count, bh, chunk_samples, flags)
    empty = _alloc(device)
    out = empty((G + 1, rows, job.width, 3), "float64")
    image = empty((rows, job.width, 3), "uint8") if rgb else None
    ids = empty((rows, job.width, spp, 2), "int32") if want_hit_ids else None
    map_ = (C.c_uint8 * max(n_lights, 1))(*groups)
    lg = capi.rh_light_groups()
    lg.group_of_light, lg.n_groups, lg.out = C.addressof(map_), G, _ptr(out)
    st = capi.rh_stats()
    check(lib().rh_render_light_groups(job.scene.device, C.byref(job.camera), C.byref(o), C.byref(lg),
                                       _ptr(image) if rgb else None, _ptr(ids) if want_hit_ids else None, C.byref(st)))
    return LightGroups(out[:G], out[G], image, ids, st.as_dict())


# ---- camera batches (many views of one scene in one wavefront)

@dataclass
class Views:
    """rh_render_views of a batch of cameras, view-major over the shard's rows: pixels [V, rows, w, 3] uint8 (None unless
    asked for), view v being render(camera v)'s RGB8 rows; linear [V, rows, w, 3] float64 (None unless asked for), the
    colours toIntC is applied to, as a fresh Accumulator's first add returns them; hit_ids [V, rows, w, spp, 2] when
    asked for; and the call's stats (ray counts summed over the views).  numpy arrays, or CUDA tensors with device
    outputs."""
    pixels: object = None
    linear: object = None
    hit_ids: object = None
    stats: dict = field(default_factory=dict)


def renderViews(job: Rendering, cameras, spp: int = 1, offsets=None, seed: int | None = None, seeds=None, rgb: bool = True,
                linear: bool = False, want_hit_ids: bool = False, device: bool = False, shard_index: int = 0, shard_count: int = 1,
                band_height: int = 0, chunk_samples: int = 0, exact_boxes: bool = False, shadow: str | None = None,
                light_maps: bool = True, offset_tile: int = 0, shard_offsets: bool = False, profile: bool = False) -> Views:
    """One wavefront for a batch of views of job's scene: view v is render(job with cameras[v], spp, offsets / seed,
    ...).  `cameras`: a sequence of capi.rh_camera (job.camera is not used; width, height and maxDepth are job's).
    `offsets`: full-frame [width*height, spp, 2] float64 / float32 (with `shard_offsets`, the shard's rows only; with
    `offset_tile`, the [tile*tile, spp, 2] tile), numpy, a CPU tensor or a CUDA tensor, the same for every view; `seed`:
    the SplitMix64 stream instead; `seeds`: one SplitMix64 seed per view.  CUDA offsets or device=True: the outputs are
    CUDA tensors.  `rgb` / `linear`: which of the two images to return (at least one)."""
    cams = list(cameras)
    V = len(cams)
    if not rgb and not linear:
        raise ValueError("ask for rgb, linear or both")
    if seeds is not None:
        seeds = [int(x) for x in seeds]
        if len(seeds) != V:
            raise ValueError(f"seeds has {len(seeds)} entries for {V} cameras")
        if offsets is not None:
            raise ValueError("pass either offsets or seeds")
        if seed is None:
            seed = seeds[0] if seeds else 0
    bh, rows = _shard_rows(job, shard_count, band_height)
    mode, off_ptr, keep, dev_off = _offsets(job, spp, offsets, seed, offset_tile, rows if shard_offsets else None)
    device = device or dev_off
    flags = (_flags(want_hit_ids=want_hit_ids, exact_boxes=exact_boxes, shadow=shadow, light_maps=light_maps, profile=profile,
                    device=device) | (capi.RH_FLAG_DEVICE_OFFSETS if dev_off else 0)
             | (capi.RH_FLAG_SHARD_OFFSETS if shard_offsets else 0))
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, chunk_samples, flags)
    empty = _alloc(device)
    shape = (V, rows, job.width)
    out = Views(empty(shape + (3,), "uint8") if rgb else None, empty(shape + (3,), "float64") if linear else None,
                empty(shape + (spp, 2), "int32") if want_hit_ids else None)
    table = (capi.rh_camera * max(V, 1))(*cams)
    seed_table = (C.c_uint64 * max(V, 1))(*seeds) if seeds is not None else None
    vw = capi.rh_views()
    vw.cameras, vw.n_views = C.cast(table, C.POINTER(capi.rh_camera)), V
    if seed_table is not None:
        vw.seeds = C.cast(seed_table, C.POINTER(C.c_uint64))
    st = capi.rh_stats()
    check(lib().rh_render_views(job.scene.device, C.byref(vw), C.byref(o), _ptr(out.pixels) if rgb else None,
                                _ptr(out.linear) if linear else None, _ptr(out.hit_ids) if want_hit_ids else None, C.byref(st)))
    out.stats = st.as_dict()
    return out


def scene_setup_ms(scene: Scene) -> dict:
    """Milliseconds rh_scene_create spent on its parts (host-side trees, light-space tables, uploads)."""
    ms, info = scene._info()
    return {"trees": ms[0], "light_tables": ms[1], "upload": ms[2], "deep_stack_entries_per_thread": info[3], "max_tree_depth": info[2]}


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

    bh, rows = _shard_rows(job, shard_count, band_height)
    if peer_frames is None and (tuple(rgb_dev.shape) != (rows, job.width, 3) or rgb_dev.dtype != torch.uint8 or not rgb_dev.is_cuda):
        raise ValueError("rgb_dev must be a CUDA uint8 tensor of shape [rows, width, 3]")
    mode, off_ptr, keep, dev_off = _offsets(job, spp, offsets_dev, seed, offset_tile, rows if shard_offsets else None)
    flags = (_flags(device=True, count=count, profile=profile, shadow=shadow, light_maps=light_maps, want_hit_ids=hit_ids_dev is not None)
             | (capi.RH_FLAG_SHARD_OFFSETS if shard_offsets else 0))
    if dev_off:
        flags |= capi.RH_FLAG_DEVICE_OFFSETS
        torch.cuda.current_stream().synchronize()
    ptrs = None
    if peer_frames is not None:  # fused exchange: rows go straight into every shard's full frame (PeerFrames.pointers)
        flags |= capi.RH_FLAG_PEER_FRAMES
        ptrs = (C.c_void_p * len(peer_frames))(*peer_frames)
    o = _opts(job, spp, mode, off_ptr, offset_tile, shard_index, shard_count, bh, chunk_samples, flags)
    if ptrs is not None:
        o.n_peer_frames, o.peer_frames = len(peer_frames), ptrs
    st = capi.rh_stats()
    check(lib().rh_render(job.scene.device, C.byref(job.camera), C.byref(o), rgb_dev.data_ptr() if rgb_dev is not None else None,
                          hit_ids_dev.data_ptr() if hit_ids_dev is not None else None, C.byref(st)))
    return st.as_dict()


def render_multi(job: Rendering, n_gpus: int, spp: int = 1, offsets=None, seed: int | None = None, band_height: int = 0,
                 shadow: str | None = None) -> Image:
    """rh_multi_render: the whole frame on `n_gpus` GPUs of this process (one host thread per GPU, row bands interleaved,
    finished rows stored into one frame on GPU 0 over NVLink) — what a single-process host such as the Haskell
    front end calls.  The multi context and the replicated scene are created on first use."""
    mode, off_ptr, keep, on_device = _offsets(job, spp, offsets, seed, 0)
    if on_device:
        raise ValueError("CUDA offsets go to render_device; render_multi takes host offsets")
    L = lib()
    if L.rh_multi_gpu_count() == 0:
        check(L.rh_multi_init(int(n_gpus)))
    elif L.rh_multi_gpu_count() != n_gpus:
        raise ValueError(f"multi context already open on {L.rh_multi_gpu_count()} GPUs")
    sc = job.scene
    if getattr(sc, "_multi", None) is None:
        sc._multi = C.c_void_p()
        check(L.rh_multi_scene_create(sc.flat, C.byref(sc._multi)))
    o = _opts(job, spp, mode, off_ptr, 0, 0, 1, band_height, 0, _flags(shadow=shadow))
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

    G, rank = dist.get_world_size(), dist.get_rank()
    bh, rows = _shard_rows(job, G, kw.pop("band_height", 0))
    img = render(job, spp=spp, offsets=offsets, offset_tile=offset_tile, shard_index=rank, shard_count=G, band_height=bh, **kw)
    if dist.get_backend() == "nccl":
        mine = torch.from_numpy(img.pixels).cuda()
        gathered = torch.empty((G, rows, job.width, 3), dtype=torch.uint8, device=mine.device)
        dist.all_gather_into_tensor(gathered, mine)
        full = torch.empty((job.height, job.width, 3), dtype=torch.uint8, device=mine.device)
        torch.cuda.current_stream().synchronize()
        check(lib().rh_deinterleave_bands(gathered.data_ptr(), full.data_ptr(), job.width, job.height, G, bh))
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


class _PixelState:
    """Per-pixel state of one view that the library keeps between calls: the shard geometry of its rows (as for render)
    and the handle `create` makes, released by close() through `destroy`."""
    _what = "state"  # (for the error of a call after close())

    def __init__(self, job: Rendering, stream_spp: int, shard_index: int, shard_count: int, band_height: int, device: bool,
                 create, destroy):
        init()
        self.job, self.device, self.stream_spp = job, bool(device), int(stream_spp)
        self.shard_index, self.shard_count = shard_index, shard_count
        self.band_height, self.rows = _shard_rows(job, shard_count, band_height)
        self._destroy, self._h = destroy, C.c_void_p()
        check(create(job.width, job.height, shard_index, shard_count, self.band_height, self.stream_spp, C.byref(self._h)))

    def _handle(self):
        if not self._h:
            raise ValueError(f"the {self._what} is closed")
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Accumulator(_PixelState):
    """Progressive rendering (rh_render_accumulate): running per-pixel sums of the sample colours of one view, kept on
    the device between calls, so that an image can be refined over several calls instead of rendered again.  Each
    add(spp) traces spp new samples per pixel exactly as render would, continues the sums in sample order and returns
    the image of all samples so far: K calls of s samples give the bytes of one render of K*s samples.

    `stream_spp`: samples per pixel of the SplitMix64 stream that add(seed=...) draws from (sample_offsets(n, stream_spp,
    seed) sliced into consecutive ranges); `shard_index` / `shard_count` / `band_height` as for render (the outputs are
    shard-compact).  `device`: outputs are CUDA tensors (and `offsets` may be one); else numpy arrays.  The first add()
    after creation or reset() fixes the scene, camera and max_depth of the job; reset() returns to 0 samples."""

    _what = "accumulator"

    def __init__(self, job: Rendering, stream_spp: int = 0, shard_index: int = 0, shard_count: int = 1, band_height: int = 0,
                 device: bool = False):
        L = lib()
        super().__init__(job, stream_spp, shard_index, shard_count, band_height, device, L.rh_accum_create, L.rh_accum_destroy)
        self._n = 0

    @property
    def samples(self) -> int:
        """Samples per pixel in the running sums."""
        return self._n

    def add(self, spp: int, offsets=None, seed: int | None = None, rgb: bool = True, linear: bool = True,
            want_hit_ids: bool = False, shadow: str | None = None, exact_boxes: bool = False, light_maps: bool = True,
            chunk_samples: int = 0, profile: bool = False) -> Image:
        """Traces `spp` new samples per pixel and returns the Image of all samples so far: `pixels` (RGB8, when `rgb`),
        `linear` (float64, when `linear`), `hit_ids` of this call's samples [rows, width, spp, 2] (`want_hit_ids`) and
        this call's stats.  `offsets`: this call's samples, full-frame [width*height, spp, 2] float64 / float32 (numpy, a
        CPU tensor or, with device=True, a CUDA tensor; a strided view such as stream[:, n:n + spp] is copied to a dense array
        first); `seed`: the next spp samples of the accumulator's SplitMix64
        stream instead; neither: one sample at the pixel coordinate per spp.  `profile`: time every launch on its own
        (stats ms_trace / ms_shadow / ms_resolve; slower)."""
        h = self._handle()
        job = self.job
        mode, off_ptr, keep, dev_off = _offsets(job, spp, offsets, seed, 0)
        if dev_off and not self.device:
            raise ValueError("CUDA offsets need an accumulator with device=True")
        flags = (_flags(want_hit_ids=want_hit_ids, exact_boxes=exact_boxes, shadow=shadow, light_maps=light_maps, device=self.device,
                        profile=profile) | (capi.RH_FLAG_DEVICE_OFFSETS if dev_off else 0))
        o = _opts(job, spp, mode, off_ptr, 0, self.shard_index, self.shard_count, self.band_height, chunk_samples, flags)
        empty = _alloc(self.device)
        px = empty((self.rows, job.width, 3), "uint8") if rgb else None
        lin = empty((self.rows, job.width, 3), "float64") if linear else None
        ids = empty((self.rows, job.width, spp, 2), "int32") if want_hit_ids else None
        st = capi.rh_stats()
        check(lib().rh_render_accumulate(job.scene.device, C.byref(job.camera), C.byref(o), h,
                                         *(_ptr(a) if a is not None else None for a in (px, lin, ids)), C.byref(st)))
        self._n += spp
        return Image(job.width, self.rows, px, st.as_dict(), ids, lin)

    def reset(self) -> None:
        """Back to 0 samples; the next add() may use another scene, camera or max_depth."""
        check(lib().rh_accum_reset(self._h))
        self._n = 0


def progressiveRayTrace(job: Rendering, spp: int = 64, batch: int = 8, seed: int = 24):
    """distributedRayTrace (RayHs.hs:190-195) refined over several calls: yields the RGB8 Image of the samples so far
    after each batch of `batch` samples per pixel (the last batch holds what is left), drawn from the SplitMix64 stream
    distributedRayTrace(job, spp, seed) uses, so the last image is that frame byte for byte."""
    if spp < 1 or batch < 1:
        raise ValueError(f"spp and batch must be at least 1, got {spp} and {batch}")
    acc = Accumulator(job, stream_spp=spp)
    try:
        done = 0
        while done < spp:
            k = min(batch, spp - done)
            img = acc.add(k, seed=seed, linear=False)
            done += k
            yield img
    finally:
        acc.close()


class AdaptiveAccumulator(_PixelState):
    """Adaptive sampling (rh_render_adaptive): progressive rendering that traces new samples only for the pixels whose
    standard error of the mean is still above a threshold in some channel.  Every pixel continues its own slice of the
    SplitMix64 stream sample_offsets(n, stream_spp, seed), so a pixel that ends with n samples has exactly the bytes of
    an n-sample render of that stream.  The state per pixel (count, sums of the colours and of their squares) stays on
    the device between calls.

    `shard_index` / `shard_count` / `band_height` as for render (the outputs are shard-compact).  `device`: outputs are
    CUDA tensors, else numpy arrays.  The first add() after creation or reset() fixes the scene, camera and max_depth."""

    _what = "adaptive accumulator"

    def __init__(self, job: Rendering, stream_spp: int, shard_index: int = 0, shard_count: int = 1, band_height: int = 0,
                 device: bool = False):
        L = lib()
        super().__init__(job, stream_spp, shard_index, shard_count, band_height, device, L.rh_adaptive_create, L.rh_adaptive_destroy)

    def add(self, spp: int, seed: int, threshold: float, min_spp: int = 8, rgb: bool = True, linear: bool = True,
            shadow: str | None = None, exact_boxes: bool = False, light_maps: bool = True, chunk_samples: int = 0,
            profile: bool = False, count: bool = False) -> Image:
        """One round: `spp` new samples for each pixel that is active by the rule of include/rayhs_b200.h (fewer than
        `min_spp` samples, or a channel's standard error above `threshold`, and room left in the stream).  Returns the
        Image of every pixel's samples so far: `pixels` (RGB8, when `rgb`), `linear` (float64, when `linear`) and this
        call's stats, with stats["n_active"] the number of pixels traced."""
        h = self._handle()
        job = self.job
        seed_box = C.c_uint64(seed)
        flags = _flags(exact_boxes=exact_boxes, shadow=shadow, light_maps=light_maps, device=self.device, profile=profile, count=count)
        o = _opts(job, spp, capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed_box), 0, self.shard_index, self.shard_count,
                  self.band_height, chunk_samples, flags)
        ao = capi.rh_adaptive_opts()
        ao.threshold, ao.min_spp = float(threshold), int(min_spp)
        shape = (self.rows, job.width, 3)
        empty = _alloc(self.device)
        px = empty(shape, "uint8") if rgb else None
        lin = empty(shape, "float64") if linear else None
        n_active = C.c_uint64()
        st = capi.rh_stats()
        check(lib().rh_render_adaptive(job.scene.device, C.byref(job.camera), C.byref(o), C.byref(ao), h,
                                       _ptr(px) if px is not None else None, _ptr(lin) if lin is not None else None,
                                       C.byref(n_active), C.byref(st)))
        stats = st.as_dict()
        stats["n_active"] = n_active.value
        return Image(job.width, self.rows, px, stats, None, lin)

    def state(self):
        """(counts uint32 [rows, width], sums float64 [rows, width, 3], sums of squares float64 [rows, width, 3]), numpy
        arrays or, with device=True, CUDA tensors."""
        shape = (self.rows, self.job.width)
        empty = _alloc(self.device)
        counts = empty(shape, "int32" if self.device else "uint32")  # (torch has no uint32 arithmetic to speak of)
        sums, sumsq = empty(shape + (3,), "float64"), empty(shape + (3,), "float64")
        check(lib().rh_adaptive_state(self._h, _ptr(counts), _ptr(sums), _ptr(sumsq), _flags(device=self.device)))
        return counts, sums, sumsq

    def reset(self) -> None:
        """Every count and sum back to 0; the next add() may use another scene, camera or max_depth."""
        check(lib().rh_adaptive_reset(self._h))


def adaptiveRayTrace(job: Rendering, max_spp: int = 64, batch: int = 4, min_spp: int = 8, threshold: float = 0.5 / 255,
                     seed: int = 24):
    """distributedRayTrace (RayHs.hs:190-195) refined adaptively: yields the RGB8 Image (stats["n_active"]: pixels traced
    in that round) after each round of `batch` new samples for every pixel still active, until no pixel is.  A pixel
    gets at least min(min_spp, max_spp) samples rounded up to whole batches and at most max_spp; it stops once every
    channel's standard error of the mean is at most `threshold`.  The default, half an RGB8 step (0.5 / 255), stops a
    pixel when one standard error of its mean no longer reaches the next quantisation step from the middle of one, so
    more samples would rarely change its byte.  Samples come from the stream distributedRayTrace(job, max_spp, seed)
    uses: a pixel that reaches max_spp has that frame's bytes."""
    if max_spp < 1 or batch < 1 or batch > max_spp:
        raise ValueError(f"need 1 <= batch <= max_spp, got batch {batch} and max_spp {max_spp}")
    if min_spp < 2:
        raise ValueError(f"min_spp must be at least 2, got {min_spp}")
    ad = AdaptiveAccumulator(job, stream_spp=max_spp)
    try:
        while True:
            img = ad.add(batch, seed, threshold, min_spp=min_spp, linear=False)
            if img.stats["n_active"] == 0:
                return
            yield img
    finally:
        ad.close()


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
