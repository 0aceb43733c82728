"""ctypes binding of the C ABI in include/rayhs_b200.h.

This is the same binding a Haskell `foreign import ccall` shim makes (INTEGRATION.md), written
for Python.  Loading fails loudly when librayhs_b200.so has not been built: there is no CPU
fallback anywhere in the product path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RAYHS_B200_LIB") or os.path.join(_HERE, "librayhs_b200.so")  # override: A/B builds only

# error classes
RH_OK, RH_ERR_ARG, RH_ERR_CUDA, RH_ERR_NCCL, RH_ERR_OOM, RH_ERR_STATE, RH_ERR_IO, RH_ERR_OVERFLOW = 0, -1, -2, -3, -4, -5, -6, -7
# kinds
RH_OBJ_PLANE, RH_OBJ_SPHERE, RH_OBJ_MESH = 0, 1, 2
RH_MAT_MIRROR, RH_MAT_DIFFUSE, RH_MAT_PLASTIC, RH_MAT_EMMIT, RH_MAT_TRANSPARENT, RH_MAT_SHOWNORMAL, RH_MAT_SHOWUV = range(7)
RH_CMAP_FLAT, RH_CMAP_CHECKER, RH_CMAP_TEXTURE = 0, 1, 2
RH_LIGHT_DIRECTIONAL, RH_LIGHT_POINT = 0, 1
RH_PROJ_ORTHOGRAPHIC, RH_PROJ_PERSPECTIVE = 0, 1
RH_OFFSETS_NONE, RH_OFFSETS_F64, RH_OFFSETS_F32, RH_OFFSETS_TILED_F64, RH_OFFSETS_SPLITMIX64 = 0, 1, 2, 3, 4
RH_FLAG_HIT_IDS, RH_FLAG_DEVICE_OUT, RH_FLAG_DEVICE_OFFSETS, RH_FLAG_COUNT, RH_FLAG_PROFILE, RH_FLAG_EXACT_BOXES = 1, 2, 4, 8, 16, 32
RH_FLAG_SHADOW_POOLED, RH_FLAG_SHADOW_SPLIT, RH_FLAG_PEER_FRAMES = 64, 128, 256
RH_FLAG_NO_LIGHT_MAPS = 2048
RH_FLAG_SHARD_OFFSETS = 4096
RH_NO_NODE = 0xFFFFFFFF

d3 = C.c_double * 3
d2 = C.c_double * 2


class rh_material(C.Structure):
    _fields_ = [("kind", C.c_int32), ("cmap_kind", C.c_int32), ("ior", C.c_double), ("color1", d3), ("color2", d3),
                ("size", C.c_double), ("texture", C.c_int32), ("pad_", C.c_int32), ("pad2_", d2)]


class rh_light(C.Structure):
    _fields_ = [("kind", C.c_int32), ("pad_", C.c_int32), ("vec", d3), ("color", d3), ("radius", C.c_double)]


class rh_texture(C.Structure):
    _fields_ = [("w", C.c_int32), ("h", C.c_int32), ("offset", C.c_uint64)]


class rh_camera(C.Structure):
    _fields_ = [("position", d3), ("target", d3), ("up", d3), ("projection", C.c_int32), ("pad_", C.c_int32),
                ("fovy", C.c_double), ("proj_width", C.c_double), ("proj_height", C.c_double), ("near_", C.c_double)]


class rh_raw_object(C.Structure):
    _fields_ = [("kind", C.c_int32), ("material", C.c_int32), ("a", d3), ("b", d3), ("c", d3), ("n_verts", C.c_uint32),
                ("n_indices", C.c_uint32), ("positions", C.POINTER(C.c_double)), ("normals", C.POINTER(C.c_double)),
                ("uvs", C.POINTER(C.c_double)), ("indices", C.POINTER(C.c_uint32))]


class rh_raw_scene(C.Structure):
    _fields_ = [("n_objects", C.c_uint32), ("n_materials", C.c_uint32), ("n_lights", C.c_uint32), ("n_textures", C.c_uint32),
                ("objects", C.POINTER(rh_raw_object)), ("materials", C.POINTER(rh_material)), ("lights", C.POINTER(rh_light)),
                ("textures", C.POINTER(rh_texture)), ("texels", C.POINTER(C.c_double)), ("n_texels", C.c_uint64)]


class rh_node(C.Structure):
    _fields_ = [("lo", d3), ("hi", d3), ("left", C.c_uint32), ("right", C.c_uint32), ("leaf_index", C.c_uint32),
                ("is_leaf", C.c_uint32)]


class rh_tri(C.Structure):
    _fields_ = [("p0", d3), ("e1", d3), ("e2", d3), ("tri_id", C.c_uint32), ("pad_", C.c_uint32)]


class rh_tri_shade(C.Structure):
    _fields_ = [("n0", d3), ("n1", d3), ("n2", d3), ("uv0", d2), ("uv1", d2), ("uv2", d2), ("pad_", C.c_double)]


class rh_object(C.Structure):
    _fields_ = [("kind", C.c_int32), ("material", C.c_int32), ("a", d3), ("b", d3), ("c", d3), ("root", C.c_uint32),
                ("n_leaves", C.c_uint32), ("depth", C.c_uint32), ("pad_", C.c_uint32)]


class rh_scene_desc(C.Structure):
    _fields_ = [("n_objects", C.c_uint32), ("n_materials", C.c_uint32), ("n_lights", C.c_uint32), ("n_textures", C.c_uint32),
                ("n_nodes", C.c_uint32), ("n_tris", C.c_uint32), ("objects", C.POINTER(rh_object)),
                ("materials", C.POINTER(rh_material)), ("lights", C.POINTER(rh_light)), ("textures", C.POINTER(rh_texture)),
                ("texels", C.POINTER(C.c_double)), ("n_texels", C.c_uint64), ("nodes", C.POINTER(rh_node)),
                ("tris", C.POINTER(rh_tri)), ("tri_shade", C.POINTER(rh_tri_shade))]


class rh_render_opts(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("max_depth", C.c_int32), ("spp", C.c_int32),
                ("offset_mode", C.c_int32), ("offset_tile", C.c_int32), ("offsets", C.c_void_p), ("shard_index", C.c_int32),
                ("shard_count", C.c_int32), ("band_height", C.c_int32), ("chunk_samples", C.c_int32), ("flags", C.c_int32),
                ("n_peer_frames", C.c_int32), ("peer_frames", C.POINTER(C.c_void_p))]


class rh_stats(C.Structure):
    _fields_ = [("rays_primary", C.c_uint64), ("rays_reflect", C.c_uint64), ("rays_probe", C.c_uint64),
                ("rays_exit", C.c_uint64), ("rays_shadow", C.c_uint64), ("rays_shadow_culled", C.c_uint64), ("shadow_tasks", C.c_uint64),
                ("shadow_tasks_queued", C.c_uint64), ("shadow_walk_pairs", C.c_uint64), ("deep_stack_pushes", C.c_uint64), ("queued_rays", C.c_uint64),
                ("box_tests", C.c_uint64), ("tri_tests", C.c_uint64), ("prim_tests", C.c_uint64),
                ("shade_fetches", C.c_uint64), ("texel_fetches", C.c_uint64), ("node_visits", C.c_uint64),
                ("shadow_box_tests", C.c_uint64), ("shadow_tri_tests", C.c_uint64), ("shadow_prim_tests", C.c_uint64),
                ("shadow_node_visits", C.c_uint64), ("node_visits_global", C.c_uint64), ("shadow_node_visits_global", C.c_uint64),
                ("tri_records", C.c_uint64), ("shadow_tri_records", C.c_uint64),
                ("upload_bytes", C.c_uint64), ("ms_total", C.c_double), ("ms_trace", C.c_double), ("ms_shadow", C.c_double),
                ("ms_resolve", C.c_double), ("trace_launches", C.c_uint32), ("shadow_launches", C.c_uint32),
                ("kernel_launches", C.c_uint32), ("chunks", C.c_uint32), ("negative_channels", C.c_uint32),
                ("queue_factor", C.c_uint32), ("shadow_split", C.c_uint32), ("reserved_", C.c_uint32)]

    def rays_total(self) -> int:
        return self.rays_primary + self.rays_reflect + self.rays_probe + self.rays_exit + self.rays_shadow

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class rh_hit(C.Structure):
    _fields_ = [("t", C.c_double), ("p", d3), ("n", d3), ("uv", d2), ("object", C.c_int32), ("tri", C.c_int32)]


class rh_trace_opts(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("flags", C.c_int32), ("chunk_rays", C.c_uint32), ("reserved_", C.c_uint32)]


# struct sizes the header promises (checked by tests/test_abi.py against the compiled library too)
assert C.sizeof(rh_material) == 96 and C.sizeof(rh_light) == 64 and C.sizeof(rh_node) == 64
assert C.sizeof(rh_tri) == 80 and C.sizeof(rh_tri_shade) == 128 and C.sizeof(rh_object) == 96
assert C.sizeof(rh_hit) == 80 and C.sizeof(rh_trace_opts) == 16

vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/rayhs_b200.h declares
SIGNATURES = {
    "rh_init": (C.c_int, [C.c_int]),
    "rh_shutdown": (None, []),
    "rh_last_error": (C.c_char_p, []),
    "rh_abi_version": (C.c_int, []),
    "rh_launch_count": (C.c_uint64, []),
    "rh_scene_create": (C.c_int, [C.POINTER(rh_scene_desc), C.POINTER(vp)]),
    "rh_scene_destroy": (None, [vp]),
    "rh_scene_info": (C.c_int, [vp, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "rh_scene_record_bytes": (C.c_int, [vp, C.POINTER(C.c_uint64)]),
    "rh_scene_light_tables": (C.c_int, [vp, C.POINTER(C.c_uint32), vp, vp, vp]),
    "rh_render": (C.c_int, [vp, C.POINTER(rh_camera), C.POINTER(rh_render_opts), vp, vp, C.POINTER(rh_stats)]),
    "rh_closest_intersection": (C.c_int, [vp, vp, C.c_uint64, vp, C.c_int32]),
    "rh_shadow_intersection": (C.c_int, [vp, C.c_uint32, vp, C.c_uint64, vp, C.c_int32]),
    "rh_trace_rays": (C.c_int, [vp, vp, C.c_uint64, C.POINTER(rh_trace_opts), vp, vp, C.POINTER(rh_stats)]),
    "rh_shard_rows": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "rh_default_band_height": (C.c_int, [C.c_int, C.c_int]),
    "rh_deinterleave_bands": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "rh_multi_init": (C.c_int, [C.c_int]),
    "rh_multi_shutdown": (None, []),
    "rh_multi_gpu_count": (C.c_int, []),
    "rh_multi_scene_create": (C.c_int, [C.POINTER(rh_scene_desc), C.POINTER(vp)]),
    "rh_multi_scene_destroy": (None, [vp]),
    "rh_multi_render": (C.c_int, [vp, C.POINTER(rh_camera), C.POINTER(rh_render_opts), vp, C.POINTER(rh_stats)]),
    "rh_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp), C.c_char_p]),
    "rh_peer_open": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "rh_peer_close": (C.c_int, [vp]),
    "rh_peer_free": (C.c_int, [vp]),
    "rh_bench_gather": (C.c_int, [C.c_uint64, C.c_int, C.POINTER(C.c_double)]),
    "rh_bench_stream": (C.c_int, [C.c_uint64, C.c_int, C.POINTER(C.c_double)]),
    "rh_bench_dfma": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "rh_flatten": (C.c_int, [C.POINTER(rh_raw_scene), C.POINTER(vp)]),
    "rh_flat_desc": (C.POINTER(rh_scene_desc), [vp]),
    "rh_flat_destroy": (None, [vp]),
    "rh_load_json": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(vp)]),
    "rh_load_pack": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "rh_save_pack": (C.c_int, [vp, C.c_char_p]),
    "rh_make_synthetic": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint64, C.POINTER(vp)]),
    "rh_loaded_raw": (C.POINTER(rh_raw_scene), [vp]),
    "rh_loaded_camera": (C.POINTER(rh_camera), [vp]),
    "rh_loaded_size": (None, [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rh_loaded_destroy": (None, [vp]),
    "rh_sample_offsets_f64": (None, [C.c_uint64, C.c_uint64, C.c_int, vp]),
    "rh_sample_offsets_f32": (None, [C.c_uint64, C.c_uint64, C.c_int, vp]),
    "rh_sample_offsets_f64_at": (None, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, vp]),
    "rh_write_ppm": (C.c_int, [C.c_char_p, vp, C.c_int, C.c_int]),
    "rh_light_map_build": (C.c_int, [C.POINTER(C.c_double), C.POINTER(rh_tri), C.c_uint32, C.c_int, vp, C.POINTER(C.c_int),
                                     C.POINTER(C.c_double)]),
    "rh_lit_triangles": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(rh_tri), C.c_uint32, vp]),
    "rh_cull_tree_build": (C.c_int, [C.POINTER(rh_tri), C.c_uint32, vp, vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
}

_lib = None


class RayHsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rayhs_b200 error {code}: {message}")
        self.code = code


def lib() -> C.CDLL:
    """Load librayhs_b200.so (once).  Raises if it has not been built — no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m rayhs_b200.build` (the product has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int) -> None:
    if code != RH_OK:
        raise RayHsError(code, lib().rh_last_error().decode("utf-8", "replace"))
