"""ctypes binding of oracle/_build/liborc.so — the CPU restatement of the reference path.

TEST INFRASTRUCTURE ONLY (see the header of oracle.cpp): imported by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs, never by
rayhs_b200/.  The scene is handed over as the POD `rh_raw_scene` (objects before any tree
build); the oracle builds its own tree with the KDTree.hs rule.

Besides renders and one-ray queries, the library answers the tests' batch questions over
caller-built rays [n, 6] (origin, direction) on host threads: closest hits, shadow verdicts,
traceRay colours and first-hit features (OracleScene.*_batch), and camera rays (camera_rays);
batch.cpp defines them, after oracle.cpp, in the same library.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "liborc.so")

# one rh_hit record (include/rayhs_b200.h), as orc_closest_batch writes it; declared here on its own so that the tests
# can hold it against the product's rayhs_b200.HIT_DTYPE and the header
HIT_DTYPE = np.dtype([("t", "<f8"), ("p", "<f8", 3), ("n", "<f8", 3), ("uv", "<f8", 2), ("object", "<i4"), ("tri", "<i4")])
assert HIT_DTYPE.itemsize == 80
# orc_trace_batch's ray counts, in its order, under the names of the product's stats
COUNT_NAMES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")


class orc_result_counts(C.Structure):
    _fields_ = [("rays", C.c_uint64 * 5), ("box_tests", C.c_uint64), ("tri_tests", C.c_uint64), ("prim_tests", C.c_uint64),
                ("seconds", C.c_double), ("threads", C.c_int32), ("pad_", C.c_int32)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} missing: run `python -m rayhs_b200.build`")
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        L.orc_scene_create.restype = vp
        L.orc_scene_create.argtypes = [vp]
        L.orc_scene_destroy.argtypes = [vp]
        L.orc_tree_stats.argtypes = [vp, C.c_int, C.POINTER(C.c_uint32)]
        L.orc_ray_from_pixel.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double)]
        L.orc_closest.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
        L.orc_color_at.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double)]
        L.orc_mod1.restype = C.c_double
        L.orc_mod1.argtypes = [C.c_double, C.c_double]
        L.orc_render.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp,
                                 vp, C.POINTER(orc_result_counts)]
        L.orc_render2.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.POINTER(orc_result_counts)]
        L.orc_camera_rays.argtypes = [vp, C.c_double, C.c_double, vp, C.c_uint64, vp]
        L.orc_closest_batch.argtypes = [vp, vp, C.c_uint64, vp, C.c_int]
        L.orc_shadow_batch.argtypes = [vp, C.c_uint32, vp, C.c_uint64, vp, C.c_int]
        L.orc_trace_batch.argtypes = [vp, vp, C.c_uint64, C.c_int, vp, vp, vp, C.c_int]
        L.orc_feature_batch.argtypes = [vp, vp, C.c_uint64, vp, vp, vp, vp, vp, C.c_int]
        _lib = L
    return _lib


class OracleScene:
    def __init__(self, raw_scene_ptr):
        """raw_scene_ptr: ctypes pointer to an rh_raw_scene (kept alive by the caller)."""
        self._h = lib().orc_scene_create(C.cast(raw_scene_ptr, C.c_void_p))

    def close(self):
        if self._h:
            lib().orc_scene_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tree_stats(self, obj: int):
        out = (C.c_uint32 * 5)()
        if lib().orc_tree_stats(self._h, obj, out) != 0:
            return None
        return dict(inner=out[0], leaves=out[1], empties=out[2], max_depth=out[3], max_leaf=out[4])

    def ray_from_pixel(self, camera, w, h, px, py):
        out = (C.c_double * 6)()
        lib().orc_ray_from_pixel(C.cast(C.pointer(camera), C.c_void_p), w, h, px, py, out)
        return np.array(out[:3]), np.array(out[3:])

    def closest(self, o, d):
        out = (C.c_double * 9)()
        ids = (C.c_int32 * 2)()
        hit = lib().orc_closest(self._h, (C.c_double * 3)(*o), (C.c_double * 3)(*d), out, ids)
        if not hit:
            return None
        return dict(p=np.array(out[0:3]), n=np.array(out[3:6]), uv=np.array(out[6:8]), t=out[8], object=ids[0], tri=ids[1])

    def color_at(self, material: int, u: float, v: float):
        out = (C.c_double * 3)()
        lib().orc_color_at(self._h, material, u, v, out)
        return np.array(out[:])

    def closest_batch(self, rays, threads=0):
        """closestIntersection for every row of rays [n, 6] (origin, direction): a record array of HIT_DTYPE."""
        rays = _rays(rays)
        out = np.empty(len(rays), dtype=HIT_DTYPE)
        assert lib().orc_closest_batch(self._h, rays.ctypes.data, len(rays), out.ctypes.data, threads) == 0
        return out

    def shadow_batch(self, light, rays, threads=0):
        """shadowIntersection towards light `light` for every row of rays [n, 6]: a bool array."""
        rays = _rays(rays)
        out = np.empty(len(rays), dtype=np.uint8)
        assert lib().orc_shadow_batch(self._h, int(light), rays.ctypes.data, len(rays), out.ctypes.data, threads) == 0
        return out.view(np.bool_)

    def trace_batch(self, rays, max_depth, threads=0):
        """traceRay sc 0 max_depth for every row of rays [n, 6]: (colors [n, 3], ids [n, 2], counts dict of COUNT_NAMES)."""
        rays = _rays(rays)
        colors = np.empty((len(rays), 3))
        ids = np.empty((len(rays), 2), dtype=np.int32)
        counts = np.zeros(5, dtype=np.uint64)
        assert lib().orc_trace_batch(self._h, rays.ctypes.data, len(rays), int(max_depth), colors.ctypes.data, ids.ctypes.data,
                                     counts.ctypes.data, threads) == 0
        return colors, ids, dict(zip(COUNT_NAMES, (int(c) for c in counts)))

    def features_batch(self, rays, threads=0):
        """The first-hit features of every row of rays [n, 6]: dict of t [n], n and albedo [n, 3], ids and uv [n, 2]."""
        rays = _rays(rays)
        n = len(rays)
        t, nn, al, uv = np.empty(n), np.empty((n, 3)), np.empty((n, 3)), np.empty((n, 2))
        ids = np.empty((n, 2), dtype=np.int32)
        assert lib().orc_feature_batch(self._h, rays.ctypes.data, n, t.ctypes.data, nn.ctypes.data, al.ctypes.data, ids.ctypes.data,
                                       uv.ctypes.data, threads) == 0
        return dict(t=t, n=nn, albedo=al, ids=ids, uv=uv)

    def render(self, camera, w, h, max_depth, spp=1, offsets=None, rows=(0, None, 1), threads=0, want_ids=True):
        """rayTrace / distributedRayTrace over rows[0]:rows[1]:rows[2].  Returns a dict with full-frame arrays
        rgb_f64 [h,w,3], rgb_u8, rgb_int (raw toIntC), hit_ids [h,w,spp,2] and the ray counters."""
        r0, r1, rs = rows
        r1 = h if r1 is None else r1
        rgb_f64 = np.zeros((h, w, 3), dtype=np.float64)
        rgb_u8 = np.zeros((h, w, 3), dtype=np.uint8)
        rgb_int = np.zeros((h, w, 3), dtype=np.int32)
        ids = np.full((h, w, spp, 2), -2, dtype=np.int32) if want_ids else None
        off_ptr = None
        if offsets is not None:
            offsets = np.ascontiguousarray(offsets, dtype=np.float64)
            assert offsets.size == w * h * spp * 2
            off_ptr = offsets.ctypes.data
        cnt = orc_result_counts()
        rc = lib().orc_render(self._h, C.cast(C.pointer(camera), C.c_void_p), w, h, max_depth, spp, off_ptr, r0, r1, rs, threads,
                              rgb_f64.ctypes.data, rgb_u8.ctypes.data, rgb_int.ctypes.data,
                              ids.ctypes.data if ids is not None else None, C.byref(cnt))
        assert rc == 0
        names = ["primary", "reflect", "probe", "exit", "shadow"]
        return dict(rgb_f64=rgb_f64, rgb_u8=rgb_u8, rgb_int=rgb_int, hit_ids=ids,
                    rays={n: int(cnt.rays[i]) for i, n in enumerate(names)}, rays_total=int(sum(cnt.rays)),
                    box_tests=int(cnt.box_tests), tri_tests=int(cnt.tri_tests), prim_tests=int(cnt.prim_tests),
                    seconds=cnt.seconds, threads=cnt.threads)


    def render_sample(self, camera, w, h, max_depth, spp=1, seed=None, rows=(0, None, 1), cols=(0, None, 1), threads=0,
                      want_ids=True):
        """The same for the pixels rows x cols only, with COMPACT outputs [n_rows, n_cols, ...] and the sample offsets
        taken from the SplitMix64 stream of `seed` in place (rh_sample_offsets_f64's stream; None: one sample at the
        pixel corner).  For frames whose full-size arrays do not fit the host (configs[4]: 8K x 64 spp)."""
        r0, r1, rs = rows
        c0, c1, cs = cols
        r1 = h if r1 is None else r1
        c1 = w if c1 is None else c1
        ys, xs = np.arange(r0, min(r1, h), rs), np.arange(c0, min(c1, w), cs)
        rgb_f64 = np.zeros((len(ys), len(xs), 3), dtype=np.float64)
        rgb_u8 = np.zeros((len(ys), len(xs), 3), dtype=np.uint8)
        ids = np.full((len(ys), len(xs), spp, 2), -2, dtype=np.int32) if want_ids else None
        cnt = orc_result_counts()
        rc = lib().orc_render2(self._h, C.cast(C.pointer(camera), C.c_void_p), w, h, max_depth, spp, None, 0 if seed is None else 1,
                               0 if seed is None else int(seed), r0, r1, rs, c0, c1, cs, 1, threads, rgb_f64.ctypes.data,
                               rgb_u8.ctypes.data, None, ids.ctypes.data if ids is not None else None, C.byref(cnt))
        assert rc == 0
        names = ["primary", "reflect", "probe", "exit", "shadow"]
        return dict(rows=ys, cols=xs, rgb_f64=rgb_f64, rgb_u8=rgb_u8, hit_ids=ids,
                    rays={n: int(cnt.rays[i]) for i, n in enumerate(names)}, rays_total=int(sum(cnt.rays)),
                    seconds=cnt.seconds, threads=cnt.threads)


def _rays(rays):
    return np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)


def camera_rays(camera, w, h, xy=None):
    """rayFromPixel (Projection.hs:22-46) of a w x h view at pixel coordinates xy [n, 2] (default: every pixel's (x, y),
    row-major), in one call: rays [n, 6] = origin, direction."""
    if xy is None:
        rows, cols = np.divmod(np.arange(h * w), w)
        xy = np.stack([cols, rows], axis=1)
    xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    rays = np.empty((len(xy), 6))
    lib().orc_camera_rays(C.cast(C.pointer(camera), C.c_void_p), w, h, xy.ctypes.data, len(xy), rays.ctypes.data)
    return rays


def mod1(n: float, d: float) -> float:
    return lib().orc_mod1(n, d)
