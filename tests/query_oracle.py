"""Batch oracle of the ray-query tests: tests/query_oracle.cpp (oracle/oracle.cpp as it stands + two batch entry
points) compiled with the oracle's own flags into a library in the temporary directory, named by a digest of its
sources, so that the repository tree is never written.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "query_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
           os.path.join(ROOT, "include", "rayhs_b200.h")]
FLAGS = ["-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared"]  # rayhs_b200/build.py's oracle flags

# one rh_hit record (include/rayhs_b200.h)
HIT_DTYPE = np.dtype([("t", "<f8"), ("p", "<f8", 3), ("n", "<f8", 3), ("uv", "<f8", 2), ("object", "<i4"), ("tri", "<i4")])
assert HIT_DTYPE.itemsize == 80

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = temp_library("query_oracle", SOURCES, FLAGS)
        vp = C.c_void_p
        L.orc_scene_create.restype = vp
        L.orc_scene_create.argtypes = [vp]
        L.orc_scene_destroy.argtypes = [vp]
        L.orc_ray_from_pixel.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double)]
        L.orc_closest_batch.argtypes = [vp, vp, C.c_uint64, vp, C.c_int]
        L.orc_shadow_batch.argtypes = [vp, C.c_uint32, vp, C.c_uint64, vp, C.c_int]
        _lib = L
    return _lib


class BatchOracle:
    """closestIntersection / shadowIntersection of the oracle over many rays at once (and its camera rays)."""

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

    @staticmethod
    def ray_from_pixel(camera, w, h, px, py):
        """rayFromPixel (Projection.hs:22-46): origin, direction."""
        out = (C.c_double * 6)()
        lib().orc_ray_from_pixel(C.cast(C.pointer(camera), C.c_void_p), w, h, px, py, out)
        return np.array(out[:3]), np.array(out[3:])

    def closest_batch(self, rays, threads=0):
        """closestIntersection for every row of rays [n, 6] (origin, direction): a record array of HIT_DTYPE."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        out = np.empty(len(rays), dtype=HIT_DTYPE)
        assert lib().orc_closest_batch(self._h, rays.ctypes.data, len(rays), out.ctypes.data, threads) == 0
        return out

    def shadow_batch(self, light, rays, threads=0):
        """shadowIntersection towards light `light` for every row of rays [n, 6]: a bool array."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        out = np.empty(len(rays), dtype=np.uint8)
        assert lib().orc_shadow_batch(self._h, int(light), rays.ctypes.data, len(rays), out.ctypes.data, threads) == 0
        return out.view(np.bool_)
