"""Batch oracle of the radiance-query tests: tests/trace_oracle.cpp (oracle/oracle.cpp as it stands + a batch traceRay)
compiled with the oracle's own flags into a library in the temporary directory, named by a digest of its sources, so
that the repository tree is never written.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "trace_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
           os.path.join(ROOT, "include", "rayhs_b200.h")]
FLAGS = ["-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared"]  # rayhs_b200/build.py's oracle flags
COUNT_NAMES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = temp_library("trace_oracle", SOURCES, FLAGS)
        vp = C.c_void_p
        L.orc_scene_create.restype = vp
        L.orc_scene_create.argtypes = [vp]
        L.orc_scene_destroy.argtypes = [vp]
        L.orc_ray_from_pixel.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double)]
        L.orc_trace_batch.argtypes = [vp, vp, C.c_uint64, C.c_int, vp, vp, vp, C.c_int]
        _lib = L
    return _lib


class TraceOracle:
    """traceRay of the oracle over many rays at once (and its camera rays)."""

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
    def camera_rays(camera, w, h):
        """The pixel-centre camera rays (rayFromPixel, Projection.hs:22-46) of a w x h view, row-major: [w * h, 6]."""
        out = np.empty((h * w, 6))
        buf = (C.c_double * 6)()
        cam = C.cast(C.pointer(camera), C.c_void_p)
        for y in range(h):
            for x in range(w):
                lib().orc_ray_from_pixel(cam, w, h, x, y, buf)
                out[y * w + x] = buf[:]
        return out

    def trace_batch(self, rays, max_depth, threads=0):
        """traceRay sc 0 max_depth for every row of rays [n, 6]: (colors [n, 3], ids [n, 2], counts dict)."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        colors = np.empty((len(rays), 3))
        ids = np.empty((len(rays), 2), dtype=np.int32)
        counts = np.zeros(5, dtype=np.uint64)
        assert lib().orc_trace_batch(self._h, rays.ctypes.data, len(rays), int(max_depth), colors.ctypes.data, ids.ctypes.data,
                                     counts.ctypes.data, threads) == 0
        return colors, ids, dict(zip(COUNT_NAMES, (int(c) for c in counts)))
