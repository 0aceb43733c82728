"""The oracle's view of sphere lights (RH_LIGHT_SPHERE), for the tests and scripts/sphere_light_rate.py.

oracle/oracle.cpp restates the reference, whose lights are points and directions; the sphere light is this project's
extension.  tests/sphere_light_oracle.cpp restates the shading (accumDiffuse .. traceRay, RayHs.hs:89-154) on top of the
unchanged oracle with each sphere light sampled per shading point, and SphereOracle.trace_batch answers what
OracleScene.trace_batch answers.  So tests.lens_oracle's render / render_sample (the pixel fold of RayHs.hs:156-195,
any camera) render with it as the oracle renders."""
import ctypes as C
import os

import numpy as np

from tests import lens_oracle
from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNT_NAMES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
_lib = None


def lib():
    global _lib
    if _lib is None:
        from rayhs_b200.build import ORACLE_FLAGS

        srcs = [os.path.join(ROOT, "tests", "sphere_light_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
                os.path.join(ROOT, "include", "rayhs_b200.h")]
        _lib = temp_library("sphere_light_oracle", srcs, ORACLE_FLAGS)
        vp = C.c_void_p
        _lib.orc_scene_create.restype = vp
        _lib.orc_scene_create.argtypes = [vp]
        _lib.orc_scene_destroy.argtypes = [vp]
        _lib.sl_sphere_points.argtypes = [vp, C.c_uint32, vp, C.c_uint64, vp]
        _lib.sl_trace_batch.argtypes = [vp, vp, C.c_uint64, C.c_int, vp, vp, vp]
    return _lib


class SphereOracle:
    """The oracle's scene (oracle.cpp's orc_scene_create, compiled into this library) of an rh_raw_scene pointer."""

    def __init__(self, raw_scene_ptr):
        self._h = lib().orc_scene_create(C.cast(raw_scene_ptr, C.c_void_p))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_scene_destroy(self._h)
            self._h = None

    def sphere_points(self, light, points):
        """L' of light `light` for shading points [n, 3]: [n, 3] (the light's sample, whatever its kind)."""
        p = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        out = np.empty_like(p)
        assert lib().sl_sphere_points(self._h, int(light), p.ctypes.data, len(p), out.ctypes.data) == 0
        return out

    def trace_batch(self, rays, max_depth, threads=0):
        """traceRay sc 0 max_depth with sphere lights for every row of rays [n, 6]: (colors [n, 3], ids [n, 2], counts)."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        colors = np.empty((len(rays), 3))
        ids = np.empty((len(rays), 2), dtype=np.int32)
        counts = np.zeros(5, dtype=np.uint64)
        assert lib().sl_trace_batch(self._h, rays.ctypes.data, len(rays), int(max_depth), colors.ctypes.data, ids.ctypes.data,
                                    counts.ctypes.data) == 0
        return colors, ids, dict(zip(COUNT_NAMES, (int(c) for c in counts)))

    def render(self, camera, w, h, max_depth, spp=1, offsets=None):
        """OracleScene.render's outputs (rgb_f64, rgb_u8, hit_ids, rays) of the whole frame."""
        return lens_oracle.render(self, camera, w, h, max_depth, spp, offsets)

    def render_sample(self, camera, w, h, max_depth, spp, seed, rows=(0, None, 1), cols=(0, None, 1)):
        """OracleScene.render_sample's outputs with the SplitMix64 stream of `seed`."""
        return lens_oracle.render_sample(self, camera, w, h, max_depth, spp, seed, rows, cols)
