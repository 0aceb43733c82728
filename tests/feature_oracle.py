"""Oracle of the feature-buffer tests: tests/feature_oracle.cpp (oracle/oracle.cpp as it stands + camera rays and a
batch of closestIntersection + colorAt) compiled with the oracle's own flags into a library in the temporary directory,
named by a digest of its sources, so that the repository tree is never written.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "feature_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
           os.path.join(ROOT, "include", "rayhs_b200.h")]
FLAGS = ["-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared"]  # rayhs_b200/build.py's oracle flags

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = temp_library("feature_oracle", SOURCES, FLAGS)
        vp = C.c_void_p
        L.orc_scene_create.restype = vp
        L.orc_scene_create.argtypes = [vp]
        L.orc_scene_destroy.argtypes = [vp]
        L.orc_camera_rays.argtypes = [vp, C.c_double, C.c_double, vp, C.c_uint64, vp]
        L.orc_feature_batch.argtypes = [vp, vp, C.c_uint64, vp, vp, vp, vp, vp, C.c_int]
        L.orc_color_at.argtypes = [vp, C.c_int, C.c_double, C.c_double, vp]
        _lib = L
    return _lib


class FeatureOracle:
    """Per-sample first-hit features of the oracle, and the per-pixel buffers rh_render_features defines from them."""

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

    def samples(self, camera, w, h, ox, oy):
        """The camera rays at pixel coordinates (col + ox, row + oy) for ox, oy [h * w, spp] (float64, pixel-major), through
        the batch: dict of rays [h*w*spp, 6] and, per pixel and sample, t [h*w, spp], n and albedo [h*w, spp, 3], ids and
        uv [h*w, spp, 2]."""
        spp = ox.shape[1]
        rows, cols = np.divmod(np.arange(h * w), w)
        xy = np.empty((h * w, spp, 2))
        xy[..., 0] = cols[:, None] + ox
        xy[..., 1] = rows[:, None] + oy
        n = h * w * spp
        rays = np.empty((n, 6))
        lib().orc_camera_rays(C.cast(C.pointer(camera), C.c_void_p), w, h, np.ascontiguousarray(xy).ctypes.data, n, rays.ctypes.data)
        t, nn, al, uv = np.empty(n), np.empty((n, 3)), np.empty((n, 3)), np.empty((n, 2))
        ids = np.empty((n, 2), dtype=np.int32)
        assert lib().orc_feature_batch(self._h, rays.ctypes.data, n, t.ctypes.data, nn.ctypes.data, al.ctypes.data, ids.ctypes.data,
                                       uv.ctypes.data, 0) == 0
        return dict(rays=rays, t=t.reshape(h * w, spp), n=nn.reshape(h * w, spp, 3), albedo=al.reshape(h * w, spp, 3),
                    ids=ids.reshape(h * w, spp, 2), uv=uv.reshape(h * w, spp, 2))

    def color_at(self, material, u, v):
        """colorAt (ColorMap.hs:18-58) of the scene's material `material` at (u, v)."""
        out = (C.c_double * 3)()
        lib().orc_color_at(self._h, int(material), float(u), float(v), out)
        return np.array(out[:])

    @staticmethod
    def fold(s, w, h):
        """The per-pixel buffers of samples `s`: albedo [h, w, 3], normal [h, w, 3], depth [h, w], hits [h, w] and ids
        [h, w, spp, 2]; foldl (+) 0 over the samples in sample order, per channel, then times 1.0 / spp (depth: 1.0 / hits
        over the hitting samples' t)."""
        spp = s["t"].shape[1]
        hit = s["ids"][..., 0] >= 0
        a, nn, ts = np.zeros((h * w, 3)), np.zeros((h * w, 3)), np.zeros(h * w)
        for k in range(spp):
            a = a + s["albedo"][:, k]
            nn = nn + s["n"][:, k]
            ts = ts + np.where(hit[:, k], s["t"][:, k], 0.0)
        inv = 1.0 / spp
        hits = hit.sum(axis=1).astype(np.uint32)
        with np.errstate(divide="ignore", invalid="ignore"):
            depth = np.where(hits > 0, (1.0 / hits.astype(np.float64)) * ts, np.inf)
        return dict(albedo=(inv * a).reshape(h, w, 3), normal=(inv * nn).reshape(h, w, 3), depth=depth.reshape(h, w),
                    hits=hits.reshape(h, w), ids=s["ids"].reshape(h, w, spp, 2))
