"""The oracle's view of thin-lens cameras (RH_PROJ_THIN_LENS), for the tests and scripts/lens_rate.py.

oracle/oracle.cpp restates the reference, whose cameras are orthographic and perspective; the thin lens is this
project's extension.  tests/lens_oracle.cpp adds the lens ray on top of the unchanged oracle, and this module renders
with it as the oracle renders: camera_rays gives the rays of any camera at pixel coordinates, and render /
render_sample trace them with OracleScene.trace_batch (traceRay, RayHs.hs:149-154) and fold the samples as
distributedTracePixel does (RayHs.hs:169-188: a left sum in sample order, then times 1 / spp; one sample at the pixel
corner without offsets), returning what OracleScene.render / render_sample return."""
import ctypes as C
import os

import numpy as np

from tests.util import temp_library, to_int_c

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNT_NAMES = ("primary", "reflect", "probe", "exit", "shadow")
GAMMA = np.uint64(0x9E3779B97F4A7C15)
_lib = None


def lib():
    global _lib
    if _lib is None:
        from rayhs_b200.build import ORACLE_FLAGS

        srcs = [os.path.join(ROOT, "tests", "lens_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
                os.path.join(ROOT, "include", "rayhs_b200.h")]
        _lib = temp_library("lens_oracle", srcs, ORACLE_FLAGS)
        vp = C.c_void_p
        _lib.lens_camera_rays.argtypes = [vp, C.c_double, C.c_double, vp, C.c_uint64, vp]
        _lib.lens_camera_rays.restype = None
    return _lib


def camera_rays(camera, w, h, xy=None):
    """The rays [n, 6] (origin, direction) of any rh_camera of a w x h view at pixel coordinates xy [n, 2] (default:
    every pixel's (x, y), row-major): the oracle's rayFromPixel, and the lens ray for a thin lens of radius != 0."""
    if xy is None:
        rows, cols = np.divmod(np.arange(h * w), w)
        xy = np.stack([cols, rows], axis=1)
    xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    rays = np.empty((len(xy), 6))
    lib().lens_camera_rays(C.cast(C.pointer(camera), C.c_void_p), w, h, xy.ctypes.data, len(xy), rays.ctypes.data)
    return rays


def splitmix_offsets(seed, pixels, spp):
    """[len(pixels), spp, 2]: the offsets rh_sample_offsets_f64(seed, ...) gives the pixels (row-major indices) of a frame
    with spp samples per pixel, evaluated in place (value k of the stream: the state after k + 1 steps)."""
    g = (np.asarray(pixels, dtype=np.uint64)[:, None] * np.uint64(spp) + np.arange(spp, dtype=np.uint64)[None, :])
    out = np.empty(g.shape + (2,))
    with np.errstate(over="ignore"):
        for c in range(2):
            z = np.uint64(seed) + (np.uint64(2) * g + np.uint64(c) + np.uint64(1)) * GAMMA
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
            out[..., c] = (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0) - 0.5
    return out


def _trace(orc, camera, w, h, max_depth, rows, cols, spp, offsets):
    """Colours [n_rows, n_cols, 3], hit ids [n_rows, n_cols, spp, 2] and counts of pixels rows x cols; offsets
    [n_rows * n_cols, spp, 2] (None: one sample at the pixel corner)."""
    yy, xx = np.meshgrid(np.asarray(rows, dtype=np.float64), np.asarray(cols, dtype=np.float64), indexing="ij")
    base = np.stack([xx.ravel(), yy.ravel()], axis=1)
    n = len(base)
    xy = base[:, None, :] if offsets is None else base[:, None, :] + offsets.reshape(n, spp, 2)
    col, ids, counts = orc.trace_batch(camera_rays(camera, w, h, xy.reshape(-1, 2)), max_depth)
    counts = {k: counts["rays_" + k] for k in COUNT_NAMES}
    col = col.reshape(n, -1, 3)
    if offsets is None:
        lin = col[:, 0]
    else:
        s = np.zeros((n, 3))
        for k in range(spp):
            s = s + col[:, k]
        lin = (1.0 / spp) * s
    shape = (len(rows), len(cols))
    return lin.reshape(shape + (3,)), ids.reshape(shape + (-1, 2)), counts


def render(orc, camera, w, h, max_depth, spp=1, offsets=None):
    """OracleScene.render's outputs (rgb_f64, rgb_u8, hit_ids, rays) of the whole frame, for any camera."""
    off = None if offsets is None else np.asarray(offsets, dtype=np.float64).reshape(w * h, spp, 2)
    lin, ids, counts = _trace(orc, camera, w, h, max_depth, range(h), range(w), spp, off)
    return dict(rgb_f64=lin, rgb_u8=to_int_c(lin), hit_ids=ids, rays=counts, rays_total=sum(counts.values()))


def render_sample(orc, camera, w, h, max_depth, spp, seed, rows=(0, None, 1), cols=(0, None, 1)):
    """OracleScene.render_sample's outputs (compact rows x cols) with the SplitMix64 stream of `seed`, for any camera."""
    ys = np.arange(rows[0], h if rows[1] is None else min(rows[1], h), rows[2])
    xs = np.arange(cols[0], w if cols[1] is None else min(cols[1], w), cols[2])
    pix = (ys[:, None] * w + xs[None, :]).ravel()
    lin, ids, counts = _trace(orc, camera, w, h, max_depth, ys, xs, spp, splitmix_offsets(seed, pix, spp))
    return dict(rows=ys, cols=xs, rgb_f64=lin, rgb_u8=to_int_c(lin), hit_ids=ids, rays=counts)
