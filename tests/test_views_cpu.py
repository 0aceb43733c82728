"""CPU tests of the camera batches (rh_render_views / renderViews): the entry point is exported and bound, rh_views'
layout in the header equals the ctypes mirror, a call without a device fails loudly, and the Python layer's output
shapes, dtypes, flag bits, camera and seed tables and refusals with the library stubbed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["cameras", "n_views", "reserved_", "seeds"]


def test_symbol_is_exported_and_bound():
    L = capi.lib()
    args = capi.SIGNATURES["rh_render_views"][1]
    assert L.rh_render_views.argtypes == args
    assert len(args) == 7 and args[1]._type_ is capi.rh_views and args[2]._type_ is capi.rh_render_opts
    assert args[6]._type_ is capi.rh_stats
    assert rh.renderViews is host.renderViews and rh.Views is host.Views
    assert "renderViews" in rh.__all__ and "Views" in rh.__all__


def test_rh_views_layout_matches_the_header():
    """sizeof / offsetof from a C program compiled against the header equal the ctypes mirror (24 bytes)."""
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){' + \
        'printf("size %zu\\n", sizeof(rh_views));' + \
        "".join(f'printf("{f} %zu\\n", offsetof(rh_views, {f}));' for f in FIELDS) + "return 0;}"
    exe = os.path.join(ROOT, "build", "abi_rh_views")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    out = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert out["size"] == C.sizeof(capi.rh_views) == 24
    for f in FIELDS:
        assert out[f] == getattr(capi.rh_views, f).offset, f


def test_without_a_device_the_call_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    o = capi.rh_render_opts()
    o.width, o.height, o.spp = 4, 4, 1
    cams = (capi.rh_camera * 2)()
    vw = capi.rh_views()
    vw.cameras, vw.n_views = C.cast(cams, C.POINTER(capi.rh_camera)), 2
    rgb = np.empty((2, 4, 4, 3), np.uint8)
    assert L.rh_render_views(None, C.byref(vw), C.byref(o), rgb.ctypes.data, None, None, None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()


# ---------------------------------------------------------------- Python layer
class _FakeLib:
    """Stands in for librayhs_b200.so: records the rh_render_views call (the cameras and seeds it would read)."""

    def __init__(self):
        self.calls = []

    def rh_default_band_height(self, h, g):
        return h if g <= 1 else 4

    def rh_shard_rows(self, h, g, bh):
        n_bands = (h + bh - 1) // bh
        return (n_bands + g - 1) // g * bh

    def rh_render_views(self, scene, views, opts, rgb, linear, ids, stats):
        o, v = opts._obj, views._obj
        seeds = [v.seeds[i] for i in range(v.n_views)] if v.seeds else None
        seed = C.c_uint64.from_address(o.offsets).value if o.offset_mode == capi.RH_OFFSETS_SPLITMIX64 else None
        self.calls.append(dict(scene=scene, size=(o.width, o.height, o.spp, o.max_depth), mode=o.offset_mode, offsets=o.offsets,
                               seed=seed, tile=o.offset_tile, shard=(o.shard_index, o.shard_count, o.band_height),
                               chunk=o.chunk_samples, flags=o.flags, n_views=v.n_views, reserved=v.reserved_,
                               positions=[tuple(v.cameras[i].position) for i in range(v.n_views)],
                               projections=[v.cameras[i].projection for i in range(v.n_views)], seeds=seeds,
                               rgb=rgb, linear=linear, ids=ids))
        stats._obj.rays_primary = 13
        return 0


class _Job:
    class scene:
        device = "scene-handle"

    camera = capi.rh_camera()
    width, height, maxDepth = 10, 6, 3


def cameras(n):
    out = []
    for i in range(n):
        c = capi.rh_camera()
        c.position[:] = (i, 0.5 * i, -2.0)
        c.target[:] = (0, 0, 1)
        c.up[:] = (0, 1, 0)
        c.projection = capi.RH_PROJ_PERSPECTIVE if i % 2 else capi.RH_PROJ_ORTHOGRAPHIC
        c.fovy = 1.0
        out.append(c)
    return out


@pytest.fixture
def fake(monkeypatch):
    L = _FakeLib()
    monkeypatch.setattr(host, "lib", lambda: L)
    return L


def test_shapes_dtypes_and_the_camera_table(fake):
    vs = rh.renderViews(_Job, cameras(3), spp=2, seed=5, want_hit_ids=True)
    assert vs.pixels.shape == (3, 6, 10, 3) and vs.pixels.dtype == np.uint8 and vs.linear is None
    assert vs.hit_ids.shape == (3, 6, 10, 2, 2) and vs.hit_ids.dtype == np.int32
    assert vs.stats["rays_primary"] == 13
    (c,) = fake.calls
    assert c["scene"] == "scene-handle" and c["size"] == (10, 6, 2, 3) and c["n_views"] == 3 and c["reserved"] == 0
    assert c["positions"] == [(0, 0, -2), (1, 0.5, -2), (2, 1, -2)] and c["projections"] == [0, 1, 0]
    assert c["mode"] == capi.RH_OFFSETS_SPLITMIX64 and c["seed"] == 5 and c["seeds"] is None
    assert c["flags"] == capi.RH_FLAG_HIT_IDS and c["linear"] is None
    assert c["rgb"] == vs.pixels.ctypes.data and c["ids"] == vs.hit_ids.ctypes.data


def test_linear_only_flags_and_shards(fake):
    vs = rh.renderViews(_Job, cameras(2), rgb=False, linear=True, shadow="split", exact_boxes=True, light_maps=False,
                        chunk_samples=40, shard_index=1, shard_count=2, band_height=2, profile=True)
    assert vs.pixels is None and vs.hit_ids is None
    assert vs.linear.shape == (2, 4, 10, 3) and vs.linear.dtype == np.float64
    c = fake.calls[-1]
    assert c["rgb"] is None and c["linear"] == vs.linear.ctypes.data and c["ids"] is None
    assert c["shard"] == (1, 2, 2) and c["chunk"] == 40 and c["mode"] == capi.RH_OFFSETS_NONE
    assert c["flags"] == (capi.RH_FLAG_SHADOW_SPLIT | capi.RH_FLAG_EXACT_BOXES | capi.RH_FLAG_NO_LIGHT_MAPS | capi.RH_FLAG_PROFILE)
    vs = rh.renderViews(_Job, cameras(1), rgb=True, linear=True)
    assert vs.pixels.shape == (1, 6, 10, 3) and vs.linear.shape == (1, 6, 10, 3)


def test_offsets_and_seeds(fake):
    off = np.zeros((60, 2, 2))
    rh.renderViews(_Job, cameras(2), spp=2, offsets=off)
    c = fake.calls[-1]
    assert c["mode"] == capi.RH_OFFSETS_F64 and c["offsets"] == off.ctypes.data and c["flags"] == 0
    rh.renderViews(_Job, cameras(2), spp=2, offsets=off.astype(np.float32))
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_F32
    tile = np.zeros((9, 2, 2))
    rh.renderViews(_Job, cameras(2), spp=2, offsets=tile, offset_tile=3)
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_TILED_F64 and fake.calls[-1]["tile"] == 3
    shard = np.zeros((4 * 10, 2, 2))  # shard 0 of 2 with bands of 2 rows: 4 rows
    rh.renderViews(_Job, cameras(2), spp=2, offsets=shard, shard_offsets=True, shard_count=2, band_height=2)
    assert fake.calls[-1]["flags"] == capi.RH_FLAG_SHARD_OFFSETS
    rh.renderViews(_Job, cameras(3), seeds=[7, 8, 2**64 - 1])
    c = fake.calls[-1]
    assert c["mode"] == capi.RH_OFFSETS_SPLITMIX64 and c["seeds"] == [7, 8, 2**64 - 1] and c["seed"] == 7
    rh.renderViews(_Job, cameras(2), seed=4, seeds=[1, 2])
    assert fake.calls[-1]["seed"] == 4 and fake.calls[-1]["seeds"] == [1, 2]


def test_an_empty_batch_reaches_the_library(fake):
    """n_views == 0 is the library's refusal (RH_ERR_ARG), not the wrapper's."""
    vs = rh.renderViews(_Job, [])
    assert vs.pixels.shape == (0, 6, 10, 3) and fake.calls[-1]["n_views"] == 0


def test_argument_checks(fake):
    for kw in (dict(rgb=False, linear=False), dict(seeds=[1]), dict(seeds=[1, 2, 3]), dict(seeds=[1, 2], offsets=np.zeros((60, 1, 2))),
               dict(spp=2, offsets=np.zeros((60, 1, 2))), dict(spp=2, offsets=np.zeros((60, 2, 2)), seed=3),
               dict(spp=2, offsets=np.zeros((60, 2, 2)), shard_offsets=True, shard_count=2, band_height=2),
               dict(shadow="sideways")):
        with pytest.raises((ValueError, KeyError)):
            rh.renderViews(_Job, cameras(2), **kw)
    assert not fake.calls  # rejected before the library is reached
