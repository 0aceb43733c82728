"""CPU tests of the feature buffers (rh_render_features / renderFeatures): the entry point is exported and bound, the
rh_features layout of the header equals the ctypes mirror, the call fails loudly without a device, and renderFeatures'
argument handling and output shapes with the library stubbed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["albedo", "normal", "depth", "hits", "stream_spp", "stream_base"]


def test_symbol_is_exported_and_bound():
    L = capi.lib()
    fn = L.rh_render_features
    assert fn.argtypes == capi.SIGNATURES["rh_render_features"][1]
    args = capi.SIGNATURES["rh_render_features"][1]
    assert len(args) == 6 and args[3]._type_ is capi.rh_features and args[5]._type_ is capi.rh_stats
    assert rh.renderFeatures is host.renderFeatures and rh.Features is host.Features


def test_rh_features_layout_matches_the_header():
    """sizeof / offsetof from a C program compiled against the header equal the ctypes mirror (40 bytes)."""
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){' + \
        'printf("size %zu\\n", sizeof(rh_features));' + "".join(f'printf("{f} %zu\\n", offsetof(rh_features, {f}));' for f in FIELDS) + \
        "return 0;}"
    exe = os.path.join(ROOT, "build", "abi_rh_features")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    out = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert out["size"] == C.sizeof(capi.rh_features) == 40
    for f in FIELDS:
        assert out[f] == getattr(capi.rh_features, f).offset, f


def test_without_a_device_the_call_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    o = capi.rh_render_opts()
    o.width, o.height, o.spp = 4, 4, 1
    ft = capi.rh_features()
    depth = np.empty((4, 4))
    ft.depth = depth.ctypes.data
    assert L.rh_render_features(None, None, C.byref(o), C.byref(ft), None, None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()


class _FakeLib:
    """Stands in for librayhs_b200.so: records the rh_render_features call and fills the outputs it was given."""

    def __init__(self):
        self.calls = []

    def rh_default_band_height(self, h, g):
        return h if g <= 1 else 4

    def rh_shard_rows(self, h, g, bh):
        n_bands = (h + bh - 1) // bh
        return (n_bands + g - 1) // g * bh

    def rh_render_features(self, scene, cam, opts, ft, ids, stats):
        o, f = opts._obj, ft._obj
        self.calls.append(dict(scene=scene, width=o.width, height=o.height, spp=o.spp, mode=o.offset_mode, tile=o.offset_tile,
                               offsets=o.offsets, shard=(o.shard_index, o.shard_count, o.band_height), flags=o.flags,
                               stream=(f.stream_spp, f.stream_base), ptrs=(f.albedo, f.normal, f.depth, f.hits), ids=ids))
        stats._obj.rays_primary = 7
        return 0


class _Job:
    class scene:
        device = "scene-handle"

    camera = capi.rh_camera()
    width, height, maxDepth = 10, 6, 3


@pytest.fixture
def fake(monkeypatch):
    L = _FakeLib()
    monkeypatch.setattr(host, "lib", lambda: L)
    return L


def test_shapes_and_dtypes(fake):
    fe = rh.renderFeatures(_Job, spp=3, seed=5, want_hit_ids=True)
    assert fe.albedo.shape == (6, 10, 3) and fe.normal.shape == (6, 10, 3) and fe.depth.shape == (6, 10) and fe.hits.shape == (6, 10)
    assert fe.albedo.dtype == np.float64 and fe.depth.dtype == np.float64 and fe.hits.dtype == np.uint32
    assert fe.hit_ids.shape == (6, 10, 3, 2) and fe.hit_ids.dtype == np.int32
    assert fe.stats["rays_primary"] == 7
    (c,) = fake.calls
    assert c["scene"] == "scene-handle" and (c["width"], c["height"], c["spp"]) == (10, 6, 3)
    assert c["mode"] == capi.RH_OFFSETS_SPLITMIX64 and c["flags"] == capi.RH_FLAG_HIT_IDS
    assert c["ptrs"] == tuple(a.ctypes.data for a in (fe.albedo, fe.normal, fe.depth, fe.hits)) and c["ids"] == fe.hit_ids.ctypes.data
    fe = rh.renderFeatures(_Job)
    assert fe.hit_ids is None and fake.calls[-1]["ids"] is None and fake.calls[-1]["mode"] == capi.RH_OFFSETS_NONE


def test_shards_give_the_compact_rows(fake):
    fe = rh.renderFeatures(_Job, shard_index=1, shard_count=2, band_height=2)
    assert fe.albedo.shape == (4, 10, 3) and fe.hits.shape == (4, 10)
    assert fake.calls[-1]["shard"] == (1, 2, 2)


def test_offsets_modes_and_checks(fake):
    off = rh.host.np.zeros((60, 2, 2))
    rh.renderFeatures(_Job, spp=2, offsets=off)
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_F64 and fake.calls[-1]["offsets"] == off.ctypes.data
    rh.renderFeatures(_Job, spp=2, offsets=off.astype(np.float32))
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_F32
    rh.renderFeatures(_Job, spp=2, offsets=np.zeros((9, 2, 2)), offset_tile=3)
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_TILED_F64 and fake.calls[-1]["tile"] == 3
    wide = np.zeros((60, 4, 2))
    rh.renderFeatures(_Job, spp=2, offsets=wide[:, 1:3])  # a strided slice of a stream is copied dense
    assert fake.calls[-1]["offsets"] != wide.ctypes.data
    rh.renderFeatures(_Job, spp=2, seed=1, stream_spp=8, stream_base=6, exact_boxes=True)
    assert fake.calls[-1]["stream"] == (8, 6) and fake.calls[-1]["flags"] == capi.RH_FLAG_EXACT_BOXES
    n = len(fake.calls)
    for kw in (dict(spp=2, offsets=np.zeros((60, 1, 2))), dict(spp=2, offsets=off, seed=3), dict(stream_spp=4),
               dict(stream_base=1), dict(spp=2, offsets=np.zeros((8, 2, 2)), offset_tile=3)):
        with pytest.raises(ValueError):
            rh.renderFeatures(_Job, **kw)
    assert len(fake.calls) == n  # rejected before the library is reached
