"""GPU tests of the round-2 ABI additions."""
import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi
from tests.util import load_scene

pytestmark = pytest.mark.gpu


def test_shard_compact_offsets_equal_the_full_frame_stream():
    """RH_FLAG_SHARD_OFFSETS: a shard that is handed only its own rows of the offset stream (shard-compact order, host
    or device memory) renders the bytes it renders from the full-frame stream."""
    import torch

    sc = load_scene("dragon_low")
    w, h, spp, G, bh = 200, 120, 4, 4, 8
    job = rh.renderingFromScene(sc, w, h)
    off = rh.sample_offsets(w * h, spp, 24)
    L = capi.lib()
    rows = L.rh_shard_rows(h, G, bh)
    for g in (0, 3):
        want = rh.render(job, spp=spp, offsets=off, shard_index=g, shard_count=G, band_height=bh).pixels
        compact = np.zeros((rows * w, spp, 2), dtype=np.float64)
        for lb in range(rows // bh):
            grow = (lb * G + g) * bh
            n = max(0, min(bh, h - grow))
            if n:
                L.rh_sample_offsets_f64_at(24, grow * w, n * w, spp, compact[lb * bh * w:].ctypes.data)
        out = torch.empty((rows, w, 3), dtype=torch.uint8, device="cuda")
        host = torch.from_numpy(compact).pin_memory()
        rh.render_device(job, out, spp=spp, offsets_dev=host, shard_index=g, shard_count=G, band_height=bh, shard_offsets=True)
        assert np.array_equal(out.cpu().numpy(), want)
        rh.render_device(job, out, spp=spp, offsets_dev=host.cuda(), shard_index=g, shard_count=G, band_height=bh, shard_offsets=True)
        assert np.array_equal(out.cpu().numpy(), want)
        rh.render_device(job, out, spp=spp, seed=24, shard_index=g, shard_count=G, band_height=bh)
        assert np.array_equal(out.cpu().numpy(), want)


def test_a_shard_of_single_row_bands_picks_arbitrary_rows():
    """bench.py's parity sample: shard r0 of H / 16 single-row bands = rows r0, r0 + H/16, ...; with hit ids on the device."""
    import torch

    sc = load_scene("cornellBox")
    w, h, spp = 96, 64, 2
    job = rh.renderingFromScene(sc, w, h)
    full = rh.render(job, spp=spp, seed=7, want_hit_ids=True)
    step, r0 = h // 16, 3
    rows = capi.lib().rh_shard_rows(h, step, 1)
    rgb = torch.empty((rows, w, 3), dtype=torch.uint8, device="cuda")
    ids = torch.empty((rows * w * spp, 2), dtype=torch.int32, device="cuda")
    rh.render_device(job, rgb, spp=spp, seed=7, shard_index=r0, shard_count=step, band_height=1, hit_ids_dev=ids)
    ys = np.arange(r0, h, step)
    assert np.array_equal(rgb.cpu().numpy()[:len(ys)], full.pixels[ys])
    assert np.array_equal(ids.cpu().numpy().reshape(rows, w, spp, 2)[:len(ys)], full.hit_ids.reshape(h, w, spp, 2)[ys])


# hand-built scenes at the limits of the packed tables (tests/test_limits_gpu.py): 42 maps at 512^2 cells per face, 48
# at 256^2, and 12 lights x 8 meshes with directional lights first (lit bit 11 and map index 11 * 8 + 7 in use)
LIMIT_SCENES = {"map_res_42": lambda L: L.map_res_scene(7), "map_res_48": lambda L: L.map_res_scene(8),
                "packed_12x8": lambda L: L.packed_scene(12)}


@pytest.mark.parametrize("name", ["dragon_low", "dragon_full", "transform", "cornellBox"] + list(LIMIT_SCENES))
def test_device_built_light_tables_equal_the_host_built_ones(name, monkeypatch):
    """rh_scene_create builds the cube maps and the lit-triangle flags with CUDA kernels (setup_kernels.cu); the host
    builders of light_maps.cpp (RAYHS_B200_SETUP=host) run the same geometry code (light_geom.h) and must produce the
    same tables bit for bit — the host builders are what tests/test_light_maps.py checks against brute force."""
    import os

    from tests import test_limits_gpu
    from tests.util import GOLDEN, RawScene

    def make():
        if name in LIMIT_SCENES:
            return RawScene(*LIMIT_SCENES[name](test_limits_gpu), camera=test_limits_gpu.CAMERA)
        return rh.Scene.from_pack(os.path.join(GOLDEN, name + ".pack"))

    monkeypatch.delenv("RAYHS_B200_SETUP", raising=False)
    dev = make()
    t_dev = rh.Scene.light_tables(dev)
    monkeypatch.setenv("RAYHS_B200_SETUP", "host")
    host = make()
    t_host = rh.Scene.light_tables(host)
    assert t_dev["res"] == t_host["res"]
    assert np.array_equal(t_dev["index"], t_host["index"])
    assert t_dev["maps"].shape == t_host["maps"].shape
    assert np.array_equal(t_dev["maps"].view(np.uint32), t_host["maps"].view(np.uint32))
    assert (t_dev["lit"] is None) == (t_host["lit"] is None)
    if t_dev["lit"] is not None:
        assert np.array_equal(t_dev["lit"], t_host["lit"])
        if name.startswith("dragon"):
            assert (t_dev["lit"] & 0x0fff).astype(bool).mean() > 0.3   # the flags are not trivially empty
    if name in LIMIT_SCENES:   # the tables are not trivially empty either
        assert len(t_dev["maps"]) and t_dev["lit"] is not None and (t_dev["lit"] & 0x0fff).any(), name
    print(name, "res", t_dev["res"], "maps", len(t_dev["maps"]))
    dev.close()
    host.close()
