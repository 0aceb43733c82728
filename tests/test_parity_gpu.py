"""GPU parity tests: the sm_100a path, called through the C ABI, against the oracle on the same inputs."""
import numpy as np
import pytest

import rayhs_b200 as rh
from tests.util import SCENES, assert_oracle_exact, compare_images, load_scene, oracle_for, render_linear

pytestmark = pytest.mark.gpu

RES = {"cornellBox": (256, 256), "texture": (320, 180), "transform": (320, 180), "dragon_superlow": (256, 256),
       "dragon_low": (320, 180), "dragon_full": (320, 180), "outScene": (320, 180)}


@pytest.mark.parametrize("shadow", ["pooled", "split"])
@pytest.mark.parametrize("name", SCENES)
def test_one_sample_parity(name, shadow):
    """rayTrace (RayHs.hs:161-166): hit ids bit-exact, the image the oracle's channel by channel (linear colours within
    the sum order's roundings, bytes equal but at a straddled quantisation step), ray counts equal — with either
    schedule of the shadow walks (pooled per light in warp-local rounds, or one queued hit per lane with per-lane
    refill)."""
    sc = load_scene(name)
    w, h = RES[name]
    job = rh.renderingFromScene(sc, w, h)
    img = render_linear(job, shadow=shadow)
    assert img.stats["shadow_split"] == (1 if shadow == "split" else 0)
    ref = oracle_for(sc).render(sc.camera, w, h, sc.max_depth)
    ids_gpu = img.hit_ids.reshape(h, w, 2)
    ids_ref = ref["hit_ids"].reshape(h, w, 2)
    mism = np.any(ids_gpu != ids_ref, axis=-1)
    assert mism.sum() == 0, (name, int(mism.sum()), np.argwhere(mism)[:5], ids_gpu[mism][:5], ids_ref[mism][:5])
    straddled = assert_oracle_exact(img.pixels, img.linear, ref, name)
    st = img.stats
    got = (st["rays_primary"], st["rays_reflect"], st["rays_probe"], st["rays_exit"], st["rays_shadow"])
    want = tuple(ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow"))
    assert got == want, (name, got, want)
    print(name, shadow, "straddled channels", straddled, got)


@pytest.mark.parametrize("name", ["cornellBox", "dragon_low"])
def test_multi_sample_parity(name):
    """distributedRayTrace (RayHs.hs:190-195) with uploaded offsets, double and float: hit ids and the image as above."""
    sc = load_scene(name)
    w, h, spp = 160, 120, 4
    job = rh.renderingFromScene(sc, w, h)
    off = rh.sample_offsets(w * h, spp, seed=24)
    img = render_linear(job, spp=spp, offsets=off)
    ref = oracle_for(sc).render(sc.camera, w, h, sc.max_depth, spp=spp, offsets=off)
    assert np.array_equal(img.hit_ids, ref["hit_ids"])
    s64 = assert_oracle_exact(img.pixels, img.linear, ref, name)
    off32 = off.astype(np.float32)
    img32 = render_linear(job, spp=spp, offsets=off32)
    ref32 = oracle_for(sc).render(sc.camera, w, h, sc.max_depth, spp=spp, offsets=off32.astype(np.float64))
    assert np.array_equal(img32.hit_ids, ref32["hit_ids"])
    s32 = assert_oracle_exact(img32.pixels, img32.linear, ref32, name + " f32 offsets")
    print(name, "straddled channels", s64, s32)


def test_chunking_and_shards_give_identical_bytes():
    """Any chunk size and any shard count must give the same RGB8 bytes (SURVEY 8e parity gate)."""
    sc = load_scene("cornellBox")
    w, h = 200, 150
    job = rh.renderingFromScene(sc, w, h)
    base = rh.render(job).pixels
    small = rh.render(job, chunk_samples=w * 7).pixels
    assert np.array_equal(base, small)
    for G in (2, 4, 8):
        bh = 4
        parts = [rh.render(job, shard_index=g, shard_count=G, band_height=bh).pixels for g in range(G)]
        full = rh.assemble_bands(parts, h, bh)
        # transparent forks accumulate with atomics: allow the documented 1-LSB wobble, nothing more
        m = compare_images(full, base)
        assert m["maxdiff"] <= 1 and m["exact"] > 0.9999, (G, m)


@pytest.mark.parametrize("name", ["cornellBox", "dragon_full", "outScene"])
def test_float_cull_equals_exact_boxes(name):
    """The conservative float box cull must give the same hits and bytes as the reference's double slab
    test at every box (RH_FLAG_EXACT_BOXES), at a resolution large enough to matter."""
    sc = load_scene(name)
    w, h = 960, 540
    job = rh.renderingFromScene(sc, w, h)
    fast = rh.render(job, want_hit_ids=True)
    exact = rh.render(job, want_hit_ids=True, exact_boxes=True)
    assert np.array_equal(fast.hit_ids, exact.hit_ids)
    m = compare_images(fast.pixels, exact.pixels)
    assert m["maxdiff"] <= 1 and m["exact"] >= 0.99999, m
    for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert fast.stats[k] == exact.stats[k], k


@pytest.mark.parametrize("shadow", ["pooled", "split"])
@pytest.mark.parametrize("name", ["cornellBox", "texture", "transform", "dragon_full"])
def test_light_maps_change_no_byte_and_save_walks(name, shadow):
    """The per-light cube maps of nearest possible occluder distance and the lit-triangle flags (light_maps.cpp; the
    flags also for directional lights: transform.json has no other kind) only skip tree walks that could not find an
    occluder in front of the light: same bytes, same ray counts with RH_FLAG_NO_LIGHT_MAPS, under either shadow schedule — and on the dragon a third of the shadow rays' node visits are gone."""
    sc = load_scene(name)
    w, h = 960, 540
    job = rh.renderingFromScene(sc, w, h)
    on = rh.render(job, shadow=shadow, count=True)
    off = rh.render(job, shadow=shadow, count=True, light_maps=False)
    assert np.array_equal(on.pixels, off.pixels) or name == "cornellBox"
    m = compare_images(on.pixels, off.pixels)  # (cornellBox: transparent forks add with atomics, 1-LSB wobble)
    assert m["maxdiff"] <= 1 and m["exact"] >= 0.99999, m
    for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow", "rays_shadow_culled"):
        assert on.stats[k] == off.stats[k], k
    assert on.stats["shadow_node_visits"] <= off.stats["shadow_node_visits"]
    assert on.stats["shadow_tri_tests"] <= off.stats["shadow_tri_tests"]
    print(name, shadow, "shadow node visits", off.stats["shadow_node_visits"], "->", on.stats["shadow_node_visits"],
          "triangle tests", off.stats["shadow_tri_tests"], "->", on.stats["shadow_tri_tests"])
    if name == "dragon_full":
        assert on.stats["shadow_node_visits"] < 0.8 * off.stats["shadow_node_visits"]  # measured: 0.68


def test_shadow_schedule_is_chosen_per_scene_and_keeps_the_bytes():
    """Default flags: the first three large frames of a scene are timing frames (warm-up, pooled, per-lane refill) and the
    faster schedule is kept; every frame must carry the same bytes whichever schedule rendered it.  Small frames never
    take part in the timing: they render pooled."""
    sc = load_scene("dragon_low")
    small = rh.renderingFromScene(sc, 160, 90)
    assert [rh.render(small).stats["shadow_split"] for _ in range(3)] == [0, 0, 0]   # too small to time: pooled, not counted
    w, h = 2400, 1350   # > 2 Mi samples and enough walked pairs: counts as a timing frame
    job = rh.renderingFromScene(sc, w, h)
    frames = [rh.render(job) for _ in range(4)]
    assert [f.stats["shadow_split"] for f in frames[:3]] == [0, 0, 1]
    assert all(np.array_equal(frames[0].pixels, f.pixels) for f in frames[1:])
    assert rh.render(small).stats["shadow_split"] == frames[3].stats["shadow_split"]   # decided: small frames follow
    forced = rh.render(job, shadow="split")
    assert forced.stats["shadow_split"] == 1 and np.array_equal(forced.pixels, frames[0].pixels)


def test_offsets_regenerated_on_the_device_equal_the_uploaded_stream():
    """RH_OFFSETS_SPLITMIX64: the kernel regenerates the SplitMix64 stream from its seed (counter-based: value k needs no
    predecessor).  Same hit ids and bytes as uploading rh_sample_offsets_f64's output, also for a row shard."""
    sc = load_scene("dragon_low")
    w, h, spp = 200, 120, 5
    job = rh.renderingFromScene(sc, w, h)
    off = rh.sample_offsets(w * h, spp, seed=24)
    up = rh.render(job, spp=spp, offsets=off, want_hit_ids=True)
    gen = rh.render(job, spp=spp, seed=24, want_hit_ids=True)
    assert gen.stats["upload_bytes"] == 0 and up.stats["upload_bytes"] == off.nbytes
    assert np.array_equal(up.hit_ids, gen.hit_ids) and np.array_equal(up.pixels, gen.pixels)
    other = rh.render(job, spp=spp, seed=25)
    assert not np.array_equal(other.pixels, gen.pixels)
    a = rh.render(job, spp=spp, offsets=off, shard_index=1, shard_count=4, band_height=8).pixels
    b = rh.render(job, spp=spp, seed=24, shard_index=1, shard_count=4, band_height=8).pixels
    assert np.array_equal(a, b)


def test_peer_frame_stores_assemble_the_frame_without_a_gather():
    """RH_FLAG_PEER_FRAMES: the resolve kernel stores finished rows at their image position in every given full frame.
    On one GPU: four shards rendered one after the other into the same frame must rebuild the single-shard image —
    also for a width that is not a multiple of 4 (byte-store path) and a height the bands do not divide."""
    import torch

    sc = load_scene("cornellBox")
    for (w, h, bh) in ((200, 150, 4), (203, 149, 8)):
        job = rh.renderingFromScene(sc, w, h)
        base = rh.render(job, shadow="pooled").pixels
        full = torch.full((h, w, 3), 7, dtype=torch.uint8, device="cuda")
        for g in range(4):
            rh.render_device(job, None, shard_index=g, shard_count=4, band_height=bh, peer_frames=[full.data_ptr()], shadow="pooled")
        d = np.abs(full.cpu().numpy().astype(np.int32) - base.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-4, (w, h, int(d.max()))   # Transparent forks: atomic order


def test_multi_gpu_entry_from_one_process():
    """rh_multi_render (what a single-process host calls): on however many GPUs this box has (1 on the test box; the
    2- and 8-GPU runs are scripts/gpu_multi_check.py), the frame must equal rh_render's."""
    import torch

    n = min(torch.cuda.device_count(), 8)
    sc = load_scene("cornellBox")
    w, h, spp = 203, 149, 3
    job = rh.renderingFromScene(sc, w, h)
    off = rh.sample_offsets(w * h, spp, seed=24)
    base = rh.render(job, spp=spp, offsets=off)
    try:
        multi = rh.render_multi(job, n, spp=spp, offsets=off)
        seeded = rh.render_multi(job, n, spp=spp, seed=24)
    finally:
        rh.multi_shutdown([sc])
    for img in (multi, seeded):
        d = np.abs(img.pixels.astype(np.int32) - base.pixels.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-4   # Transparent forks: atomic order
    for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert multi.stats[k] == base.stats[k], k


def test_cpp_cli_writes_the_oracles_ppm(tmp_path):
    """`rayhs -oFILE scene.json` (csrc/rayhs_main.cpp, the C++ stand-in for RayHs.hs:204-234) on a self-contained scene in
    the reference's JSON schema: the P3 file must carry the oracle's bytes in writePPM's format (Image.hs:60-75);
    RAYHS_GPUS routes the same run through rh_multi_render."""
    import os
    import subprocess

    import torch

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    scene = os.path.join(root, "tests", "golden", "cli_scene.json")
    job = rh.buildRendering(scene)
    ref = oracle_for(job.scene).render(job.scene.camera, job.width, job.height, job.maxDepth)["rgb_u8"]
    for gpus in (1, min(torch.cuda.device_count(), 8)):
        out = tmp_path / f"out{gpus}.ppm"
        env = dict(os.environ, RAYHS_GPUS=str(gpus))
        r = subprocess.run([os.path.join(root, "rayhs_b200", "rayhs"), f"-o{out}", scene], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout.splitlines() == [f"Loading scene from {scene}...", "Rendering...", f"Done! Output written to {out}"]
        text = out.read_text()
        head, body = text.split("\n255\n", 1)
        assert head == f"P3\n{job.width} {job.height}" and not text.endswith("\n")
        rows = body.split("\n")
        assert len(rows) == job.height and all(row.endswith("  ") for row in rows)
        got = np.array([[int(x) for x in row.split()] for row in rows], dtype=np.int32).reshape(job.height, job.width, 3)
        d = np.abs(got - ref.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-4, (gpus, int(d.max()))   # Transparent sphere: atomic order
