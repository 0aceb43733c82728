"""GPU tests of progressive rendering (rh_render_accumulate / Accumulator / progressiveRayTrace): every call equals the
one-shot render of all samples so far, byte for byte; the linear colours equal the oracle's; the SplitMix64 stream
continues across calls; chunking, shards, device buffers and the validation flags keep the bytes; an overflow retry
counts no sample twice; the accumulator's life cycle; argument errors; and a bench-sized frame."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host
from tests.test_trace_rays_gpu import growth_scene, has_transparent
from tests.util import ATOL, GOLDEN, RTOL, SCENES, assert_parity, load_scene, to_int_c

pytestmark = pytest.mark.gpu

W, H, SPP, BATCHES = 64, 48, 8, (1, 3, 4)  # odd and even batches: both fold paths of the sink
PLAIN = "dragon_low"  # no Transparent material: renders are deterministic to the byte


def job_of(sc, w=W, h=H, max_depth=None):
    return rh.Rendering(sc, sc.camera, w, h, sc.max_depth if max_depth is None else max_depth)


def part(off, a, b):
    return np.ascontiguousarray(off[:, a:b])


def same_bytes(got, want, forks, what):
    if forks:  # Transparent forks add into one accumulator with atomics: the 1-LSB wobble
        assert_parity(got, want, what)
    else:
        assert np.array_equal(got, want), (what, np.argwhere((got != want).any(axis=-1))[:5])


@pytest.mark.parametrize("name", SCENES)
def test_every_call_equals_the_one_shot_render(name):
    sc = load_scene(name)
    job, forks = job_of(sc), has_transparent(sc)
    off = rh.sample_offsets(W * H, SPP, seed=7)
    acc = rh.Accumulator(job)
    n = 0
    for b in BATCHES:
        img = acc.add(b, offsets=part(off, n, n + b), want_hit_ids=True)
        ref = rh.render(job, spp=n + b, offsets=part(off, 0, n + b), want_hit_ids=True)
        assert img.pixels.shape == (H, W, 3) and img.linear.shape == (H, W, 3) and img.hit_ids.shape == (H, W, b, 2)
        assert np.array_equal(img.hit_ids, ref.hit_ids[:, :, n:n + b]), (name, n)
        same_bytes(img.pixels, ref.pixels, forks, (name, n + b))
        assert np.array_equal(to_int_c(img.linear), img.pixels), (name, n + b)
        assert img.stats["rays_primary"] == W * H * b
        n += b
        assert acc.samples == n
    acc.close()


@pytest.mark.parametrize("name", SCENES)
def test_linear_colours_equal_the_oracle(name):
    from oracle.orc import OracleScene

    sc = load_scene(name)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=11)
    orc = OracleScene(sc.raw)
    acc = rh.Accumulator(job)
    n = 0
    for b in (3, 5):
        img = acc.add(b, offsets=part(off, n, n + b), exact_boxes=True)
        n += b
        want = orc.render(sc.camera, W, H, sc.max_depth, spp=n, offsets=part(off, 0, n), want_ids=False)["rgb_f64"]
        ok = np.isclose(img.linear, want, rtol=RTOL, atol=ATOL, equal_nan=True).all(axis=-1)
        assert ok.all(), (name, n, np.argwhere(~ok)[:5])
        assert np.array_equal(to_int_c(img.linear), img.pixels), (name, n)
    assert (img.linear > 0).any(), (name, "the view is black")


def test_splitmix64_stream_continues_across_calls():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    seed = 0x5EED
    stream = rh.sample_offsets(W * H, SPP, seed=seed)
    acc = rh.Accumulator(job, stream_spp=SPP)
    first = acc.add(3, seed=seed, want_hit_ids=True)
    ref3 = rh.render(job, spp=3, offsets=part(stream, 0, 3), want_hit_ids=True)
    assert np.array_equal(first.pixels, ref3.pixels) and np.array_equal(first.hit_ids, ref3.hit_ids)
    with pytest.raises(capi.RayHsError) as e:  # 3 + 6 > stream_spp
        acc.add(6, seed=seed)
    assert e.value.code == capi.RH_ERR_ARG and "past the end of the stream" in str(e.value)
    assert acc.samples == 3
    last = acc.add(5, seed=seed)
    ref = rh.render(job, spp=SPP, seed=seed)
    assert np.array_equal(last.pixels, ref.pixels)
    assert np.array_equal(ref.pixels, rh.render(job, spp=SPP, offsets=stream).pixels)
    with pytest.raises(capi.RayHsError) as e:  # the stream is used up
        acc.add(1, seed=seed)
    assert e.value.code == capi.RH_ERR_ARG
    # an accumulator without a stream refuses SplitMix64 calls
    with pytest.raises(capi.RayHsError) as e:
        rh.Accumulator(job).add(1, seed=seed)
    assert e.value.code == capi.RH_ERR_ARG and "stream_spp" in str(e.value)


def test_progressive_ray_trace_converges_to_the_reference_frame():
    sc = load_scene(PLAIN)
    job = job_of(sc, 96, 64)
    images = list(rh.progressiveRayTrace(job, 64, 16))
    assert len(images) == 4
    want = rh.distributedRayTrace(job, 64)
    assert np.array_equal(images[-1].pixels, want.pixels)
    assert np.array_equal(images[0].pixels, rh.render(job, spp=16, offsets=part(rh.sample_offsets(96 * 64, 64, 24), 0, 16)).pixels)
    tail = list(rh.progressiveRayTrace(job, 10, 4))  # 4 + 4 + 2
    assert len(tail) == 3 and np.array_equal(tail[-1].pixels, rh.distributedRayTrace(job, 10).pixels)


@pytest.mark.parametrize("name", [PLAIN, "cornellBox"])
def test_chunking_keeps_the_bytes(name):
    sc = load_scene(name)
    job, forks = job_of(sc), has_transparent(sc)
    off = rh.sample_offsets(W * H, SPP, seed=3)
    base, chunked = rh.Accumulator(job), rh.Accumulator(job)
    n = 0
    for b in BATCHES:
        a = base.add(b, offsets=part(off, n, n + b))
        c = chunked.add(b, offsets=part(off, n, n + b), chunk_samples=W * b * 3 + 5)  # 3 rows per chunk
        assert c.stats["chunks"] >= H // 3, c.stats["chunks"]
        same_bytes(c.pixels, a.pixels, forks, (name, "chunks", n))
        if not forks:
            assert c.linear.tobytes() == a.linear.tobytes()
        n += b


@pytest.mark.parametrize("shards,band_height", [(2, 1), (2, 5), (3, 1), (3, 5)])
def test_shards_assemble_to_the_whole_frame(shards, band_height):
    sc = load_scene(PLAIN)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=5)
    whole = rh.Accumulator(job)
    accs = [rh.Accumulator(job, shard_index=g, shard_count=shards, band_height=band_height) for g in range(shards)]
    rows = capi.lib().rh_shard_rows(H, shards, band_height)
    n = 0
    for b in BATCHES:
        want = whole.add(b, offsets=part(off, n, n + b))
        parts = [a.add(b, offsets=part(off, n, n + b)) for a in accs]
        assert all(p.pixels.shape == (rows, W, 3) for p in parts)
        assert np.array_equal(rh.assemble_bands([p.pixels for p in parts], H, band_height), want.pixels), (shards, band_height, n)
        for g, p in enumerate(parts):
            rmap = np.array(rh.shard_global_rows(H, g, shards, band_height))
            real = rmap >= 0
            assert p.linear[real].tobytes() == want.linear[rmap[real]].tobytes()
        n += b
    # a shard's accumulator refuses another shard's opts
    o = host._opts(job, 1, capi.RH_OFFSETS_NONE, None, 0, 1, shards, band_height, 0, 0)
    rgb = np.empty((rows, W, 3), dtype=np.uint8)
    assert capi.lib().rh_render_accumulate(sc.device, C.byref(job.camera), C.byref(o), accs[0]._h, rgb.ctypes.data, None,
                                           None, None) == capi.RH_ERR_ARG
    assert b"differ from the accumulator" in capi.lib().rh_last_error()


def test_device_buffers_equal_the_host_path():
    import torch

    sc = load_scene(PLAIN)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=9)
    hostacc, devacc, mixed = rh.Accumulator(job), rh.Accumulator(job, device=True), rh.Accumulator(job, device=True)
    n = 0
    for b in BATCHES:
        h = hostacc.add(b, offsets=part(off, n, n + b), want_hit_ids=True)
        d = devacc.add(b, offsets=torch.from_numpy(part(off, n, n + b)).cuda(), want_hit_ids=True)
        m = mixed.add(b, offsets=part(off, n, n + b))  # host offsets, device outputs
        assert d.pixels.is_cuda and d.linear.is_cuda and d.hit_ids.is_cuda and d.linear.dtype == torch.float64
        assert np.array_equal(d.pixels.cpu().numpy(), h.pixels) and np.array_equal(m.pixels.cpu().numpy(), h.pixels)
        assert d.linear.cpu().numpy().tobytes() == h.linear.tobytes() == m.linear.cpu().numpy().tobytes()
        assert np.array_equal(d.hit_ids.cpu().numpy(), h.hit_ids)
        n += b


def test_validation_flags_mixed_across_calls_keep_the_bytes():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=13)
    plain, mixed = rh.Accumulator(job), rh.Accumulator(job)
    n = 0
    for b, kw in zip((1, 2, 2, 3), (dict(shadow="split"), dict(exact_boxes=True), dict(light_maps=False), dict(shadow="pooled"))):
        a = plain.add(b, offsets=part(off, n, n + b))
        c = mixed.add(b, offsets=part(off, n, n + b), **kw)
        assert np.array_equal(c.pixels, a.pixels), kw
        assert c.linear.tobytes() == a.linear.tobytes(), kw
        n += b
    assert np.array_equal(a.pixels, rh.render(job, spp=SPP, offsets=off).pixels)


def test_queue_growth_retry_counts_no_sample_twice():
    """The overflowing call is one that continues existing sums (N_before > 0): a sink that added into the sums it reads
    would add the retried frame's samples twice there."""
    from oracle.orc import OracleScene

    sc = growth_scene()  # Transparent spheres in a box of mirrors: many secondary rays per sample
    w, h = 16, 256
    job = rh.Rendering(sc, sc.camera, w, h, 8)
    off = rh.sample_offsets(w * h, 4, seed=21)
    acc = rh.Accumulator(job)
    first = acc.add(1, offsets=part(off, 0, 1))
    # One-row chunks need far larger queues per sample than the first call's one chunk (every warp that produces rays
    # leaves a slab open): this call overflows at the factor the first call left and runs its frame again.
    last = acc.add(3, offsets=part(off, 1, 4), chunk_samples=3 * w)
    assert last.stats["chunks"] == h and last.stats["queue_factor"] > first.stats["queue_factor"], (first.stats, last.stats)
    assert acc.samples == 4
    want = OracleScene(sc.raw).render(sc.camera, w, h, 8, spp=4, offsets=off, want_ids=False)
    ok = np.isclose(last.linear, want["rgb_f64"], rtol=RTOL, atol=ATOL, equal_nan=True).all(axis=-1)
    assert ok.all(), np.argwhere(~ok)[:5]
    assert (want["rgb_f64"] > 0).any()
    assert_parity(last.pixels, rh.render(job, spp=4, offsets=off).pixels)


def test_offsets_may_be_views_of_one_stream():
    """A slice of one [pixels, S, 2] stream is not contiguous; add() reads the values of the view, not its base array."""
    import torch

    sc = load_scene(PLAIN)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=23)
    views, host_ref = rh.Accumulator(job), rh.Accumulator(job)
    dev = rh.Accumulator(job, device=True)
    off_dev = torch.from_numpy(off).cuda()
    n = 0
    for b in BATCHES:
        assert b == 1 or not off[:, n:n + b].flags["C_CONTIGUOUS"]
        a = views.add(b, offsets=off[:, n:n + b])
        r = host_ref.add(b, offsets=part(off, n, n + b))
        d = dev.add(b, offsets=off_dev[:, n:n + b])
        assert np.array_equal(a.pixels, r.pixels) and a.linear.tobytes() == r.linear.tobytes(), n
        assert np.array_equal(d.pixels.cpu().numpy(), r.pixels), n
        n += b
    assert np.array_equal(a.pixels, rh.render(job, spp=SPP, offsets=off).pixels)


def test_reset_output_less_calls_and_failed_calls():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=17)
    fresh = rh.Accumulator(job).add(2, offsets=part(off, 3, 5))
    acc = rh.Accumulator(job)
    acc.add(3, offsets=part(off, 0, 3))
    acc.reset()
    assert acc.samples == 0
    again = acc.add(2, offsets=part(off, 3, 5))
    assert np.array_equal(again.pixels, fresh.pixels) and again.linear.tobytes() == fresh.linear.tobytes()
    # a call without outputs only accumulates
    quiet, loud = rh.Accumulator(job), rh.Accumulator(job)
    q = quiet.add(3, offsets=part(off, 0, 3), rgb=False, linear=False)
    assert q.pixels is None and q.linear is None
    loud.add(3, offsets=part(off, 0, 3))
    a, b = quiet.add(5, offsets=part(off, 3, 8)), loud.add(5, offsets=part(off, 3, 8))
    assert np.array_equal(a.pixels, b.pixels) and a.linear.tobytes() == b.linear.tobytes()
    assert np.array_equal(a.pixels, rh.render(job, spp=SPP, offsets=off).pixels)
    # failed calls (argument errors of every kind) leave the sums and the count alone
    acc = rh.Accumulator(job)
    acc.add(3, offsets=part(off, 0, 3))
    L = capi.lib()
    o = host._opts(job, 5, capi.RH_OFFSETS_F64, part(off, 3, 8).ctypes.data, 0, 0, 1, H, 0, capi.RH_FLAG_HIT_IDS)
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    assert L.rh_render_accumulate(sc.device, C.byref(job.camera), C.byref(o), acc._h, rgb.ctypes.data, None, None, None) == capi.RH_ERR_ARG
    o.flags, o.max_depth = 0, job.maxDepth + 1
    assert L.rh_render_accumulate(sc.device, C.byref(job.camera), C.byref(o), acc._h, rgb.ctypes.data, None, None, None) == capi.RH_ERR_ARG
    o.max_depth, o.offset_mode = job.maxDepth, capi.RH_OFFSETS_SPLITMIX64
    assert L.rh_render_accumulate(sc.device, C.byref(job.camera), C.byref(o), acc._h, rgb.ctypes.data, None, None, None) == capi.RH_ERR_ARG
    last = acc.add(5, offsets=part(off, 3, 8))
    assert acc.samples == SPP and np.array_equal(last.pixels, a.pixels) and last.linear.tobytes() == a.linear.tobytes()


def test_view_is_fixed_between_resets_and_renders_are_unaffected():
    sc, other = load_scene(PLAIN), load_scene("dragon_superlow")
    job = job_of(sc)
    off = rh.sample_offsets(W * H, SPP, seed=19)
    before = rh.render(job, spp=SPP, offsets=off)
    acc = rh.Accumulator(job)
    acc.add(2, offsets=part(off, 0, 2))
    L = capi.lib()
    rgb = np.empty((H, W, 3), dtype=np.uint8)

    def call(scene=sc, camera=job.camera, max_depth=job.maxDepth):
        o = host._opts(job, 1, capi.RH_OFFSETS_F64, part(off, 2, 3).ctypes.data, 0, 0, 1, H, 0, 0)
        o.max_depth = max_depth
        return L.rh_render_accumulate(scene.device, C.byref(camera), C.byref(o), acc._h, rgb.ctypes.data, None, None, None)

    cam = capi.rh_camera.from_buffer_copy(job.camera)
    cam.position[0] += 1e-9
    for kw in (dict(camera=cam), dict(scene=other), dict(max_depth=job.maxDepth - 1)):
        assert call(**kw) == capi.RH_ERR_ARG, kw
        assert b"rh_accum_reset" in L.rh_last_error(), kw
    assert acc.samples == 2
    assert call() == capi.RH_OK
    after = rh.render(job, spp=SPP, offsets=off)
    assert np.array_equal(before.pixels, after.pixels)
    for k in ("queue_factor", "rays_reflect", "rays_shadow", "chunks"):
        assert before.stats[k] == after.stats[k], k
    acc.reset()  # after a reset another view is fine
    other_job = job_of(other)
    o = host._opts(other_job, 1, capi.RH_OFFSETS_NONE, None, 0, 0, 1, H, 0, 0)
    assert L.rh_render_accumulate(other.device, C.byref(other.camera), C.byref(o), acc._h, rgb.ctypes.data, None, None, None) == capi.RH_OK
    assert np.array_equal(rgb, rh.render(other_job).pixels)


def test_argument_errors():
    import torch

    sc = load_scene(PLAIN)
    job = job_of(sc)
    L = capi.lib()
    acc = rh.Accumulator(job, stream_spp=4)
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    lin = np.empty((H, W, 3))
    ids = np.empty((H, W, 1, 2), dtype=np.int32)

    def call(scene=True, camera=True, opts=True, a=True, r=rgb.ctypes.data, li=None, i=None, **kw):
        o = host._opts(job, 1, capi.RH_OFFSETS_NONE, None, 0, 0, 1, H, 0, 0)
        for k, v in kw.items():
            setattr(o, k, v)
        rc = L.rh_render_accumulate(sc.device if scene else None, C.byref(job.camera) if camera else None,
                                    C.byref(o) if opts else None, acc._h if a else None, r, li, i, None)
        return rc, L.rh_last_error().decode()

    assert call()[0] == capi.RH_OK
    assert call(r=None)[0] == capi.RH_OK  # no output: accumulate only
    seed = C.c_uint64(1)
    cases = [
        (dict(flags=capi.RH_FLAG_PEER_FRAMES), "RH_FLAG_PEER_FRAMES"),
        (dict(scene=False), "null argument"), (dict(camera=False), "null argument"), (dict(opts=False), "null argument"),
        (dict(a=False), "null argument"),
        (dict(spp=0), "bad width/height/spp/max_depth"), (dict(spp=-3), "bad width/height/spp/max_depth"),
        (dict(max_depth=31), "bad width/height/spp/max_depth"),
        (dict(width=W + 1), "differ from the accumulator"), (dict(height=H - 1), "differ from the accumulator"),
        (dict(shard_count=2), "differ from the accumulator"), (dict(band_height=5), "differ from the accumulator"),
        (dict(shard_index=1), "shard_index out of range"),
        (dict(offset_mode=9), "bad offset_mode"), (dict(offset_mode=capi.RH_OFFSETS_F64), "offsets is null"),
        (dict(flags=capi.RH_FLAG_HIT_IDS), "RH_FLAG_HIT_IDS without hit_ids_out"),
        (dict(offset_mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seed), flags=capi.RH_FLAG_DEVICE_OFFSETS),
         "takes a host pointer to the seed"),
        (dict(offset_mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seed), spp=5), "past the end of the stream"),
        (dict(flags=capi.RH_FLAG_DEVICE_OUT), "not device memory"),
        (dict(flags=capi.RH_FLAG_DEVICE_OUT, r=None, li=lin.ctypes.data), "not device memory"),
        (dict(flags=capi.RH_FLAG_DEVICE_OUT | capi.RH_FLAG_HIT_IDS, r=None, i=ids.ctypes.data), "not device memory"),
    ]
    for kw, msg in cases:
        rc, err = call(**kw)
        assert rc == capi.RH_ERR_ARG and msg in err and err.startswith("rh_render_accumulate"), (kw, rc, err)
    d = torch.empty(H * W * 3 + 1, dtype=torch.float64, device="cuda")
    rc, err = call(flags=capi.RH_FLAG_DEVICE_OUT, r=None, li=d.data_ptr() + 4)
    assert rc == capi.RH_ERR_ARG and "8-byte aligned" in err
    assert call(flags=capi.RH_FLAG_DEVICE_OUT, r=None, li=d.data_ptr() + 8)[0] == capi.RH_OK
    # three calls succeeded: one more sample of the 4-sample stream is left
    assert call(offset_mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seed), spp=2)[0] == capi.RH_ERR_ARG
    assert call(offset_mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seed))[0] == capi.RH_OK
    assert call(offset_mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seed))[0] == capi.RH_ERR_ARG
    # create
    h = C.c_void_p()
    for args, msg in (((0, H, 0, 1, 0, 0), "bad width/height"), ((W, -1, 0, 1, 0, 0), "bad width/height"),
                      ((W, H, 2, 2, 0, 0), "shard_index out of range"), ((W, H, -1, 1, 0, 0), "shard_index out of range")):
        assert L.rh_accum_create(*args, C.byref(h)) == capi.RH_ERR_ARG and msg in L.rh_last_error().decode(), args
    assert L.rh_accum_create(W, H, 0, 1, 0, 0, None) == capi.RH_ERR_ARG
    assert L.rh_accum_reset(None) == capi.RH_ERR_ARG


def test_another_device_context_and_destroy_after_shutdown():
    """An accumulator of a context that was shut down is refused by the next context, and can still be destroyed.  In a
    process of its own: the shutdown would orphan this process's scenes."""
    code = f"""
import ctypes as C, sys
sys.path.insert(0, {os.path.dirname(os.path.dirname(os.path.abspath(__file__)))!r})
import numpy as np
import rayhs_b200 as rh
from rayhs_b200 import capi, host
L = capi.lib()
rh.init(0)
acc = C.c_void_p()
capi.check(L.rh_accum_create(16, 8, 0, 1, 0, 0, C.byref(acc)))
rh.shutdown()
rh.init(0)
sc = rh.Scene.from_pack({os.path.join(GOLDEN, PLAIN + ".pack")!r})
job = rh.Rendering(sc, sc.camera, 16, 8, sc.max_depth)
o = host._opts(job, 1, capi.RH_OFFSETS_NONE, None, 0, 0, 1, 8, 0, 0)
rgb = np.empty((8, 16, 3), dtype=np.uint8)
rc = L.rh_render_accumulate(sc.device, C.byref(sc.camera), C.byref(o), acc, rgb.ctypes.data, None, None, None)
assert rc == capi.RH_ERR_ARG and b"another device context" in L.rh_last_error(), (rc, L.rh_last_error())
L.rh_accum_destroy(acc)
a = rh.Accumulator(job)
assert np.array_equal(a.add(1).pixels, rh.render(job).pixels)
print("ok")
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


def test_bench_sized_frame_equals_the_one_shot_render():
    import torch

    sc = load_scene("dragon_full")
    job = job_of(sc, 3840, 2160)
    acc = rh.Accumulator(job, stream_spp=16, device=True)
    for _ in range(4):
        img = acc.add(4, seed=24)
    ref = torch.empty((2160, 3840, 3), dtype=torch.uint8, device="cuda")
    rh.render_device(job, ref, spp=16, seed=24)
    assert torch.equal(img.pixels, ref)
    assert torch.equal(torch.from_numpy(to_int_c(img.linear.cpu().numpy())).cuda(), img.pixels)
