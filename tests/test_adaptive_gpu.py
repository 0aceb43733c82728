"""GPU tests of adaptive sampling (rh_render_adaptive / AdaptiveAccumulator / adaptiveRayTrace): a pixel that ends with
n samples has exactly the bytes and linear colour of an n-sample progressive render; the state (counts, sums, sums of
squares) and the selection equal their numpy restatement bit for bit; the behaviour at the thresholds' extremes;
chunking, shards, device buffers and validation flags keep the state; the scene's learned state is left alone; failed
calls change nothing and an overflow retry counts no sample twice; reset."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host
from tests.adaptive_rule import active_pixels, fold
from tests.test_trace_rays_gpu import growth_scene, has_transparent
from tests.util import SCENES, assert_parity, load_scene, to_int_c

pytestmark = pytest.mark.gpu

W, H = 64, 48
PLAIN = "dragon_low"  # no Transparent material: renders are deterministic to the byte
STREAM, SEED = 12, 0xADA
BATCHES = (2, 3, 1, 2, 4)  # odd and even: both fold paths of the sink
THRESHOLD = 0.02


def job_of(sc, w=W, h=H, max_depth=None):
    return rh.Rendering(sc, sc.camera, w, h, sc.max_depth if max_depth is None else max_depth)


def sample_colours(job, n, stream_spp=STREAM, seed=SEED):
    """float64 [n, H, W, 3]: the colour of sample s of every pixel of the stream (the linear image of a 1-sample call)."""
    off = rh.sample_offsets(job.width * job.height, stream_spp, seed=seed)
    out = []
    for s in range(n):
        acc = rh.Accumulator(job)
        out.append(acc.add(1, offsets=np.ascontiguousarray(off[:, s:s + 1]), rgb=False).linear)
        acc.close()
    return np.stack(out)


def expected_state(cols, counts):
    """S and Q of each pixel folded over its first counts[p] sample colours, in sample order."""
    S = np.zeros(cols.shape[1:])
    Q = np.zeros(cols.shape[1:])
    for n in np.unique(counts):
        s, q = fold(cols[:n])
        m = counts == n
        S[m], Q[m] = s[m], q[m]
    return S, Q


def run(ad, batches=BATCHES, threshold=THRESHOLD, min_spp=2, seed=SEED, **kw):
    img = None
    for b in batches:
        img = ad.add(b, seed, threshold, min_spp=min_spp, **kw)
    return img


@pytest.mark.parametrize("name", SCENES)
def test_each_pixel_equals_the_progressive_render_of_its_count(name):
    sc = load_scene(name)
    job, forks = job_of(sc), has_transparent(sc)
    ad = rh.AdaptiveAccumulator(job, STREAM)
    img = run(ad)
    counts, _, _ = ad.state()
    assert img.pixels.shape == (H, W, 3) and img.linear.shape == (H, W, 3)
    assert np.array_equal(to_int_c(img.linear), img.pixels)
    assert len(np.unique(counts)) >= 2 or forks, (name, np.unique(counts))  # the threshold splits the pixels
    want_px, want_lin = np.zeros_like(img.pixels), np.zeros_like(img.linear)
    for n in np.unique(counts):
        ref = rh.Accumulator(job, STREAM).add(int(n), seed=SEED)
        m = counts == n
        want_px[m], want_lin[m] = ref.pixels[m], ref.linear[m]
        if not forks:
            assert np.array_equal(img.pixels[m], ref.pixels[m]), (name, n)
            assert img.linear[m].tobytes() == ref.linear[m].tobytes(), (name, n)
    if forks:  # Transparent forks add into one accumulator with atomics: the 1-LSB wobble
        assert_parity(img.pixels, want_px, name)
    ad.close()


def test_state_and_selection_equal_the_numpy_restatement():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    cols = sample_colours(job, STREAM)
    ad = rh.AdaptiveAccumulator(job, STREAM)
    for i, (b, t, m) in enumerate(zip((3, 2, 1, 2, 3, 4), (0.05, 0.02, 0.02, 0.0, 0.01, 0.0), (4, 4, 2, 2, 6, 2))):
        c0, s0, q0 = ad.state()
        act = active_pixels(c0, s0, q0, b, STREAM, m, t)
        img = ad.add(b, SEED, t, min_spp=m)
        c1, s1, q1 = ad.state()
        assert img.stats["n_active"] == int(act.sum()), i
        assert img.stats["rays_primary"] == int(act.sum()) * b, i
        assert np.array_equal(c1 > c0, act) and np.array_equal(c1[act], c0[act] + b), i
        S, Q = expected_state(cols, c1)
        assert s1.tobytes() == S.tobytes() and q1.tobytes() == Q.tobytes(), i
        assert img.linear.tobytes() == (np.where(c1[..., None] > 0, 1.0 / np.maximum(c1, 1)[..., None], 0.0) * s1).tobytes(), i
    assert i == 5 and (c1 == STREAM).any() and (c1 < STREAM).any()


def test_thresholds_at_their_extremes():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    ad = rh.AdaptiveAccumulator(job, STREAM)
    first = ad.add(2, SEED, np.inf, min_spp=4)
    assert first.stats["n_active"] == W * H  # the first call traces every pixel
    ad.add(2, SEED, np.inf, min_spp=4)
    idle = ad.add(2, SEED, np.inf, min_spp=4)  # threshold inf: every pixel stops at min_spp
    assert idle.stats["n_active"] == 0 and idle.stats["rays_primary"] == 0 and idle.stats["rays_shadow"] == 0
    counts, s, q = ad.state()
    assert (counts == 4).all()
    assert np.array_equal(idle.pixels, rh.Accumulator(job, STREAM).add(4, seed=SEED).pixels)  # outputs still written
    # threshold 0: every pixel with d > 0 goes on to the end of the stream; converged pixels are never traced again
    stopped = np.zeros((H, W), dtype=bool)
    prev = counts
    while True:
        img = ad.add(2, SEED, 0.0, min_spp=4)
        c, s, q = ad.state()
        assert not (c[stopped] != prev[stopped]).any()
        stopped |= c == prev
        prev = c
        if img.stats["n_active"] == 0:
            break
    d = q - s * (s / c[..., None])
    assert ((c == STREAM) | ~(d > 0).any(axis=-1)).all()
    assert (c == STREAM).any()


def test_adaptive_ray_trace_yields_until_converged():
    sc = load_scene(PLAIN)
    job = job_of(sc, 96, 64)
    images = list(rh.adaptiveRayTrace(job, max_spp=16, batch=4, min_spp=8, threshold=0.01, seed=24))
    n = [img.stats["n_active"] for img in images]
    assert n[0] == n[1] == 96 * 64 and all(a >= b for a, b in zip(n, n[1:])) and len(images) <= 4
    full = rh.distributedRayTrace(job, 16)
    ad = rh.AdaptiveAccumulator(job, 16)
    last = run(ad, (4,) * 4, threshold=0.01, min_spp=8, seed=24)
    assert np.array_equal(images[-1].pixels, last.pixels)
    counts = ad.state()[0]
    assert np.array_equal(images[-1].pixels[counts == 16], full.pixels[counts == 16])


@pytest.mark.parametrize("name", [PLAIN, "cornellBox"])
def test_chunking_keeps_the_state(name):
    sc = load_scene(name)
    job, forks = job_of(sc), has_transparent(sc)
    base, chunked = rh.AdaptiveAccumulator(job, STREAM), rh.AdaptiveAccumulator(job, STREAM)
    chunks = []
    for b in BATCHES[:3]:
        a = base.add(b, SEED, THRESHOLD, min_spp=4)
        c = chunked.add(b, SEED, THRESHOLD, min_spp=4, chunk_samples=1)  # one list row (1024 pixels) per chunk
        assert c.stats["n_active"] == a.stats["n_active"]
        assert c.stats["chunks"] == -(-a.stats["n_active"] // 1024)
        chunks.append(c.stats["chunks"])
        if forks:
            assert_parity(c.pixels, a.pixels, name)
        else:
            for x, y in zip(base.state(), chunked.state()):
                assert x.tobytes() == y.tobytes()
    assert max(chunks) == 3  # the first calls trace all 64 x 48 pixels: three list rows


@pytest.mark.parametrize("shards,band_height", [(2, 1), (2, 5), (3, 1), (3, 5)])
def test_shards_hold_the_whole_frames_state(shards, band_height):
    sc = load_scene(PLAIN)
    job = job_of(sc)
    whole = rh.AdaptiveAccumulator(job, STREAM)
    parts = [rh.AdaptiveAccumulator(job, STREAM, shard_index=g, shard_count=shards, band_height=band_height) for g in range(shards)]
    for b in BATCHES:
        w = whole.add(b, SEED, THRESHOLD)
        got = [p.add(b, SEED, THRESHOLD) for p in parts]
        assert sum(g.stats["n_active"] for g in got) == w.stats["n_active"]
        assert np.array_equal(rh.assemble_bands([g.pixels for g in got], H, band_height), w.pixels)
    want = whole.state()
    for g, p in enumerate(parts):
        rmap = np.array(rh.shard_global_rows(H, g, shards, band_height))
        real = rmap >= 0
        for x, y in zip(p.state(), want):
            assert x[real].tobytes() == y[rmap[real]].tobytes()
        assert (p.state()[0][~real] == 0).all()  # padding rows are never traced


def test_device_buffers_equal_the_host_path():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    hst, dev = rh.AdaptiveAccumulator(job, STREAM), rh.AdaptiveAccumulator(job, STREAM, device=True)
    for b in BATCHES:
        h = hst.add(b, SEED, THRESHOLD)
        d = dev.add(b, SEED, THRESHOLD)
        assert d.pixels.is_cuda and d.linear.is_cuda
        assert np.array_equal(d.pixels.cpu().numpy(), h.pixels) and d.linear.cpu().numpy().tobytes() == h.linear.tobytes()
        assert d.stats["n_active"] == h.stats["n_active"]
    for x, y in zip(dev.state(), hst.state()):
        assert x.is_cuda and x.cpu().numpy().tobytes() == y.tobytes()


def test_validation_flags_mixed_across_calls_keep_the_state():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    plain, mixed = rh.AdaptiveAccumulator(job, STREAM), rh.AdaptiveAccumulator(job, STREAM)
    for b, kw in zip(BATCHES, (dict(shadow="split"), dict(exact_boxes=True), dict(light_maps=False), dict(shadow="pooled"),
                               dict(count=True, profile=True))):
        a = plain.add(b, SEED, THRESHOLD)
        c = mixed.add(b, SEED, THRESHOLD, **kw)
        assert np.array_equal(c.pixels, a.pixels), kw
    assert c.stats["box_tests"] > 0 and c.stats["ms_resolve"] > 0
    for x, y in zip(plain.state(), mixed.state()):
        assert x.tobytes() == y.tobytes()


def test_queue_growth_retry_counts_no_sample_twice_and_leaves_the_scene_alone():
    """Both calls overflow their queues (a list frame starts from the scene's factor and never raises it) and run their
    frame again; the second continues existing sums, so a sink that wrote the state would count samples twice.  After
    them the scene renders as a copy that never saw them: same queue factor and shadow schedule."""
    sc, ref_sc, fresh = growth_scene(), growth_scene(), growth_scene()  # Transparent spheres in a box of mirrors
    w = h = 512
    job, ref_job = rh.Rendering(sc, sc.camera, w, h, 8), rh.Rendering(ref_sc, ref_sc.camera, w, h, 8)
    ad, acc = rh.AdaptiveAccumulator(job, 8), rh.Accumulator(ref_job, 8)
    n = 0
    for b in (4, 4):
        img = ad.add(b, 21, 0.0, min_spp=8)  # every pixel is active: n < min_spp
        ref = acc.add(b, seed=21)
        n += b
        assert img.stats["n_active"] == w * h and img.stats["queue_factor"] > 2, img.stats
        assert (ad.state()[0] == n).all()
        ok = np.isclose(img.linear, ref.linear, rtol=1e-9, atol=1e-12, equal_nan=True).all(axis=-1)
        assert ok.all(), np.argwhere(~ok)[:5]
        assert_parity(img.pixels, ref.pixels)  # (Transparent forks: the 1-LSB wobble)
    small = dict(spp=2, seed=5)
    got = rh.render(rh.Rendering(sc, sc.camera, 64, 64, 8), **small)
    want = rh.render(rh.Rendering(fresh, fresh.camera, 64, 64, 8), **small)
    for k in ("queue_factor", "shadow_split", "chunks"):
        assert got.stats[k] == want.stats[k], k


def test_renders_are_unaffected():
    sc = load_scene(PLAIN)
    job = job_of(sc)
    before = rh.render(job, spp=4, seed=3)
    run(rh.AdaptiveAccumulator(job, STREAM))
    after = rh.render(job, spp=4, seed=3)
    assert np.array_equal(before.pixels, after.pixels)
    for k in ("queue_factor", "shadow_split", "chunks", "rays_reflect", "rays_shadow"):
        assert before.stats[k] == after.stats[k], k


def test_failed_calls_leave_the_state_and_reset_allows_another_view():
    import torch

    sc, other = load_scene(PLAIN), load_scene("dragon_superlow")
    job = job_of(sc)
    ad = rh.AdaptiveAccumulator(job, STREAM)
    ad.add(3, SEED, THRESHOLD)
    before = ad.state()
    L = capi.lib()
    seed = C.c_uint64(SEED)
    rgb = np.empty((H, W, 3), dtype=np.uint8)

    def call(scene=sc, camera=job.camera, threshold=THRESHOLD, min_spp=2, reserved=0, **kw):
        o = host._opts(job, 2, capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed), 0, 0, 1, H, 0, 0)
        for k, v in kw.items():
            setattr(o, k, v)
        ao = capi.rh_adaptive_opts()
        ao.threshold, ao.min_spp, ao.reserved_ = threshold, min_spp, reserved
        n = C.c_uint64(12345)
        rc = L.rh_render_adaptive(scene.device, C.byref(camera), C.byref(o), C.byref(ao), ad._h, rgb.ctypes.data, None,
                                  C.byref(n), None)
        return rc, L.rh_last_error().decode(), n.value

    cam = capi.rh_camera.from_buffer_copy(job.camera)
    cam.position[0] += 1e-9
    off = rh.sample_offsets(W * H, 2)
    cases = [
        (dict(offset_mode=capi.RH_OFFSETS_F64, offsets=off.ctypes.data), "RH_OFFSETS_SPLITMIX64"),
        (dict(offset_mode=capi.RH_OFFSETS_NONE, offsets=None), "RH_OFFSETS_SPLITMIX64"),
        (dict(flags=capi.RH_FLAG_HIT_IDS), "not supported"), (dict(flags=capi.RH_FLAG_PEER_FRAMES), "not supported"),
        (dict(flags=capi.RH_FLAG_SHARD_OFFSETS), "not supported"), (dict(flags=capi.RH_FLAG_DEVICE_OFFSETS), "not supported"),
        (dict(min_spp=1), "min_spp"), (dict(min_spp=0), "min_spp"), (dict(reserved=1), "reserved_"),
        (dict(threshold=-1.0), "threshold"), (dict(threshold=float("nan")), "threshold"),
        (dict(camera=cam), "rh_adaptive_reset"), (dict(scene=other), "rh_adaptive_reset"),
        (dict(max_depth=job.maxDepth - 1), "rh_adaptive_reset"),
        (dict(width=W + 1), "differ from the adaptive state"), (dict(shard_count=2), "differ from the adaptive state"),
        (dict(band_height=5), "differ from the adaptive state"), (dict(spp=0), "bad width/height/spp/max_depth"),
        (dict(flags=capi.RH_FLAG_DEVICE_OUT), "not device memory"),
    ]
    for kw, msg in cases:
        rc, err, n = call(**kw)
        assert rc == capi.RH_ERR_ARG and msg in err and err.startswith("rh_render_adaptive") and n == 12345, (kw, rc, err)
    d = torch.empty(H * W * 3 + 1, dtype=torch.float64, device="cuda")
    o = host._opts(job, 2, capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed), 0, 0, 1, H, 0, capi.RH_FLAG_DEVICE_OUT)
    ao = capi.rh_adaptive_opts(THRESHOLD, 2, 0)
    assert L.rh_render_adaptive(sc.device, C.byref(job.camera), C.byref(o), C.byref(ao), ad._h, None, d.data_ptr() + 4, None,
                                None) == capi.RH_ERR_ARG
    for x, y in zip(ad.state(), before):
        assert x.tobytes() == y.tobytes()
    assert call()[0] == capi.RH_OK
    # create errors
    h = C.c_void_p()
    for args, msg in (((0, H, 0, 1, 0, 4), "bad width/height"), ((W, H, 2, 2, 0, 4), "shard_index out of range"),
                      ((W, H, 0, 1, 0, 0), "stream_spp")):
        assert L.rh_adaptive_create(*args, C.byref(h)) == capi.RH_ERR_ARG and msg in L.rh_last_error().decode(), args
    # reset: counts back to 0, and another view is fine
    ad.reset()
    assert not ad.state()[0].any() and not ad.state()[1].any()
    other_job = job_of(other)
    ad.job = other_job  # (the job supplies the view of the next call)
    b = ad.add(4, SEED, np.inf, min_spp=4)
    assert (ad.state()[0] == 4).all()
    assert np.array_equal(b.pixels, rh.Accumulator(other_job, STREAM).add(4, seed=SEED).pixels)
