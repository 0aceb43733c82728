"""GPU tests of the camera batches (rh_render_views / renderViews): every view against its own rh_render (bytes, hit
ids, negative channels, summed ray counts) for every shipped pack and a built scene with every material kind, both
projections in one batch, every offset mode and batches of 1, 3 and 17 views; per-view seeds; the linear colours
against a fresh accumulator; chunking, shards with padding rows, shard-compact and device offsets, device outputs,
exact boxes, both shadow schedules and no light maps; many small views; the oracle directly; the scene's learned
state, scene updates and the queue-overflow retry; argument errors."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from rayhs_b200 import capi
from tests.test_features_gpu import BUILT, SIZES
from tests.test_trace_rays_gpu import growth_scene, has_transparent
from tests.util import ATOL, RTOL, SCENES, assert_parity, load_scene

pytestmark = pytest.mark.gpu

COUNTS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow", "rays_shadow_culled", "shadow_walk_pairs",
          "shadow_tasks", "shadow_tasks_queued", "queued_rays")
RAYS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
TILE = 5
_cache = {}


def scene(name):
    if name not in _cache:
        _cache[name] = BUILT[name]() if name in BUILT else load_scene(name)
    return _cache[name]


def cameras(sc, V, seed=0):
    """V cameras around the scene's own: view 0 is it, the others move position and target; every third view has the
    other projection (a perspective one gets fovy 1 when the scene's camera has none)."""
    rng = np.random.RandomState(seed * 1000 + V)
    out = []
    for v in range(V):
        c = capi.rh_camera.from_buffer_copy(sc.camera)
        if v:
            d = rng.uniform(-0.3, 0.3, 3)
            for k in range(3):
                c.position[k] += d[k]
                c.target[k] += 0.5 * d[k]
        if v % 3 == 2:
            c.projection = 1 - c.projection
            if c.projection == capi.RH_PROJ_PERSPECTIVE and not c.fovy > 0:
                c.fovy = 1.0
        out.append(c)
    return out


def job(sc, w, h, cam=None, depth=None):
    return rh.Rendering(sc, sc.camera if cam is None else cam, w, h, sc.max_depth if depth is None else depth)


def sources(w, h, spp):
    """Every offset mode: NONE, F64, F32, TILED_F64 and SPLITMIX64 (keyword arguments of render and renderViews)."""
    rng = np.random.RandomState(7 + spp)
    f64 = rng.uniform(-0.5, 0.5, (w * h, spp, 2))
    return {"none": {}, "f64": dict(offsets=f64), "f32": dict(offsets=f64.astype(np.float32)),
            "tiled": dict(offsets=rng.uniform(-0.5, 0.5, (TILE * TILE, spp, 2)), offset_tile=TILE), "splitmix": dict(seed=24)}


def host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def same(a, b, what):
    a, b = host(a), host(b)
    assert a.shape == b.shape and np.array_equal(a, b, equal_nan=True), (what, int((a != b).sum()))


def agree(sc, a, b, what):
    """Two runs of one frame: bit for bit, or, in a scene with a Transparent material, within the 1-LSB wobble of its
    forks (DESIGN §3): assert_parity on RGB8, RTOL / ATOL on 99.9 % of linear values."""
    a, b = host(a), host(b)
    assert a.shape == b.shape, what
    if not has_transparent(sc):
        assert np.array_equal(a, b, equal_nan=True), (what, int((a != b).sum()))
    elif a.dtype == np.uint8:
        for v in range(a.shape[0]):
            assert_parity(a[v], b[v], str((what, v)))
    else:
        ok = np.isclose(a, b, rtol=RTOL, atol=ATOL, equal_nan=True)
        assert ok.mean() > 0.999, (what, int((~ok).sum()))


def real_rows(h, shard_index=0, shard_count=1, band_height=0):
    bh = band_height or capi.lib().rh_default_band_height(h, shard_count)
    return [lr for lr, row in enumerate(rh.shard_global_rows(h, shard_index, shard_count, bh)) if row >= 0]


def assert_views_equal_renders(sc, vs, cams, w, h, spp, what, ids=True, counts=True, **kw):
    """Each view against rh.render of its camera (same keyword arguments), and the ray counts against the renders' sums."""
    tr = has_transparent(sc)
    sums = dict.fromkeys(COUNTS + ("negative_channels",), 0)
    rows = real_rows(h, kw.get("shard_index", 0), kw.get("shard_count", 1), kw.get("band_height", 0))
    for v, cam in enumerate(cams):
        img = rh.render(job(sc, w, h, cam), spp=spp, want_hit_ids=ids, **kw)
        got = host(vs.pixels[v])
        if tr:
            assert_parity(got, img.pixels, str((what, v)))  # (Transparent forks: the 1-LSB wobble)
        else:
            assert np.array_equal(got, img.pixels), (what, v, int((got != img.pixels).sum()))
        if ids:
            assert np.array_equal(host(vs.hit_ids[v])[rows], img.hit_ids[rows]), (what, v)
        for k in sums:
            sums[k] += img.stats[k]
    if counts:
        for k in COUNTS:
            assert vs.stats[k] == sums[k], (what, k, vs.stats[k], sums[k])
        if not tr:
            assert vs.stats["negative_channels"] == sums["negative_channels"], what


# ---------------------------------------------------------------- 1. each view equals its own render
@pytest.mark.parametrize("name", SCENES + list(BUILT))
@pytest.mark.parametrize("w,h", SIZES)
def test_each_view_equals_its_own_render(name, w, h):
    sc = scene(name)
    j = job(sc, w, h)
    for spp in (1, 4):
        for mode, src in sources(w, h, spp).items():
            for V in (1, 3, 17):
                cams = cameras(sc, V)
                vs = rh.renderViews(j, cams, spp=spp, want_hit_ids=True, **src)
                assert vs.pixels.shape == (V, h, w, 3) and vs.hit_ids.shape == (V, h, w, spp, 2)
                assert_views_equal_renders(sc, vs, cams, w, h, spp, (name, w, h, spp, mode, V), **src)


# ---------------------------------------------------------------- 2. per-view seeds
@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "built_perspective"])
def test_per_view_seeds(name):
    sc = scene(name)
    w, h = SIZES[1]
    spp = 2
    base = cameras(sc, 3)
    cams = [base[0], base[0], base[1], base[2]]
    seeds = [3, 4, 2**64 - 1, 24]
    vs = rh.renderViews(job(sc, w, h), cams, spp=spp, seeds=seeds, want_hit_ids=True)
    for v, (cam, s) in enumerate(zip(cams, seeds)):
        img = rh.render(job(sc, w, h, cam), spp=spp, seed=s, want_hit_ids=True)
        if has_transparent(sc):
            assert_parity(vs.pixels[v], img.pixels, str((name, v)))
        else:
            assert np.array_equal(vs.pixels[v], img.pixels), (name, v)
        assert np.array_equal(vs.hit_ids[v], img.hit_ids), (name, v)
    assert not np.array_equal(vs.pixels[0], vs.pixels[1])  # same camera, other seed
    assert not np.array_equal(vs.hit_ids[0], vs.hit_ids[1])
    one = rh.renderViews(job(sc, w, h), cams, spp=spp, seed=24)  # no seeds: every view uses the one seed
    if has_transparent(sc):
        assert_parity(one.pixels[3], vs.pixels[3])
    else:
        same(one.pixels[3], vs.pixels[3], (name, "seed 24"))


# ---------------------------------------------------------------- 3. linear_out
@pytest.mark.parametrize("name", SCENES + list(BUILT))
def test_linear_equals_a_fresh_accumulator(name):
    sc = scene(name)
    w, h = SIZES[0]
    cams = cameras(sc, 3)
    for spp, src in ((1, dict(seed=24)), (4, dict(seed=5)), (2, dict(offsets=sources(w, h, 2)["f64"]["offsets"]))):
        vs = rh.renderViews(job(sc, w, h), cams, spp=spp, linear=True, **src)
        lin_only = rh.renderViews(job(sc, w, h), cams, spp=spp, rgb=False, linear=True, **src)
        assert vs.linear.shape == (3, h, w, 3) and vs.linear.dtype == np.float64 and lin_only.pixels is None
        for v, cam in enumerate(cams):
            acc = rh.Accumulator(job(sc, w, h, cam), stream_spp=spp if "seed" in src else 0)
            a = acc.add(spp, **src)
            acc.close()
            for got in (vs.linear[v], lin_only.linear[v]):
                if has_transparent(sc):
                    ok = np.isclose(got, a.linear, rtol=RTOL, atol=ATOL, equal_nan=True)
                    assert ok.mean() > 0.999, (name, v, int((~ok).sum()))
                else:
                    assert got.tobytes() == a.linear.tobytes(), (name, spp, v)
            if not has_transparent(sc):
                assert np.array_equal(vs.pixels[v], a.pixels), (name, spp, v)


# ---------------------------------------------------------------- 4. the frame does not depend on how it is run
@pytest.mark.parametrize("name", [n for n in SCENES + list(BUILT) if not has_transparent(scene(n))])
def test_views_do_not_depend_on_how_the_frame_is_run(name):
    sc = scene(name)
    w, h = SIZES[0]
    spp, V = 2, 5
    j, cams = job(sc, w, h), cameras(sc, V)
    ref = rh.renderViews(j, cams, spp=spp, seed=24, linear=True, want_hit_ids=True, shadow="pooled")
    variants = {"split": dict(shadow="split"), "exact_boxes": dict(exact_boxes=True), "no_light_maps": dict(light_maps=False),
                "chunks_mid_view": dict(chunk_samples=w * spp * 7), "chunks_span_views": dict(chunk_samples=w * spp * (h + h // 2)),
                "chunks_many_views": dict(chunk_samples=w * spp * 3 * h), "device": dict(device=True), "profile": dict(profile=True),
                "default": dict(), "again": dict(shadow="pooled")}
    for tag, kw in variants.items():
        got = rh.renderViews(j, cams, spp=spp, seed=24, linear=True, want_hit_ids=True, **kw)
        same(got.pixels, ref.pixels, (name, tag))
        same(got.linear, ref.linear, (name, tag, "linear"))
        same(got.hit_ids, ref.hit_ids, (name, tag, "ids"))
        for k in RAYS:  # (the walk and queue counts depend on the flags; each variant's are checked against its renders below)
            assert got.stats[k] == ref.stats[k], (name, tag, k)
    assert rh.renderViews(j, cams, spp=spp, seed=24, chunk_samples=w * spp * 7).stats["chunks"] > V
    # each view still equals its render under the flags
    for kw in (dict(shadow="split"), dict(exact_boxes=True), dict(light_maps=False)):
        vs = rh.renderViews(j, cams, spp=spp, seed=24, want_hit_ids=True, **kw)
        assert_views_equal_renders(sc, vs, cams, w, h, spp, (name, kw), seed=24, **kw)


@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "built_orthographic", "texture"])
@pytest.mark.parametrize("G,bh", [(2, 5), (3, 7), (3, 4)])
def test_shards_with_padding_rows(name, G, bh):
    sc = scene(name)
    w, h = SIZES[0]
    spp, V = 2, 4
    j, cams = job(sc, w, h), cameras(sc, V)
    f64 = sources(w, h, spp)["f64"]["offsets"]
    for i in range(G):
        shard = dict(shard_index=i, shard_count=G, band_height=bh)
        rows = real_rows(h, i, G, bh)
        n_rows = capi.lib().rh_shard_rows(h, G, bh)
        for src in (dict(seed=24), dict(offsets=f64)):
            vs = rh.renderViews(j, cams, spp=spp, linear=True, want_hit_ids=True, chunk_samples=w * spp * 3, **shard, **src)
            assert vs.pixels.shape == (V, n_rows, w, 3)
            assert_views_equal_renders(sc, vs, cams, w, h, spp, (name, G, bh, i, list(src)), **shard, **src)
            pad = [lr for lr in range(n_rows) if lr not in rows]
            assert not vs.pixels[:, pad].any() and not vs.linear[:, pad].any()  # padding rows: 0
        # shard-compact offsets: this shard's rows only, padding rows anything
        gl = rh.shard_global_rows(h, i, G, bh)
        compact = np.full((n_rows, w, spp, 2), 0.25)
        full = f64.reshape(h, w, spp, 2)
        for lr, row in enumerate(gl):
            if row >= 0:
                compact[lr] = full[row]
        want = rh.renderViews(j, cams, spp=spp, offsets=f64, linear=True, **shard)
        got = rh.renderViews(j, cams, spp=spp, offsets=compact.reshape(-1, spp, 2), shard_offsets=True, linear=True, **shard)
        agree(sc, got.pixels, want.pixels, (name, G, bh, i, "shard offsets"))
        agree(sc, got.linear, want.linear, (name, G, bh, i, "shard offsets linear"))
        import torch

        dev = rh.renderViews(j, cams, spp=spp, offsets=torch.from_numpy(compact.reshape(-1, spp, 2)).cuda(), shard_offsets=True,
                             linear=True, **shard)
        assert dev.pixels.is_cuda and dev.linear.is_cuda
        agree(sc, dev.pixels, want.pixels, (name, G, bh, i, "device shard offsets"))
        agree(sc, dev.linear, want.linear, (name, G, bh, i, "device shard offsets linear"))


def test_device_offsets_and_outputs():
    import torch

    sc = scene("texture")
    w, h = SIZES[1]
    spp, V = 2, 3
    j, cams = job(sc, w, h), cameras(sc, V)
    for mode in ("f64", "f32", "tiled"):
        src = sources(w, h, spp)[mode]
        ref = rh.renderViews(j, cams, spp=spp, linear=True, want_hit_ids=True, **src)
        dsrc = dict(src, offsets=torch.from_numpy(src["offsets"]).cuda())
        got = rh.renderViews(j, cams, spp=spp, linear=True, want_hit_ids=True, **dsrc)
        assert got.pixels.is_cuda and got.linear.is_cuda and got.hit_ids.is_cuda
        for a, b, what in ((got.pixels, ref.pixels, "rgb"), (got.linear, ref.linear, "linear")):
            agree(sc, a, b, (mode, what))
        same(got.hit_ids, ref.hit_ids, (mode, "ids"))
        assert_views_equal_renders(sc, ref, cams, w, h, spp, ("texture", mode), **src)


# ---------------------------------------------------------------- 5. many small views
def test_many_small_views():
    sc = scene("dragon_low")
    w = h = 32
    V, spp = 256, 1
    cams = cameras(sc, V, seed=3)
    vs = rh.renderViews(job(sc, w, h), cams, spp=spp, seed=24, want_hit_ids=True, linear=True)
    assert vs.stats["chunks"] >= 1 and vs.stats["rays_primary"] == V * w * h * spp
    assert_views_equal_renders(sc, vs, cams, w, h, spp, "many", seed=24)
    chunked = rh.renderViews(job(sc, w, h), cams, spp=spp, seed=24, chunk_samples=w * h * spp * 40 + w * spp * 5, linear=True)
    assert chunked.stats["chunks"] > 1
    agree(sc, chunked.pixels, vs.pixels, "chunked")
    agree(sc, chunked.linear, vs.linear, "chunked linear")


# ---------------------------------------------------------------- 6. the oracle directly
@pytest.mark.parametrize("name", ["cornellBox", "built_perspective"])
def test_views_against_the_oracle(name):
    sc = scene(name)
    w, h = SIZES[0]
    spp, V = 2, 3
    cams = cameras(sc, V, seed=1)
    offsets = rh.sample_offsets(w * h, spp, 24)
    vs = rh.renderViews(job(sc, w, h), cams, spp=spp, seed=24, want_hit_ids=True, linear=True)
    orc = OracleScene(sc.raw)
    for v, cam in enumerate(cams):
        ref = orc.render(cam, w, h, sc.max_depth, spp=spp, offsets=offsets)
        assert np.array_equal(vs.hit_ids[v].reshape(h, w, spp, 2), ref["hit_ids"].reshape(h, w, spp, 2)), (name, v)
        diff = np.abs(vs.pixels[v].astype(int) - ref["rgb_u8"].astype(int))
        assert diff.max() <= 1 and (diff == 0).mean() > 0.999, (name, v, diff.max())
        ok = np.isclose(vs.linear[v], ref["rgb_f64"], rtol=RTOL, atol=ATOL, equal_nan=True)
        assert ok.mean() > 0.999, (name, v, int((~ok).sum()))


# ---------------------------------------------------------------- 7. scene state
GROWTH = 1024  # a frame large enough that the queues' per-warp slack is small beside its samples


def test_the_call_leaves_the_scenes_render_state_alone():
    """An overflowing views call, then a render: the render behaves as on a scene that never had the call (same bytes,
    queue factor, shadow schedule and chunks)."""
    small = lambda sc: rh.Rendering(sc, sc.camera, 256, 256, 0)  # noqa: E731
    used, fresh = growth_scene(), growth_scene()
    vs = rh.renderViews(rh.Rendering(used, used.camera, GROWTH, GROWTH, 8), [used.camera], seed=24)
    assert vs.stats["queue_factor"] > 2, vs.stats
    after, ref = rh.render(small(used)), rh.render(small(fresh))
    assert_parity(after.pixels, ref.pixels)  # (Transparent forks: the 1-LSB wobble)
    for k in ("queue_factor", "shadow_split", "chunks", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert after.stats[k] == ref.stats[k], k


def test_a_render_of_the_views_shape_behaves_as_on_a_fresh_scene():
    """Views calls at a render's own shape, with host offsets, then that render: it streams its offsets in the chunks, and
    takes the shadow schedule, of the first render of a fresh scene.  (Two views calls of 8 M samples would be the
    scene's first two shadow-timing frames if they counted, and the render its third, which runs the refill walk.)"""
    w = h = 1024
    spp = 8  # (8 M samples: more than the first streamed chunk holds)
    off = np.random.RandomState(3).uniform(-0.5, 0.5, (w * h, spp, 2))
    used, fresh = load_scene("dragon_low"), load_scene("dragon_low")
    for _ in range(2):
        rh.renderViews(job(used, w, h), [used.camera], spp=spp, offsets=off)
    after, ref = rh.render(job(used, w, h), spp=spp, offsets=off), rh.render(job(fresh, w, h), spp=spp, offsets=off)
    assert ref.stats["chunks"] > 1 and ref.stats["upload_bytes"] > 0  # (a streamed frame: the row costs would be used)
    assert np.array_equal(after.pixels, ref.pixels)
    for k in ("chunks", "shadow_split", "queue_factor", "upload_bytes"):
        assert after.stats[k] == ref.stats[k], k


def test_queue_factor_of_a_batch():
    """Small renders leave the scene a large queue factor; a batch 256 times their size still runs (its start is bounded
    by the memory a chunk is planned for) and equals the batch on a fresh scene.  A small batch remembers what it needed:
    the second call of one runs without an overflow retry."""
    w = h = 128
    used, fresh = load_scene("dragon_full"), load_scene("dragon_full")
    cams = cameras(used, 256, seed=5)
    factors = [rh.render(job(used, w, h, c), seed=24).stats["queue_factor"] for c in cams[:4]]
    got = rh.renderViews(job(used, w, h), cams, spp=16, seed=24, linear=True)
    want = rh.renderViews(job(fresh, w, h), cams, spp=16, seed=24, linear=True)
    agree(used, got.pixels, want.pixels, "large batch")
    agree(used, got.linear, want.linear, "large batch linear")
    assert got.stats["queue_factor"] <= max(factors + [want.stats["queue_factor"]]), (factors, got.stats, want.stats)
    L = capi.lib()
    small = load_scene("dragon_full")
    for k in range(2):
        before = L.rh_launch_count()
        vs = rh.renderViews(job(small, w, h), cams[:6], seed=24)
        if k == 1:
            assert L.rh_launch_count() - before == vs.stats["kernel_launches"], vs.stats  # one attempt


def test_queue_overflow_retry_keeps_the_oracle_agreement():
    sc = growth_scene()
    w = h = GROWTH
    cams = [sc.camera, cameras(sc, 2)[1]]
    vs = rh.renderViews(rh.Rendering(sc, sc.camera, w, h, 8), cams, seed=24, linear=True)
    assert vs.stats["queue_factor"] > 2, vs.stats
    offsets = rh.sample_offsets(w * h, 1, 24)
    rows = (5, None, 97)
    for v, cam in enumerate(cams):
        ref = OracleScene(sc.raw).render(cam, w, h, 8, spp=1, offsets=offsets, rows=rows)["rgb_f64"][slice(*rows)]
        ok = np.isclose(vs.linear[v][slice(*rows)], ref, rtol=RTOL, atol=ATOL, equal_nan=True)
        assert ok.all(), (v, int((~ok).sum()))


def test_views_show_a_scene_update():
    sc = load_scene("cornellBox")  # (a fresh copy: the update changes it)
    w, h = SIZES[0]
    cams = cameras(sc, 3)
    before = rh.renderViews(job(sc, w, h), cams, seed=24, linear=True)
    lights = sc.lights
    for c in range(3):
        lights[0].color[c] *= 0.5
    sc.update(lights=lights)
    after = rh.renderViews(job(sc, w, h), cams, seed=24, linear=True, want_hit_ids=True)
    assert not np.array_equal(before.linear, after.linear)
    assert_views_equal_renders(sc, after, cams, w, h, 1, "updated", seed=24)


# ---------------------------------------------------------------- 8. argument errors
def test_argument_errors():
    import torch

    sc = scene("cornellBox")
    L = capi.lib()
    w, h, spp, V = 16, 8, 1, 3
    o = rh.host._opts(job(sc, w, h), spp, capi.RH_OFFSETS_NONE, None, 0, 0, 1, h, 0, 0)
    cams = (capi.rh_camera * V)(*cameras(sc, V))
    rgb = np.full((V, h, w, 3), 9, np.uint8)
    lin = np.full((V, h, w, 3), 7.0)
    seeds = (C.c_uint64 * V)(1, 2, 3)

    def call(flags=0, n_views=V, reserved=0, cams_=cams, seeds_=None, rgb_ptr=None, lin_ptr=None, mode=capi.RH_OFFSETS_NONE,
             offsets=None):
        oo = capi.rh_render_opts.from_buffer_copy(o)
        oo.flags, oo.offset_mode, oo.offsets = flags, mode, offsets
        vw = capi.rh_views()
        vw.cameras = C.cast(cams_, C.POINTER(capi.rh_camera)) if cams_ is not None else None
        vw.n_views, vw.reserved_ = n_views, reserved
        if seeds_ is not None:
            vw.seeds = C.cast(seeds_, C.POINTER(C.c_uint64))
        return L.rh_render_views(sc.device, C.byref(vw), C.byref(oo), rgb.ctypes.data if rgb_ptr is None else rgb_ptr,
                                 lin.ctypes.data if lin_ptr is None else lin_ptr, None, None)

    bad = (capi.rh_camera * V)(*cameras(sc, V))
    bad[2].projection = 7
    f64 = np.zeros((w * h, spp, 2))
    cases = [dict(n_views=0), dict(n_views=65537), dict(cams_=None), dict(reserved=1), dict(cams_=bad),
             dict(seeds_=seeds), dict(seeds_=seeds, mode=capi.RH_OFFSETS_F64, offsets=f64.ctypes.data),
             dict(flags=capi.RH_FLAG_COUNT), dict(flags=capi.RH_FLAG_PEER_FRAMES), dict(flags=capi.RH_FLAG_HIT_IDS),
             dict(rgb_ptr=0, lin_ptr=0)]
    for kw in cases:
        assert call(**kw) == capi.RH_ERR_ARG, kw
        assert (rgb == 9).all() and (lin == 7.0).all(), kw
        if "cams_" in kw and kw["cams_"] is bad:
            assert b"cameras[2]" in L.rh_last_error(), L.rh_last_error()
    assert L.rh_render_views(sc.device, None, C.byref(o), rgb.ctypes.data, None, None, None) == capi.RH_ERR_ARG
    with pytest.raises(capi.RayHsError) as e:
        rh.renderViews(job(sc, w, h), [])
    assert e.value.code == capi.RH_ERR_ARG
    # device outputs: host memory and a misaligned device pointer
    D = capi.RH_FLAG_DEVICE_OUT
    t = torch.full((V * h * w * 3 + 1,), 5.0, dtype=torch.float64, device="cuda")
    r = torch.zeros((V, h, w, 3), dtype=torch.uint8, device="cuda")
    assert call(flags=D, lin_ptr=t.data_ptr() + 4, rgb_ptr=r.data_ptr()) == capi.RH_ERR_ARG
    assert call(flags=D, rgb_ptr=r.data_ptr()) == capi.RH_ERR_ARG
    assert (t == 5.0).all() and (lin == 7.0).all() and (rgb == 9).all()
    assert call(flags=D, lin_ptr=t.data_ptr() + 8, rgb_ptr=r.data_ptr()) == capi.RH_OK
    assert call(seeds_=seeds, mode=capi.RH_OFFSETS_SPLITMIX64, offsets=C.addressof(seeds)) == capi.RH_OK
    assert call() == capi.RH_OK and (lin != 7.0).any() and (rgb != 9).any()
    assert call(rgb_ptr=0) == capi.RH_OK and call(lin_ptr=0) == capi.RH_OK
