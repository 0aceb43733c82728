"""GPU tests of the light groups (rh_render_light_groups / renderLightGroups): the render's bytes, hit ids and ray counts
beside the groups; every group plus the remainder against the oracle's render of the scene with only that group's
lights; the group images bit for bit across shadow schedules, exact boxes, light maps, chunking, shards, buffers,
profiling and repeated calls; relighting after a colours-only scene update; the queue-overflow retry; the scene's
learned state; a non-finite light; argument errors.  Every shipped pack and a built scene with every material kind."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from rayhs_b200 import capi
from tests import value_cases as vc
from tests.test_features_gpu import BUILT, SIZES
from tests.test_trace_rays_gpu import growth_scene, has_transparent
from tests.util import ATOL, RTOL, SCENES, assert_parity, load_scene

pytestmark = pytest.mark.gpu

COUNTS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow", "rays_shadow_culled", "shadow_walk_pairs",
          "shadow_tasks", "shadow_tasks_queued", "queued_rays")
_cache = {}


def scene(name):
    if name not in _cache:
        _cache[name] = BUILT[name]() if name in BUILT else load_scene(name)
    return _cache[name]


def job(sc, w, h):
    return rh.Rendering(sc, sc.camera, w, h, sc.max_depth)


def n_lights(sc):
    return sc.raw.contents.n_lights


def f64_offsets(w, h, spp, seed=7):
    return np.random.RandomState(seed).uniform(-0.5, 0.5, (w * h, spp, 2))


def partitions(L):
    """One group per light, all lights in one group, and (with two or more lights) the first two sharing a group."""
    out = [list(range(L)), [0] * L]
    if L >= 2:
        out.append([0, 0] + list(range(1, L - 1)))
    return out


class Oracle:
    """The oracle's renders of a scene restricted to subsets of its lights (the raw scene's light table patched)."""

    def __init__(self, sc):
        self.sc, self.frames = sc, {}

    def linear(self, lights, w, h, depth, spp, offsets, rows=(0, None, 1)):
        key = (tuple(lights), w, h, depth, spp, rows)
        if key not in self.frames:
            src = self.sc.raw.contents
            raw = capi.rh_raw_scene.from_buffer_copy(src)
            table = (capi.rh_light * max(len(lights), 1))(*[src.lights[i] for i in lights])
            raw.lights, raw.n_lights = C.cast(table, C.POINTER(capi.rh_light)), len(lights)
            self.frames[key] = OracleScene(C.pointer(raw)).render(self.sc.camera, w, h, depth, spp=spp, offsets=offsets,
                                                                rows=rows)["rgb_f64"][slice(*rows)]
        return self.frames[key]


def assert_close(got, want, what):
    ok = np.isclose(got, want, rtol=RTOL, atol=ATOL, equal_nan=True)
    assert ok.all(), (what, int((~ok).sum()), np.argwhere(~ok)[:4].tolist())


def assert_oracle(lgs, orc, groups, w, h, depth, spp, offsets, what, rows=(0, None, 1)):
    """groups[g] + rest against the oracle with only g's lights, and rest against it without lights (on `rows`)."""
    L, sl = len(groups), slice(*rows)
    for g in range(lgs.groups.shape[0]):
        members = [l for l in range(L) if groups[l] == g]
        assert_close(lgs.groups[g][sl] + lgs.rest[sl], orc.linear(members, w, h, depth, spp, offsets, rows), (what, "group", g, members))
    assert_close(lgs.rest[sl], orc.linear([], w, h, depth, spp, offsets, rows), (what, "rest"))


def same(a, b, what):
    a, b = (x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x) for x in (a, b))
    assert a.shape == b.shape and np.array_equal(a, b, equal_nan=True), (what, int((a != b).sum()))


# ---------------------------------------------------------------- 1. beauty and bookkeeping
@pytest.mark.parametrize("name", SCENES + list(BUILT))
@pytest.mark.parametrize("w,h", SIZES)
def test_beauty_ids_and_counts_equal_the_render(name, w, h):
    sc = scene(name)
    j = job(sc, w, h)
    for spp in (1, 4):
        for src in (dict(offsets=f64_offsets(w, h, spp)), dict(seed=24)):
            tag = (name, w, h, spp, list(src))
            img = rh.render(j, spp=spp, want_hit_ids=True, **src)
            lgs = rh.renderLightGroups(j, spp=spp, want_hit_ids=True, **src)
            if has_transparent(sc):
                assert_parity(lgs.image, img.pixels, str(tag))  # (Transparent forks: the 1-LSB wobble)
            else:
                assert np.array_equal(lgs.image, img.pixels), tag
                assert lgs.stats["negative_channels"] == img.stats["negative_channels"], tag
            assert np.array_equal(lgs.hit_ids, img.hit_ids), tag
            for k in COUNTS:
                assert lgs.stats[k] == img.stats[k], (tag, k, lgs.stats[k], img.stats[k])


# ---------------------------------------------------------------- 2. against the oracle
@pytest.mark.parametrize("name", SCENES + list(BUILT))
@pytest.mark.parametrize("w,h", SIZES)
def test_groups_equal_the_oracle_with_their_lights_only(name, w, h):
    sc = scene(name)
    j, orc, spp = job(sc, w, h), Oracle(sc), 2
    offsets = rh.sample_offsets(w * h, spp, 24)
    for groups in partitions(n_lights(sc)):
        lgs = rh.renderLightGroups(j, spp=spp, seed=24, groups=groups)
        assert_oracle(lgs, orc, groups, w, h, sc.max_depth, spp, offsets, (name, groups))
    lgs = rh.renderLightGroups(j, spp=spp, offsets=offsets)  # F64 offsets: the same samples
    assert_oracle(lgs, orc, list(range(n_lights(sc))), w, h, sc.max_depth, spp, offsets, (name, "f64"))


# ---------------------------------------------------------------- 3. bit-for-bit invariance
@pytest.mark.parametrize("name", [n for n in SCENES + list(BUILT) if not has_transparent(scene(n))])
def test_groups_do_not_depend_on_how_the_frame_is_run(name):
    sc = scene(name)
    w, h = SIZES[1]
    j, spp = job(sc, w, h), 2
    ref = rh.renderLightGroups(j, spp=spp, seed=24, shadow="pooled")
    variants = {"split": dict(shadow="split"), "exact_boxes": dict(exact_boxes=True), "no_light_maps": dict(light_maps=False),
                "chunks": dict(chunk_samples=w * spp * 7), "device": dict(device=True), "profile": dict(profile=True),
                "default": dict(), "again": dict(shadow="pooled")}
    for tag, kw in variants.items():
        got = rh.renderLightGroups(j, spp=spp, seed=24, **kw)
        same(got.groups, ref.groups, (name, tag))
        same(got.rest, ref.rest, (name, tag, "rest"))
        same(got.image, ref.image, (name, tag, "image"))
    assert rh.renderLightGroups(j, spp=spp, seed=24, chunk_samples=w * spp * 7).stats["chunks"] > 2
    for G in (2, 4):
        bh = 8
        full_g, full_r = np.zeros_like(ref.groups), np.zeros_like(ref.rest)
        for i in range(G):
            part = rh.renderLightGroups(j, spp=spp, seed=24, shard_index=i, shard_count=G, band_height=bh)
            for lr, row in enumerate(rh.shard_global_rows(h, i, G, bh)):
                if row >= 0:
                    full_g[:, row], full_r[row] = part.groups[:, lr], part.rest[lr]
                else:
                    assert not part.groups[:, lr].any() and not part.rest[lr].any()  # padding rows are 0
        same(full_g, ref.groups, (name, "shards", G))
        same(full_r, ref.rest, (name, "shards", G, "rest"))


def test_device_offsets_and_outputs():
    import torch

    sc = scene("texture")
    w, h = SIZES[0]
    j, spp = job(sc, w, h), 2
    off = f64_offsets(w, h, spp)
    ref = rh.renderLightGroups(j, spp=spp, offsets=off, want_hit_ids=True)
    got = rh.renderLightGroups(j, spp=spp, offsets=torch.from_numpy(off).cuda(), want_hit_ids=True)
    assert got.groups.is_cuda and got.image.is_cuda
    for a, b, what in ((got.groups, ref.groups, "groups"), (got.rest, ref.rest, "rest"), (got.image, ref.image, "image"),
                       (got.hit_ids, ref.hit_ids, "ids"), (got.relight(np.ones((n_lights(sc), 3))), ref.relight(np.ones((n_lights(sc), 3))), "relight")):
        same(a, b, what)


# ---------------------------------------------------------------- 4. relighting
@pytest.mark.parametrize("name", ["cornellBox", "dragon_low"])
def test_relighting_after_a_colour_update(name):
    sc = load_scene(name)  # (a fresh copy: the update changes it)
    w, h = SIZES[0]
    j, spp, L = job(sc, w, h), 2, n_lights(sc)
    old = rh.renderLightGroups(j, spp=spp, seed=24)
    k = np.random.RandomState(9).uniform(0.25, 3.0, (L, 3))
    lights = sc.lights
    for l in range(L):
        for c in range(3):
            lights[l].color[c] *= k[l, c]
    assert sc.update(lights=lights)["colours_only"] == 1
    new = rh.renderLightGroups(j, spp=spp, seed=24)
    for g in range(L):
        assert_close(new.groups[g], k[g] * old.groups[g], (name, "group", g))
    assert_close(new.rest, old.rest, (name, "rest"))
    acc = rh.Accumulator(j, stream_spp=spp)
    a = acc.add(spp, seed=24)
    acc.close()
    assert_close(old.relight(k), a.linear, (name, "relight"))


# ---------------------------------------------------------------- 5. overflow retry, 6. learned state
GROWTH = 1024  # a frame large enough that the queues' per-warp slack is small beside its samples


def test_queue_overflow_retry_keeps_the_oracle_agreement():
    sc = growth_scene()
    w = h = GROWTH
    j = rh.Rendering(sc, sc.camera, w, h, 8)
    lgs = rh.renderLightGroups(j, spp=1, seed=24)
    assert lgs.stats["queue_factor"] > 2, lgs.stats
    assert_oracle(lgs, Oracle(sc), [0], w, h, 8, 1, rh.sample_offsets(w * h, 1, 24), "growth", rows=(5, None, 97))


def test_the_call_leaves_the_scenes_render_state_alone():
    """An overflowing light-groups call, then a render: the render behaves as on a scene that never had the call (same
    bytes, queue factor, shadow schedule and chunks)."""
    small = lambda sc: rh.Rendering(sc, sc.camera, 256, 256, 0)  # noqa: E731
    used, fresh = growth_scene(), growth_scene()
    lgs = rh.renderLightGroups(rh.Rendering(used, used.camera, GROWTH, GROWTH, 8), seed=24)
    assert lgs.stats["queue_factor"] > 2, lgs.stats
    after, ref = rh.render(small(used)), rh.render(small(fresh))
    assert_parity(after.pixels, ref.pixels)  # (Transparent forks: the 1-LSB wobble)
    for k in ("queue_factor", "shadow_split", "chunks", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert after.stats[k] == ref.stats[k], k


# ---------------------------------------------------------------- 7. a non-finite light
@pytest.mark.parametrize("light", ["colour_inf", "colour_nan", "dir_colour_nan"])
def test_a_non_finite_light_stays_in_its_group(light):
    sc = vc.lit_stage(vc.LIGHTS[light])  # light 0 ordinary, light 1 under test
    j = rh.Rendering(sc, sc.camera, sc.width, sc.height, 0)
    lgs = rh.renderLightGroups(j, spp=1, seed=24)
    img = rh.render(j, spp=1, seed=24)
    assert np.array_equal(lgs.image, img.pixels)
    assert not np.isfinite(lgs.groups[1]).all()
    assert np.isfinite(lgs.groups[0]).all() and np.isfinite(lgs.rest).all()
    offsets = rh.sample_offsets(sc.width * sc.height, 1, 24)
    assert_oracle(lgs, Oracle(sc), [0, 1], sc.width, sc.height, 0, 1, offsets, light)


# ---------------------------------------------------------------- 8. argument errors
def test_argument_errors():
    import torch

    sc = scene("cornellBox")
    L = capi.lib()
    w, h, spp = 16, 8, 1
    o = rh.host._opts(job(sc, w, h), spp, capi.RH_OFFSETS_NONE, None, 0, 0, 1, h, 0, 0)
    nl = n_lights(sc)
    out = np.full((3, h, w, 3), 7.0)
    rgb = np.full((h, w, 3), 9, np.uint8)
    good_map = (C.c_uint8 * nl)(*([0] * nl))

    def call(flags=0, n_groups=2, reserved=0, gmap=good_map, out_ptr=None, scene_=None, rgb_ptr=None, ids=None):
        oo = capi.rh_render_opts.from_buffer_copy(o)
        oo.flags = flags
        lg = capi.rh_light_groups()
        lg.group_of_light = C.addressof(gmap) if gmap is not None else None
        lg.n_groups, lg.reserved_ = n_groups, reserved
        lg.out = out.ctypes.data if out_ptr is None else out_ptr
        return L.rh_render_light_groups(scene_ or sc.device, C.byref(sc.camera), C.byref(oo), C.byref(lg),
                                        rgb.ctypes.data if rgb_ptr is None else rgb_ptr, ids, None)

    bad_map = (C.c_uint8 * nl)(*([0] * (nl - 1) + [2]))
    cases = [dict(n_groups=0), dict(n_groups=17), dict(reserved=1), dict(gmap=bad_map), dict(gmap=None), dict(out_ptr=0),
             dict(flags=capi.RH_FLAG_COUNT), dict(flags=capi.RH_FLAG_PEER_FRAMES), dict(flags=capi.RH_FLAG_HIT_IDS)]
    for kw in cases:
        if kw.get("out_ptr") == 0:
            lg = capi.rh_light_groups()
            lg.group_of_light, lg.n_groups = C.addressof(good_map), 2
            rc = L.rh_render_light_groups(sc.device, C.byref(sc.camera), C.byref(o), C.byref(lg), rgb.ctypes.data, None, None)
        else:
            rc = call(**kw)
        assert rc == capi.RH_ERR_ARG, kw
        assert (out == 7.0).all() and (rgb == 9).all(), kw
    assert L.rh_render_light_groups(sc.device, C.byref(sc.camera), C.byref(o), None, rgb.ctypes.data, None, None) == capi.RH_ERR_ARG
    # more than 32 lights
    many = vc.lambert(1, "diffuse", "flat", 40)
    mj = rh.Rendering(many, many.camera, w, h, 0)
    with pytest.raises(capi.RayHsError) as e:
        rh.renderLightGroups(mj, groups=[0] * 40)
    assert e.value.code == capi.RH_ERR_ARG
    # device outputs: host memory and a misaligned device pointer
    D = capi.RH_FLAG_DEVICE_OUT
    t = torch.full((3 * h * w * 3 + 1,), 5.0, dtype=torch.float64, device="cuda")
    r = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
    assert call(flags=D, out_ptr=t.data_ptr() + 4, rgb_ptr=r.data_ptr()) == capi.RH_ERR_ARG
    assert call(flags=D, rgb_ptr=r.data_ptr()) == capi.RH_ERR_ARG
    assert (t == 5.0).all() and (out == 7.0).all()
    assert call(flags=D, out_ptr=t.data_ptr() + 8, rgb_ptr=r.data_ptr()) == capi.RH_OK
    assert call() == capi.RH_OK and (out != 7.0).any() and call(rgb_ptr=0) == capi.RH_OK
