"""CPU characterisation of the host wrappers' argument marshalling (rayhs_b200/host.py) with the library replaced by a
recording fake: for every host-buffer entry point, each rh_render_opts field, the flags, the auxiliary structs, which
array each pointer refers to and the offset values the library reads through it.  Inputs: offsets none / float64 /
float32 / tiled / seed / CPU tensor / strided view, shards, and every boolean keyword.  render_device runs here too
with peer frames (no CUDA framebuffer) and host offsets.

The rejection tests hold the wrappers to what the library needs: offsets of exactly the expected number of values, a
dense copy of a strided view, offsets or a seed but not both, and CUDA offsets only where the call takes them."""
import ctypes as C
from types import SimpleNamespace
from unittest.mock import ANY

import numpy as np
import pytest
import torch

import rayhs_b200 as rh
from rayhs_b200 import capi, host

W, H, D = 10, 6, 3
F64, F32, TILED, SEED, NONE = (capi.RH_OFFSETS_F64, capi.RH_OFFSETS_F32, capi.RH_OFFSETS_TILED_F64, capi.RH_OFFSETS_SPLITMIX64,
                               capi.RH_OFFSETS_NONE)


def _offset_values(o):
    """What the library reads through rh_render_opts.offsets: the seed, or the float values of the full frame / tile."""
    if o.offset_mode == SEED:
        return C.c_uint64.from_address(o.offsets).value
    if o.offset_mode == NONE:
        return None
    n = (o.offset_tile * o.offset_tile if o.offset_mode == TILED else o.width * o.height) * o.spp * 2
    ctype = C.c_float if o.offset_mode == F32 else C.c_double
    return np.ctypeslib.as_array((ctype * n).from_address(o.offsets)).copy()


def _opts(opts):
    o = opts._obj
    rec = {f: getattr(o, f) for f, _ in capi.rh_render_opts._fields_}
    rec["peer_frames"] = [o.peer_frames[i] for i in range(o.n_peer_frames)] if o.n_peer_frames else None
    return rec


class _FakeLib:
    """Stands in for librayhs_b200.so: records every call with the structs it was given and what the pointers hold."""

    def __init__(self):
        self.calls, self.gpus, self.handles = [], 0, 0x1000

    def _rec(self, fn, stats=None, **kw):
        self.calls.append(dict(fn=fn, **kw))
        if stats is not None:
            stats._obj.rays_primary = 7
        return 0

    def _handle(self, out):
        self.handles += 16
        out._obj.value = self.handles
        return self.handles

    def rh_init(self, device):
        return 0

    def rh_default_band_height(self, h, g):
        return h if g <= 1 else 4

    def rh_shard_rows(self, h, g, bh):
        return ((h + bh - 1) // bh + g - 1) // g * bh

    def rh_render(self, scene, cam, opts, rgb, ids, stats):
        return self._rec("rh_render", stats, scene=scene, camera=cam._obj, opts=_opts(opts), values=_offset_values(opts._obj),
                         rgb=rgb, ids=ids)

    def rh_render_features(self, scene, cam, opts, ft, ids, stats):
        f = ft._obj
        return self._rec("rh_render_features", stats, scene=scene, camera=cam._obj, opts=_opts(opts),
                         values=_offset_values(opts._obj), ft={n: getattr(f, n) for n, _ in f._fields_}, ids=ids)

    def rh_render_light_groups(self, scene, cam, opts, lg, rgb, ids, stats):
        g = lg._obj
        return self._rec("rh_render_light_groups", stats, scene=scene, camera=cam._obj, opts=_opts(opts),
                         values=_offset_values(opts._obj), map=list((C.c_uint8 * 3).from_address(g.group_of_light)),
                         n_groups=g.n_groups, reserved=g.reserved_, out=g.out, rgb=rgb, ids=ids)

    def rh_accum_create(self, w, h, si, sc, bh, stream_spp, out):
        return self._rec("rh_accum_create", args=(w, h, si, sc, bh, stream_spp), handle=self._handle(out))

    def rh_render_accumulate(self, scene, cam, opts, acc, rgb, lin, ids, stats):
        return self._rec("rh_render_accumulate", stats, scene=scene, camera=cam._obj, opts=_opts(opts),
                         values=_offset_values(opts._obj), handle=acc.value, rgb=rgb, lin=lin, ids=ids)

    def rh_accum_reset(self, acc):
        return self._rec("rh_accum_reset", handle=acc.value)

    def rh_accum_destroy(self, acc):
        self._rec("rh_accum_destroy", handle=acc.value)

    def rh_adaptive_create(self, w, h, si, sc, bh, stream_spp, out):
        return self._rec("rh_adaptive_create", args=(w, h, si, sc, bh, stream_spp), handle=self._handle(out))

    def rh_render_adaptive(self, scene, cam, opts, ao, ad, rgb, lin, n_active, stats):
        a = ao._obj
        n_active._obj.value = 5
        return self._rec("rh_render_adaptive", stats, scene=scene, camera=cam._obj, opts=_opts(opts),
                         values=_offset_values(opts._obj), ao=(a.threshold, a.min_spp, a.reserved_), handle=ad.value, rgb=rgb,
                         lin=lin)

    def rh_adaptive_state(self, ad, counts, sums, sumsq, flags):
        return self._rec("rh_adaptive_state", handle=ad.value, ptrs=(counts, sums, sumsq), flags=flags)

    def rh_adaptive_reset(self, ad):
        return self._rec("rh_adaptive_reset", handle=ad.value)

    def rh_adaptive_destroy(self, ad):
        self._rec("rh_adaptive_destroy", handle=ad.value)

    def _rays(self, rays, n):
        return np.ctypeslib.as_array((C.c_double * (6 * n)).from_address(rays)).reshape(n, 6).copy()

    def rh_closest_intersection(self, scene, rays, n, rec, flags):
        return self._rec("rh_closest_intersection", scene=scene, rays=self._rays(rays, n), n=n, out=rec, flags=flags)

    def rh_shadow_intersection(self, scene, light, rays, n, out, flags):
        return self._rec("rh_shadow_intersection", scene=scene, light=light, rays=self._rays(rays, n), n=n, out=out, flags=flags)

    def rh_trace_rays(self, scene, rays, n, opts, colors, ids, stats):
        o = opts._obj
        return self._rec("rh_trace_rays", stats, scene=scene, rays=self._rays(rays, n), n=n,
                         opts=(o.max_depth, o.flags, o.chunk_rays, o.reserved_), colors=colors, ids=ids)

    def rh_multi_gpu_count(self):
        return self.gpus

    def rh_multi_init(self, n):
        self.gpus = n
        return self._rec("rh_multi_init", n=n)

    def rh_multi_scene_create(self, flat, out):
        return self._rec("rh_multi_scene_create", flat=flat, handle=self._handle(out))

    def rh_multi_render(self, ms, cam, opts, rgb, stats):
        return self._rec("rh_multi_render", stats, handle=ms.value, camera=cam._obj, opts=_opts(opts),
                         values=_offset_values(opts._obj), rgb=rgb)


class _Scene:
    device, flat = "scene-handle", "flat-desc"
    raw = SimpleNamespace(contents=SimpleNamespace(n_lights=3))


@pytest.fixture
def fake(monkeypatch):
    L = _FakeLib()
    monkeypatch.setattr(host, "lib", lambda: L)
    monkeypatch.setattr(host, "_initialised", False)
    return L


@pytest.fixture
def job():
    return host.Rendering(_Scene(), capi.rh_camera(), W, H, D)


def opts(**kw):
    """The rh_render_opts a call of the full frame without shards, offsets or flags passes, with `kw` changed."""
    o = dict(width=W, height=H, max_depth=D, spp=1, offset_mode=NONE, offset_tile=0, offsets=None, shard_index=0, shard_count=1,
             band_height=H, chunk_samples=0, flags=0, n_peer_frames=0, peer_frames=None)
    o.update(kw)
    return o


def _values(n, spp, dtype=np.float64, seed=0):
    return np.random.RandomState(seed).uniform(-0.5, 0.5, (n, spp, 2)).astype(dtype)


def source(kind, spp, tile=3):
    """(keyword arguments, expected opts fields, expected values read) of one sample source of `spp` samples per pixel."""
    if kind == "none":
        return {}, dict(offset_mode=NONE), None
    if kind == "seed":
        return dict(seed=77), dict(offset_mode=SEED, offsets=ANY), 77
    if kind == "tiled":
        a = _values(tile * tile, spp)
        return dict(offsets=a, offset_tile=tile), dict(offset_mode=TILED, offset_tile=tile, offsets=a.ctypes.data), a.ravel()
    dtype = np.float32 if kind == "f32" else np.float64
    a = _values(W * H, spp, dtype)
    if kind == "tensor":
        t = torch.from_numpy(a)
        return dict(offsets=t), dict(offset_mode=F64, offsets=t.data_ptr()), a.ravel()
    return dict(offsets=a), dict(offset_mode=F32 if kind == "f32" else F64, offsets=a.ctypes.data), a.ravel()


def assert_values(got, want):
    if want is None or isinstance(want, int):
        assert got == want
    else:
        assert got.dtype == want.dtype and np.array_equal(got, want)


KEYWORDS = {
    "want_hit_ids": (dict(want_hit_ids=True), capi.RH_FLAG_HIT_IDS),
    "count": (dict(count=True), capi.RH_FLAG_COUNT),
    "profile": (dict(profile=True), capi.RH_FLAG_PROFILE),
    "exact_boxes": (dict(exact_boxes=True), capi.RH_FLAG_EXACT_BOXES),
    "no_light_maps": (dict(light_maps=False), capi.RH_FLAG_NO_LIGHT_MAPS),
    "pooled": (dict(shadow="pooled"), capi.RH_FLAG_SHADOW_POOLED),
    "split": (dict(shadow="split"), capi.RH_FLAG_SHADOW_SPLIT),
}


def keyword_cases(*names):
    """One case per keyword, none, and all of them at once (with 'split' for the shadow schedule)."""
    cases = [pytest.param({}, 0, id="none")] + [pytest.param(*KEYWORDS[n], id=n) for n in names]
    kw, flags = {}, 0
    for n in names:
        if n != "pooled":
            kw.update(KEYWORDS[n][0])
            flags |= KEYWORDS[n][1]
    return cases + [pytest.param(kw, flags, id="all")]


SHARDS = [pytest.param({}, (0, 1, H), H, id="whole"), pytest.param(dict(shard_index=1, shard_count=2, band_height=2), (1, 2, 2), 4, id="bh2"),
          pytest.param(dict(shard_index=1, shard_count=2), (1, 2, 4), 4, id="default_bh")]


def shard_opts(shard):
    return dict(shard_index=shard[0], shard_count=shard[1], band_height=shard[2])


# ---------------------------------------------------------------- render (host buffers)
@pytest.mark.parametrize("kind", ["none", "f64", "f32", "tiled", "seed", "tensor"])
def test_render_sources(fake, job, kind):
    kw, want, values = source(kind, 2)
    img = rh.render(job, spp=2, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=2, **want)
    assert_values(c["values"], values)
    assert c["scene"] == "scene-handle" and c["camera"] is job.camera
    assert img.pixels.shape == (H, W, 3) and img.pixels.dtype == np.uint8 and c["rgb"] == img.pixels.ctypes.data
    assert img.hit_ids is None and c["ids"] is None and img.stats["rays_primary"] == 7 and (img.width, img.height) == (W, H)


@pytest.mark.parametrize("kw,flags", keyword_cases(*KEYWORDS))
def test_render_keywords(fake, job, kw, flags):
    img = rh.render(job, spp=3, chunk_samples=40, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=3, chunk_samples=40, flags=flags)
    if kw.get("want_hit_ids"):
        assert img.hit_ids.shape == (H, W, 3, 2) and img.hit_ids.dtype == np.int32 and c["ids"] == img.hit_ids.ctypes.data
    else:
        assert img.hit_ids is None and c["ids"] is None


@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_render_shards_and_out(fake, job, kw, shard, rows):
    out = np.empty((rows, W, 3), dtype=np.uint8)
    img = rh.render(job, out=out, want_hit_ids=True, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(flags=capi.RH_FLAG_HIT_IDS, **shard_opts(shard))
    assert img.pixels is out and c["rgb"] == out.ctypes.data and img.height == rows and img.hit_ids.shape == (rows, W, 1, 2)


# ---------------------------------------------------------------- render_multi
@pytest.mark.parametrize("kind", ["none", "f64", "f32", "seed", "tensor"])
@pytest.mark.parametrize("kw,flags", keyword_cases("pooled", "split"))
def test_render_multi(fake, job, kind, kw, flags):
    src, want, values = source(kind, 2)
    img = rh.render_multi(job, 4, spp=2, band_height=3, **src, **kw)
    init, create, c = fake.calls
    assert init == dict(fn="rh_multi_init", n=4) and create == dict(fn="rh_multi_scene_create", flat="flat-desc", handle=c["handle"])
    assert c["opts"] == opts(spp=2, band_height=3, flags=flags, **want)  # band_height 0: the library's choice
    assert_values(c["values"], values)
    assert c["camera"] is job.camera and c["rgb"] == img.pixels.ctypes.data and img.pixels.shape == (H, W, 3)
    rh.render_multi(job, 4)  # the context and the replicated scene are made once
    assert [x["fn"] for x in fake.calls[3:]] == ["rh_multi_render"] and fake.calls[-1]["opts"]["band_height"] == 0


# ---------------------------------------------------------------- render_device (peer frames: no CUDA framebuffer needed)
@pytest.mark.parametrize("kind", ["none", "f64", "f32", "tiled", "seed", "tensor"])
@pytest.mark.parametrize("kw,flags", keyword_cases("count", "profile", "no_light_maps", "pooled", "split"))
def test_render_device_with_host_offsets(fake, job, kind, kw, flags):
    src, want, values = source(kind, 2)
    if "offsets" in src:
        src = dict(offsets_dev=torch.as_tensor(src.pop("offsets")), **src)
        want["offsets"] = src["offsets_dev"].data_ptr()
    st = rh.render_device(job, None, spp=2, chunk_samples=8, peer_frames=[0x7000, 0x8000], **src, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=2, chunk_samples=8, n_peer_frames=2, peer_frames=[0x7000, 0x8000],
                             flags=flags | capi.RH_FLAG_DEVICE_OUT | capi.RH_FLAG_PEER_FRAMES, **want)
    assert_values(c["values"], values)
    assert c["rgb"] is None and c["ids"] is None and st["rays_primary"] == 7


@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_render_device_shard_offsets_and_hit_ids(fake, job, kw, shard, rows):
    off = torch.from_numpy(_values(rows * W, 2))
    ids = torch.empty((rows * W * 2, 2), dtype=torch.int32)
    rh.render_device(job, None, spp=2, offsets_dev=off, shard_offsets=True, hit_ids_dev=ids, peer_frames=[0x7000], **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=2, offset_mode=F64, offsets=off.data_ptr(), n_peer_frames=1, peer_frames=[0x7000],
                             flags=capi.RH_FLAG_DEVICE_OUT | capi.RH_FLAG_SHARD_OFFSETS | capi.RH_FLAG_HIT_IDS | capi.RH_FLAG_PEER_FRAMES,
                             **shard_opts(shard))
    assert c["ids"] == ids.data_ptr()


# ---------------------------------------------------------------- renderFeatures
@pytest.mark.parametrize("kind", ["none", "f64", "f32", "tiled", "seed", "tensor"])
@pytest.mark.parametrize("kw,flags", keyword_cases("want_hit_ids", "exact_boxes"))
def test_render_features(fake, job, kind, kw, flags):
    src, want, values = source(kind, 2)
    if kind == "seed":
        src.update(stream_spp=8, stream_base=6)
    fe = rh.renderFeatures(job, spp=2, **src, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=2, flags=flags, **want)
    assert_values(c["values"], values)
    assert c["ft"] == dict(albedo=fe.albedo.ctypes.data, normal=fe.normal.ctypes.data, depth=fe.depth.ctypes.data,
                           hits=fe.hits.ctypes.data, stream_spp=8 if kind == "seed" else 0, stream_base=6 if kind == "seed" else 0)
    assert fe.albedo.shape == fe.normal.shape == (H, W, 3) and fe.depth.shape == fe.hits.shape == (H, W)
    assert fe.albedo.dtype == fe.normal.dtype == fe.depth.dtype == np.float64 and fe.hits.dtype == np.uint32
    assert (c["ids"] == fe.hit_ids.ctypes.data and fe.hit_ids.shape == (H, W, 2, 2)) if kw.get("want_hit_ids") else c["ids"] is None
    assert fe.stats["rays_primary"] == 7


@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_render_features_shards(fake, job, kw, shard, rows):
    fe = rh.renderFeatures(job, **kw)
    assert fake.calls[-1]["opts"] == opts(**shard_opts(shard)) and fe.albedo.shape == (rows, W, 3)


# ---------------------------------------------------------------- renderLightGroups
@pytest.mark.parametrize("kind", ["none", "f64", "f32", "seed", "tensor"])
@pytest.mark.parametrize("kw,flags", keyword_cases("want_hit_ids", "exact_boxes", "profile", "no_light_maps", "pooled", "split"))
def test_render_light_groups(fake, job, kind, kw, flags):
    src, want, values = source(kind, 2)
    lgs = rh.renderLightGroups(job, spp=2, groups=[1, 0, 1], chunk_samples=24, **src, **kw)
    (c,) = fake.calls
    assert c["opts"] == opts(spp=2, chunk_samples=24, flags=flags, **want)
    assert_values(c["values"], values)
    assert c["map"] == [1, 0, 1] and c["n_groups"] == 2 and c["reserved"] == 0
    assert lgs.groups.shape == (2, H, W, 3) and lgs.rest.shape == (H, W, 3) and c["out"] == lgs.groups.ctypes.data
    assert lgs.image.shape == (H, W, 3) and lgs.image.dtype == np.uint8 and c["rgb"] == lgs.image.ctypes.data
    assert (c["ids"] == lgs.hit_ids.ctypes.data) if kw.get("want_hit_ids") else (c["ids"] is None and lgs.hit_ids is None)


@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_render_light_groups_shards(fake, job, kw, shard, rows):
    lgs = rh.renderLightGroups(job, rgb=False, **kw)
    c = fake.calls[-1]
    assert c["opts"] == opts(**shard_opts(shard)) and c["rgb"] is None and lgs.image is None
    assert lgs.groups.shape == (3, rows, W, 3)


# ---------------------------------------------------------------- Accumulator
@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_accumulator_lifetime_and_shards(fake, job, kw, shard, rows):
    acc = rh.Accumulator(job, stream_spp=12, **kw)
    create = fake.calls[0]
    assert create["fn"] == "rh_accum_create" and create["args"] == (W, H, shard[0], shard[1], shard[2], 12)
    assert (acc.shard_index, acc.shard_count, acc.band_height, acc.rows, acc.device) == shard + (rows, False)
    img = acc.add(2, seed=5)
    c = fake.calls[-1]
    assert c["opts"] == opts(spp=2, offset_mode=SEED, offsets=ANY, **shard_opts(shard)) and c["handle"] == create["handle"]
    assert img.pixels.shape == img.linear.shape == (rows, W, 3) and acc.samples == 2
    acc.reset()
    assert fake.calls[-1] == dict(fn="rh_accum_reset", handle=create["handle"]) and acc.samples == 0
    acc.close()
    assert fake.calls[-1] == dict(fn="rh_accum_destroy", handle=create["handle"])
    acc.close()
    assert fake.calls[-1]["fn"] == "rh_accum_destroy" and len(fake.calls) == 4
    with pytest.raises(ValueError):
        acc.add(1)


@pytest.mark.parametrize("kind", ["none", "f64", "f32", "seed", "tensor"])
@pytest.mark.parametrize("kw,flags", keyword_cases("want_hit_ids", "exact_boxes", "profile", "no_light_maps", "pooled", "split"))
def test_accumulator_add(fake, job, kind, kw, flags):
    acc = rh.Accumulator(job, stream_spp=8)
    src, want, values = source(kind, 2)
    img = acc.add(2, chunk_samples=16, **src, **kw)
    c = fake.calls[-1]
    assert c["opts"] == opts(spp=2, chunk_samples=16, flags=flags, **want)
    assert_values(c["values"], values)
    assert c["rgb"] == img.pixels.ctypes.data and c["lin"] == img.linear.ctypes.data
    assert img.pixels.dtype == np.uint8 and img.linear.dtype == np.float64 and img.stats["rays_primary"] == 7
    assert (c["ids"] == img.hit_ids.ctypes.data and img.hit_ids.shape == (H, W, 2, 2)) if kw.get("want_hit_ids") else c["ids"] is None
    img = acc.add(1, rgb=False, linear=False)
    assert fake.calls[-1]["rgb"] is None and fake.calls[-1]["lin"] is None and img.pixels is None and img.linear is None
    assert acc.samples == 3
    acc.close()


# ---------------------------------------------------------------- AdaptiveAccumulator
@pytest.mark.parametrize("kw,shard,rows", SHARDS)
def test_adaptive_lifetime_shards_and_state(fake, job, kw, shard, rows):
    ad = rh.AdaptiveAccumulator(job, stream_spp=32, **kw)
    create = fake.calls[0]
    assert create["fn"] == "rh_adaptive_create" and create["args"] == (W, H, shard[0], shard[1], shard[2], 32)
    assert (ad.shard_index, ad.shard_count, ad.band_height, ad.rows, ad.stream_spp, ad.device) == shard + (rows, 32, False)
    counts, sums, sumsq = ad.state()
    c = fake.calls[-1]
    assert c == dict(fn="rh_adaptive_state", handle=create["handle"], ptrs=(counts.ctypes.data, sums.ctypes.data, sumsq.ctypes.data),
                     flags=0)
    assert counts.shape == (rows, W) and counts.dtype == np.uint32 and sums.shape == sumsq.shape == (rows, W, 3)
    assert sums.dtype == sumsq.dtype == np.float64
    ad.reset()
    assert fake.calls[-1] == dict(fn="rh_adaptive_reset", handle=create["handle"])
    ad.close()
    assert fake.calls[-1] == dict(fn="rh_adaptive_destroy", handle=create["handle"])
    ad.close()
    assert len(fake.calls) == 4
    with pytest.raises(ValueError):
        ad.add(1, 24, 0.1)


@pytest.mark.parametrize("kw,flags", keyword_cases("count", "exact_boxes", "profile", "no_light_maps", "pooled", "split"))
def test_adaptive_add(fake, job, kw, flags):
    ad = rh.AdaptiveAccumulator(job, stream_spp=32)
    img = ad.add(4, 99, 0.25, min_spp=6, chunk_samples=12, **kw)
    c = fake.calls[-1]
    assert c["opts"] == opts(spp=4, offset_mode=SEED, offsets=ANY, chunk_samples=12, flags=flags) and c["values"] == 99
    assert c["ao"] == (0.25, 6, 0) and c["handle"] == fake.calls[0]["handle"]
    assert c["rgb"] == img.pixels.ctypes.data and c["lin"] == img.linear.ctypes.data and img.pixels.shape == img.linear.shape == (H, W, 3)
    assert img.stats["n_active"] == 5 and img.stats["rays_primary"] == 7 and img.hit_ids is None
    img = ad.add(4, 99, 0.25, rgb=False, linear=False)
    assert fake.calls[-1]["rgb"] is None and fake.calls[-1]["lin"] is None and img.pixels is None and img.linear is None
    ad.close()


# ---------------------------------------------------------------- ray and radiance queries
RAYS_O = np.arange(12, dtype=np.float64).reshape(4, 3)
RAYS_D = -np.arange(12, dtype=np.float64).reshape(4, 3) - 1


@pytest.mark.parametrize("kw,flags", keyword_cases("exact_boxes"))
def test_closest_intersection(fake, kw, flags):
    hits = rh.closestIntersection(_Scene(), RAYS_O, RAYS_D, **kw)
    (c,) = fake.calls
    assert c["scene"] == "scene-handle" and c["n"] == 4 and c["flags"] == flags
    assert np.array_equal(c["rays"], np.concatenate([RAYS_O, RAYS_D], axis=1))
    assert c["out"] == hits.records.ctypes.data and hits.records.dtype == host.HIT_DTYPE and hits.records.shape == (4,)
    assert hits.t.shape == (4,) and hits.p.shape == hits.n.shape == (4, 3) and hits.uv.shape == (4, 2) and hits.tri.dtype == np.int32


@pytest.mark.parametrize("kw,flags", keyword_cases("exact_boxes"))
def test_shadow_intersection(fake, kw, flags):
    occluded = rh.shadowIntersection(_Scene(), 2, RAYS_O, RAYS_D, **kw)
    (c,) = fake.calls
    assert c["scene"] == "scene-handle" and c["light"] == 2 and c["n"] == 4 and c["flags"] == flags
    assert np.array_equal(c["rays"], np.concatenate([RAYS_O, RAYS_D], axis=1))
    assert c["out"] == occluded.ctypes.data and occluded.dtype == np.bool_ and occluded.shape == (4,)


@pytest.mark.parametrize("kw,flags", keyword_cases("want_hit_ids", "exact_boxes", "no_light_maps", "pooled", "split"))
def test_trace_ray(fake, kw, flags):
    r = rh.traceRay(_Scene(), RAYS_O, RAYS_D, 5, chunk_rays=3, **kw)
    (c,) = fake.calls
    assert c["scene"] == "scene-handle" and c["n"] == 4 and c["opts"] == (5, flags, 3, 0)
    assert np.array_equal(c["rays"], np.concatenate([RAYS_O, RAYS_D], axis=1))
    assert c["colors"] == r.colors.ctypes.data and r.colors.shape == (4, 3) and r.colors.dtype == np.float64
    assert (c["ids"] == r.hit_ids.ctypes.data and r.hit_ids.shape == (4, 2)) if kw.get("want_hit_ids") else c["ids"] is None
    assert r.stats["rays_primary"] == 7


# ---------------------------------------------------------------- what every entry point rejects before the library
class _CudaLike:
    """Looks like a dense CUDA float64 tensor to the host layer; its memory is a host array, so a wrapper that passes
    it on anyway hands the fake a readable pointer."""
    is_cuda = True

    def __init__(self, a):
        self._a, self.dtype, self.shape = a, torch.float64, a.shape

    def numel(self):
        return self._a.size

    def data_ptr(self):
        return self._a.ctypes.data

    def contiguous(self):
        return self


def _short(spp):
    """A dense float64 array two values short of a full frame of `spp` samples, inside a larger buffer (so that a
    wrapper that passes it on anyway hands the fake a readable pointer)."""
    return np.zeros(2 * W * H * spp * 2)[:W * H * spp * 2 - 2]


def _calls(job):
    """Each entry point that takes offsets or a seed, as f(**source)."""
    acc = rh.Accumulator(job)
    return {"render": lambda **kw: rh.render(job, spp=2, **kw),
            "render_multi": lambda **kw: rh.render_multi(job, 2, spp=2, **kw),
            "render_device": lambda offsets=None, **kw: rh.render_device(job, None, spp=2, offsets_dev=offsets, peer_frames=[1], **kw),
            "renderFeatures": lambda **kw: rh.renderFeatures(job, spp=2, **kw),
            "renderLightGroups": lambda **kw: rh.renderLightGroups(job, spp=2, **kw),
            "Accumulator.add": lambda **kw: acc.add(2, **kw)}


ENTRY_POINTS = ["render", "render_multi", "render_device", "renderFeatures", "renderLightGroups", "Accumulator.add"]


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_offsets_with_seed_are_rejected(fake, job, name):
    call = _calls(job)[name]
    n = len(fake.calls)
    with pytest.raises(ValueError, match="either offsets or seed"):
        call(offsets=torch.from_numpy(_values(W * H, 2)), seed=3)
    assert len(fake.calls) == n


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_a_short_offsets_array_is_rejected(fake, job, name):
    call = _calls(job)[name]
    n = len(fake.calls)
    with pytest.raises(ValueError, match="values, expected"):
        call(offsets=torch.from_numpy(_short(2)))
    assert len(fake.calls) == n


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_a_strided_view_is_read_dense(fake, job, name):
    """samples 1 .. 2 of a wider stream, stream[:, 1:3], reach the library as a dense copy of the view."""
    call = _calls(job)[name]
    for wide in (_values(W * H, 4), torch.from_numpy(_values(W * H, 4, seed=1))):
        call(offsets=wide[:, 1:3])
        c = fake.calls[-1]
        assert c["opts"]["offset_mode"] == F64
        assert_values(c["values"], np.ascontiguousarray(np.asarray(wide)[:, 1:3]).ravel())


@pytest.mark.parametrize("name", ["render", "render_device", "renderFeatures"])
def test_a_short_tile_is_rejected(fake, job, name):
    call = _calls(job)[name]
    n = len(fake.calls)
    with pytest.raises(ValueError, match="values, expected"):
        call(offsets=torch.zeros(2 * 9 * 2 * 2, dtype=torch.float64)[:8 * 2 * 2], offset_tile=3)
    assert len(fake.calls) == n


def test_shard_offsets_hold_the_shard_rows(fake, job):
    """render_device(shard_offsets=True) reads this shard's rows only: rows * width samples, not the full frame's."""
    full = torch.from_numpy(_values(W * H, 2))
    with pytest.raises(ValueError, match="values, expected"):
        rh.render_device(job, None, spp=2, offsets_dev=full, shard_offsets=True, shard_index=1, shard_count=2, band_height=2,
                         peer_frames=[1])
    assert not fake.calls


@pytest.mark.parametrize("name", ["render", "render_multi", "renderFeatures", "Accumulator.add"])
def test_cuda_offsets_need_a_call_with_device_outputs(fake, job, name):
    """render and render_multi take host offsets only (render_device takes CUDA ones); renderFeatures and a host
    Accumulator write host outputs, so CUDA offsets are an error there too."""
    call = _calls(job)[name]
    n = len(fake.calls)
    with pytest.raises(ValueError, match="CUDA offsets"):
        call(offsets=_CudaLike(_values(W * H, 2)))
    assert len(fake.calls) == n


def test_unknown_shadow_schedule_is_rejected(fake, job):
    with pytest.raises(KeyError):
        rh.render(job, shadow="both")
    assert not fake.calls
