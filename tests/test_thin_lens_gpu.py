"""GPU tests of the thin-lens camera (RH_PROJ_THIN_LENS): rh_render of lens cameras on every pack against the oracle's
render (tests/lens_oracle.py: bytes, linear colours, hit ids and ray counts) at two apertures and two focus distances; every offset mode, host
and device, and shard-compact offsets; radius 0 against the perspective frame in rh_render, rh_render_views and
rh_render_features; each entry point against its own definition with lens cameras (progressive slices, adaptive pixels,
features, light groups, views that mix the three projections with per-view seeds, rh_multi_render); bad lens
arguments."""
import ctypes as C
import math

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from rayhs_b200 import capi
from tests import lens_oracle, test_features_gpu
from tests.test_features_gpu import assert_same, expected
from tests.test_trace_rays_gpu import has_transparent
from tests.util import SCENES, assert_oracle_exact, assert_parity, load_scene, render_linear

pytestmark = pytest.mark.gpu

W, H, SPP, SEED = 40, 24, 4, 24
RAYS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
TILE = 5
_cache = {}


def scene(name):
    if name not in _cache:
        sc = load_scene(name)
        _cache[name] = (sc, OracleScene(sc.raw))
    return _cache[name]


def lens(sc, aperture, focus):
    """A thin lens on the scene's camera: aperture and focus distance as fractions of the distance from the position to
    the target (a perspective fovy of 1 when the scene's camera has none)."""
    c = sc.camera
    dist = math.dist(c.position, c.target)
    cam = rh.thinLens(c, aperture * dist, focus * dist)
    if not cam.fovy > 0:
        cam.fovy = 1.0
    return cam


def job(sc, cam, w=W, h=H):
    return rh.Rendering(sc, cam, w, h, sc.max_depth)


def full_offsets(w, h, spp, mode, rng):
    """(keyword arguments of render, the float64 full-frame offsets the oracle takes) of one offset mode."""
    if mode == "none":
        return {}, None
    if mode == "splitmix":
        return dict(seed=SEED), rh.sample_offsets(w * h, spp, SEED)
    f64 = rng.uniform(-0.5, 0.5, (w * h, spp, 2))
    if mode == "f64":
        return dict(offsets=f64), f64
    if mode == "f32":
        f32 = f64.astype(np.float32)
        return dict(offsets=f32), f32.astype(np.float64)
    tile = rng.uniform(-0.5, 0.5, (TILE * TILE, spp, 2))
    rows, cols = np.divmod(np.arange(w * h), w)
    return dict(offsets=tile, offset_tile=TILE), tile[(rows % TILE) * TILE + cols % TILE]


def assert_render_is_the_oracles(sc, orc, cam, img, w, h, spp, offsets, what):
    ref = lens_oracle.render(orc, cam, w, h, sc.max_depth, spp=spp, offsets=offsets)
    assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"]), what
    assert_oracle_exact(img.pixels, img.linear, ref, str(what))
    got = tuple(img.stats[k] for k in RAYS)
    want = tuple(ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow"))
    assert got == want, (what, got, want)


def same(sc, a, b, what):
    """Two frames of one render: bit for bit, or within the 1-LSB wobble of a Transparent scene's forks (DESIGN §3)."""
    a, b = np.asarray(a), np.asarray(b)
    if has_transparent(sc) and a.dtype == np.uint8:
        assert_parity(a, b, str(what))
    else:
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), (what, int((a != b).sum()))


# ---------------------------------------------------------------- 1. every pack against the oracle
@pytest.mark.parametrize("name", SCENES)
def test_lens_renders_equal_the_oracle(name):
    sc, orc = scene(name)
    blurred = 0
    for aperture in (0.02, 0.15):
        for focus in (0.6, 1.0):
            cam = lens(sc, aperture, focus)
            img = render_linear(job(sc, cam), spp=SPP, seed=SEED)
            assert_render_is_the_oracles(sc, orc, cam, img, W, H, SPP, rh.sample_offsets(W * H, SPP, SEED), (name, aperture, focus))
            pin = render_linear(job(sc, sc.camera), spp=SPP, seed=SEED)
            blurred += int((img.pixels != pin.pixels).any())
    assert blurred >= 2, name  # (the lens changes the picture)


# ---------------------------------------------------------------- 2. every offset mode, host and device, shard offsets
@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "texture"])
def test_every_offset_mode(name):
    import torch

    sc, orc = scene(name)
    cam = lens(sc, 0.1, 0.8)
    j = job(sc, cam)
    rng = np.random.RandomState(5)
    for mode in ("none", "f64", "f32", "tiled", "splitmix"):
        spp = 1 if mode == "none" else SPP
        kw, off = full_offsets(W, H, spp, mode, rng)
        # (progressive rendering takes no tile: its frame of the tiled mode reads the tiles expanded to the full frame)
        img = render_linear(j, spp=spp, **(dict(offsets=off) if mode == "tiled" else kw))
        assert_render_is_the_oracles(sc, orc, cam, img, W, H, spp, off, (name, mode))
        plain = rh.render(j, spp=spp, want_hit_ids=True, **kw)
        same(sc, plain.pixels, img.pixels, (name, mode, "rh_render"))
        assert np.array_equal(plain.hit_ids, img.hit_ids), (name, mode)
        # device offsets (or the seed) and a device frame
        dkw = {k: (torch.from_numpy(v).cuda() if k == "offsets" else v) for k, v in kw.items()}
        if "offsets" in dkw:
            dkw["offsets_dev"] = dkw.pop("offsets")
        rgb = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda")
        ids = torch.zeros((H * W * spp, 2), dtype=torch.int32, device="cuda")
        st = rh.render_device(j, rgb, spp=spp, hit_ids_dev=ids, **dkw)
        same(sc, rgb.cpu().numpy(), img.pixels, (name, mode, "device"))
        assert np.array_equal(ids.cpu().numpy().reshape(img.hit_ids.shape), img.hit_ids), (name, mode, "device ids")
        assert tuple(st[k] for k in RAYS) == tuple(img.stats[k] for k in RAYS), (name, mode)
    # shard-compact offsets, host and device, G = 1, 2 and 4 bands assembled
    f64 = rng.uniform(-0.5, 0.5, (W * H, SPP, 2))
    want = render_linear(j, spp=SPP, offsets=f64)
    assert_render_is_the_oracles(sc, orc, cam, want, W, H, SPP, f64, (name, "shards"))
    full = f64.reshape(H, W, SPP, 2)
    for G in (1, 2, 4):
        bh = 4
        for on_device in (False, True):
            parts = []
            for g in range(G):
                gl = rh.shard_global_rows(H, g, G, bh)
                compact = np.full((len(gl), W, SPP, 2), 0.25)
                for lr, row in enumerate(gl):
                    if row >= 0:
                        compact[lr] = full[row]
                t = torch.from_numpy(compact.reshape(-1, SPP, 2))
                rgb = torch.zeros((len(gl), W, 3), dtype=torch.uint8, device="cuda")
                rh.render_device(j, rgb, spp=SPP, offsets_dev=t.cuda() if on_device else t.pin_memory(), shard_index=g, shard_count=G,
                                 band_height=bh, shard_offsets=True)
                parts.append(rgb.cpu().numpy())
            same(sc, rh.assemble_bands(parts, H, bh), want.pixels, (name, G, on_device))


# ---------------------------------------------------------------- 3. radius 0 is the perspective camera
@pytest.mark.parametrize("name", ["dragon_low", "outScene", "texture"])
def test_radius_zero_is_the_perspective_frame(name):
    sc, _ = scene(name)
    zero = lens(sc, 0.0, 0.7)
    persp = sc.camera
    a = rh.render(job(sc, zero), spp=SPP, seed=SEED, want_hit_ids=True)
    b = rh.render(job(sc, persp), spp=SPP, seed=SEED, want_hit_ids=True)
    assert a.pixels.tobytes() == b.pixels.tobytes() and a.hit_ids.tobytes() == b.hit_ids.tobytes(), name
    for k in RAYS + ("shadow_walk_pairs", "shadow_tasks"):
        assert a.stats[k] == b.stats[k], (name, k)
    va = rh.renderViews(job(sc, persp), [zero, persp], spp=SPP, seed=SEED, linear=True, want_hit_ids=True)
    assert va.pixels[0].tobytes() == va.pixels[1].tobytes() == b.pixels.tobytes(), name
    assert va.linear[0].tobytes() == va.linear[1].tobytes() and va.hit_ids[0].tobytes() == va.hit_ids[1].tobytes(), name
    fa = rh.renderFeatures(job(sc, zero), spp=SPP, seed=SEED, want_hit_ids=True)
    fb = rh.renderFeatures(job(sc, persp), spp=SPP, seed=SEED, want_hit_ids=True)
    for k in ("albedo", "normal", "depth", "hits", "hit_ids"):
        assert np.asarray(getattr(fa, k)).tobytes() == np.asarray(getattr(fb, k)).tobytes(), (name, k)


# ---------------------------------------------------------------- 4. each entry point against its own definition
class _WithCamera:
    """The scene with another camera (what tests.test_features_gpu.expected reads)."""

    def __init__(self, sc, cam):
        self._sc, self.camera = sc, cam

    def __getattr__(self, k):
        return getattr(self._sc, k)


@pytest.mark.parametrize("name", ["dragon_low", "cornellBox", "outScene"])
def test_entry_points_match_their_definitions(name, monkeypatch):
    sc, orc = scene(name)
    forks = has_transparent(sc)
    cam = lens(sc, 0.12, 0.9)
    j = job(sc, cam)
    # progressive: K slices of s samples equal one K*s render
    K, s = 3, 2
    ref = render_linear(j, spp=K * s, seed=SEED)
    acc = rh.Accumulator(j, stream_spp=K * s)
    for _ in range(K):
        last = acc.add(s, seed=SEED)
    acc.close()
    same(sc, last.pixels, ref.pixels, (name, "accumulate"))
    if not forks:
        assert last.linear.tobytes() == ref.linear.tobytes(), name
    # adaptive: a pixel that ends with n samples equals the n-sample render
    stream = 8
    ad = rh.AdaptiveAccumulator(j, stream)
    for b in (2, 3, 1, 2):
        img = ad.add(b, SEED, 0.02, min_spp=2)
    counts, _, _ = ad.state()
    ad.close()
    assert len(np.unique(counts)) >= 2 or forks, (name, np.unique(counts))
    want = np.zeros_like(img.pixels)
    for n in np.unique(counts):
        r = rh.Accumulator(j, stream).add(int(n), seed=SEED)
        m = counts == n
        want[m] = r.pixels[m]
        if not forks:
            assert img.linear[m].tobytes() == r.linear[m].tobytes(), (name, n)
    same(sc, img.pixels, want, (name, "adaptive"))
    # features: the oracle's first hits of its own lens rays
    off = rh.sample_offsets(W * H, SPP, SEED)
    monkeypatch.setattr(test_features_gpu, "camera_rays", lens_oracle.camera_rays)  # (the lens rays of tests/lens_oracle.py)
    e = expected(_WithCamera(sc, cam), orc, W, H, off[..., 0].copy(), off[..., 1].copy())
    fe = rh.renderFeatures(j, spp=SPP, offsets=off, want_hit_ids=True)
    assert_same(fe, e, (name, "features"))
    assert np.array_equal(fe.hit_ids, e["ids"]), name
    # light groups: rgb_out is the render's
    lg = rh.renderLightGroups(j, spp=SPP, seed=SEED)
    plain = rh.render(j, spp=SPP, seed=SEED)
    same(sc, lg.image, plain.pixels, (name, "light groups"))
    # views mixing the three projections, with per-view seeds: each view is its own render
    ortho = capi.rh_camera.from_buffer_copy(sc.camera)
    ortho.projection, ortho.proj_width, ortho.proj_height = capi.RH_PROJ_ORTHOGRAPHIC, 2.0, 2.0
    cams = [cam, sc.camera, ortho, lens(sc, 0.3, 0.5), cam]
    seeds = [3, 4, 5, 2**64 - 1, 9]
    vs = rh.renderViews(j, cams, spp=SPP, seeds=seeds, want_hit_ids=True, linear=True)
    for v, (c, sd) in enumerate(zip(cams, seeds)):
        r = rh.render(job(sc, c), spp=SPP, seed=sd, want_hit_ids=True)
        same(sc, vs.pixels[v], r.pixels, (name, "view", v))
        assert np.array_equal(vs.hit_ids[v], r.hit_ids), (name, "view ids", v)
    assert not np.array_equal(vs.hit_ids[0], vs.hit_ids[4])  # same lens, other seed
    # rh_multi_render on one GPU
    try:
        multi = rh.render_multi(j, 1, spp=SPP, seed=SEED)
    finally:
        rh.multi_shutdown([sc])
    same(sc, multi.pixels, plain.pixels, (name, "multi"))
    for k in RAYS:
        assert multi.stats[k] == plain.stats[k], (name, k)


# ---------------------------------------------------------------- 5. bad lens arguments
BAD = [("proj_width", -0.1), ("proj_width", math.nan), ("proj_width", math.inf), ("proj_width", -math.inf),
       ("proj_height", 0.0), ("proj_height", -0.0), ("proj_height", -1.0), ("proj_height", math.nan), ("proj_height", math.inf),
       ("proj_height", -math.inf), ("fovy", 0.0), ("fovy", -0.5), ("fovy", math.nan), ("fovy", math.inf), ("fovy", -math.inf)]


def test_bad_lens_arguments_write_nothing():
    sc, _ = scene("cornellBox")
    L = capi.lib()
    w, h = 16, 8
    good = lens(sc, 0.1, 1.0)
    o = rh.host._opts(job(sc, good, w, h), 1, capi.RH_OFFSETS_NONE, None, 0, 0, 1, h, 0, 0)
    rgb = np.full((3, h, w, 3), 9, np.uint8)
    lin = np.full((3, h, w, 3), 7.0)
    for field, value in BAD:
        bad = capi.rh_camera.from_buffer_copy(good)
        setattr(bad, field, value)
        assert L.rh_render(sc.device, C.byref(bad), C.byref(o), rgb.ctypes.data, None, None) == capi.RH_ERR_ARG, (field, value)
        msg = L.rh_last_error()
        assert field.encode() in msg and b"thin-lens" in msg, (field, value, msg)
        cams = (capi.rh_camera * 3)(good, good, bad)
        vw = capi.rh_views()
        vw.cameras, vw.n_views = C.cast(cams, C.POINTER(capi.rh_camera)), 3
        assert L.rh_render_views(sc.device, C.byref(vw), C.byref(o), rgb.ctypes.data, lin.ctypes.data, None, None) == capi.RH_ERR_ARG
        msg = L.rh_last_error()
        assert b"cameras[2]" in msg and field.encode() in msg, (field, value, msg)
        assert (rgb == 9).all() and (lin == 7.0).all(), (field, value)
    # the edges that are valid: R = 0 and R = -0; perspective and orthographic cameras keep their own checks
    for R in (0.0, -0.0):
        ok = capi.rh_camera.from_buffer_copy(good)
        ok.proj_width = R
        assert L.rh_render(sc.device, C.byref(ok), C.byref(o), rgb[0].ctypes.data, None, None) == capi.RH_OK
    persp = capi.rh_camera.from_buffer_copy(sc.camera)
    persp.fovy, persp.proj_width, persp.proj_height = -1.0, math.nan, -1.0
    assert L.rh_render(sc.device, C.byref(persp), C.byref(o), rgb[0].ctypes.data, None, None) == capi.RH_OK
    with pytest.raises(capi.RayHsError) as e:
        rh.render(job(sc, rh.thinLens(sc.camera, 0.1, -2.0), w, h))
    assert e.value.code == capi.RH_ERR_ARG
