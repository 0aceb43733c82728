"""GPU tests of the feature buffers (rh_render_features / renderFeatures) against the oracle (orc_feature_batch):
every shipped pack and a built scene with every material kind, checker and texture maps on planes and meshes and a
ShowUV sphere, seen through both projections; the render's own hits; every offset mode, shards, device buffers, the
exact walk and chunked host buffers giving the same bytes; scene updates; argument errors."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene, camera_rays
from rayhs_b200 import capi
from tests.util import SCENES, RawScene, load_scene

pytestmark = pytest.mark.gpu

SPHERE_UV_ULP = 8  # as in the ray-query tests: CUDA's atan / acos against glibc's, for a sphere's u and v
SIZES = [(48, 32), (203, 97)]


def built_scene(projection):
    """Every material kind; checker and texture maps on a plane and on meshes; a ShowUV sphere."""
    rng = np.random.RandomState(5)
    tex = rng.uniform(0, 1, (5, 7, 3))
    mats = [{"kind": "diffuse", "cmap": "checker", "color1": (0.9, 0.2, 0.1), "color2": (0.1, 0.3, 0.8), "size": 0.7},  # 0
            {"kind": "plastic", "cmap": "texture", "texture": 0, "ior": 1.4},                                             # 1
            {"kind": "diffuse", "cmap": "texture", "texture": 0},                                                          # 2
            {"kind": "plastic", "cmap": "checker", "color1": (0.2, 0.8, 0.3), "color2": (0.7, 0.7, 0.1), "size": 0.3},  # 3
            {"kind": "mirror"}, {"kind": "transparent", "ior": 1.5}, {"kind": "emmit", "color1": (3, 2.5, 2)},            # 4 5 6
            {"kind": "shownormal"}, {"kind": "showuv"}, {"kind": "diffuse", "color1": (0.5, 0.6, 0.7)}]                    # 7 8 9

    def quad(center, sx, sy, z_tilt, material):
        c = np.array(center, dtype=np.float64)
        pos = np.array([c + (-sx, -sy, -z_tilt), c + (sx, -sy, -z_tilt), c + (sx, sy, z_tilt), c + (-sx, sy, z_tilt)])
        nrm = np.array([[0.1, 0.2, -1], [0, 0, -1], [-0.2, 0.1, -1], [0.3, -0.1, -0.9]])
        uv = np.array([[0, 0], [1.3, 0], [1.3, 1.7], [0, 1.7]])
        return {"kind": "mesh", "positions": pos, "normals": nrm, "uvs": uv, "indices": [0, 1, 2, 0, 2, 3], "material": material}

    objs = [{"kind": "plane", "point": (0, -1, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0},
            {"kind": "plane", "point": (0, 0, 3), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 2},
            quad((-0.9, 0.5, 1.2), 0.45, 0.4, 0.1, 1), quad((0.9, 0.5, 1.2), 0.45, 0.4, -0.15, 3),
            {"kind": "sphere", "center": (0, 0.1, 0.8), "radius": 0.35, "material": 8},
            {"kind": "sphere", "center": (-0.8, -0.6, 0.6), "radius": 0.3, "material": 4},
            {"kind": "sphere", "center": (0.8, -0.6, 0.6), "radius": 0.3, "material": 5},
            {"kind": "sphere", "center": (0, -0.7, 0.2), "radius": 0.2, "material": 6},
            {"kind": "sphere", "center": (-0.3, 0.8, 0.5), "radius": 0.2, "material": 7},
            {"kind": "sphere", "center": (0.4, 0.8, 0.5), "radius": 0.2, "material": 9}]
    lights = [{"kind": "point", "vec": (0, 2, -1), "color": (4, 4, 4)}, {"kind": "directional", "vec": (0.2, 1, -0.3), "color": (0.5, 0.5, 0.5)}]
    return RawScene(objs, mats, lights, textures=[tex], camera={"position": (0, 0, -2.5), "projection": projection}, size=(64, 48, 2))


BUILT = {"built_perspective": lambda: built_scene("perspective"), "built_orthographic": lambda: built_scene("orthographic")}
_cache = {}


def scene(name):
    if name not in _cache:
        sc = BUILT[name]() if name in BUILT else load_scene(name)
        _cache[name] = (sc, OracleScene(sc.raw))
    return _cache[name]


def job(sc, w, h):
    return rh.Rendering(sc, sc.camera, w, h, 3)


def uv_dependent(sc):
    """Per object: True for a sphere whose albedo depends on its uv (a non-flat Diffuse / Plastic, or ShowUV)."""
    raw = sc.raw.contents
    out = []
    for i in range(raw.n_objects):
        o = raw.objects[i]
        m = raw.materials[o.material]
        out.append(o.kind == capi.RH_OBJ_SPHERE and (m.kind == capi.RH_MAT_SHOWUV or (
            m.kind in (capi.RH_MAT_DIFFUSE, capi.RH_MAT_PLASTIC) and m.cmap_kind != capi.RH_CMAP_FLAT)))
    return np.array(out + [False])  # (index -1: a miss)


def samples(orc, camera, w, h, ox, oy):
    """The camera rays at pixel coordinates (col + ox, row + oy) for ox, oy [h * w, spp] (float64, pixel-major), through
    the batch: dict of rays [h*w*spp, 6] and, per pixel and sample, t [h*w, spp], n and albedo [h*w, spp, 3], ids and
    uv [h*w, spp, 2]."""
    spp = ox.shape[1]
    rows, cols = np.divmod(np.arange(h * w), w)
    xy = np.empty((h * w, spp, 2))
    xy[..., 0] = cols[:, None] + ox
    xy[..., 1] = rows[:, None] + oy
    rays = camera_rays(camera, w, h, xy.reshape(-1, 2))
    f = orc.features_batch(rays)
    return dict(rays=rays, t=f["t"].reshape(h * w, spp), n=f["n"].reshape(h * w, spp, 3), albedo=f["albedo"].reshape(h * w, spp, 3),
                ids=f["ids"].reshape(h * w, spp, 2), uv=f["uv"].reshape(h * w, spp, 2))


def fold(s, w, h):
    """The per-pixel buffers of samples `s`: albedo [h, w, 3], normal [h, w, 3], depth [h, w], hits [h, w] and ids
    [h, w, spp, 2]; foldl (+) 0 over the samples in sample order, per channel, then times 1.0 / spp (depth: 1.0 / hits
    over the hitting samples' t)."""
    spp = s["t"].shape[1]
    hit = s["ids"][..., 0] >= 0
    a, nn, ts = np.zeros((h * w, 3)), np.zeros((h * w, 3)), np.zeros(h * w)
    for k in range(spp):
        a = a + s["albedo"][:, k]
        nn = nn + s["n"][:, k]
        ts = ts + np.where(hit[:, k], s["t"][:, k], 0.0)
    inv = 1.0 / spp
    hits = hit.sum(axis=1).astype(np.uint32)
    with np.errstate(divide="ignore", invalid="ignore"):
        depth = np.where(hits > 0, (1.0 / hits.astype(np.float64)) * ts, np.inf)
    return dict(albedo=(inv * a).reshape(h, w, 3), normal=(inv * nn).reshape(h, w, 3), depth=depth.reshape(h, w),
                hits=hits.reshape(h, w), ids=s["ids"].reshape(h, w, spp, 2))


def expected(sc, orc, w, h, ox, oy):
    """The oracle's buffers for pixel offsets ox, oy [h*w, spp].  A sample on a sphere whose albedo depends on its uv takes
    the device's uv (rh_closest_intersection of the same ray), which must be within SPHERE_UV_ULP of the oracle's."""
    s = samples(orc, sc.camera, w, h, ox, oy)
    dep = uv_dependent(sc)[s["ids"][..., 0]]
    if dep.any():
        rays = s["rays"].reshape(h * w, -1, 6)[dep]
        got = rh.closestIntersection(sc, np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:])).uv
        want = s["uv"][dep]
        ok = (got == want) | (np.abs(got - want) <= SPHERE_UV_ULP * np.spacing(np.maximum(np.abs(got), np.abs(want))))
        assert ok.all(), ("sphere uv", got[~ok.all(axis=1)][:5], want[~ok.all(axis=1)][:5])
        raw = sc.raw.contents
        mats = [raw.objects[o].material for o in s["ids"][..., 0][dep]]
        al = []
        for m, (u, v) in zip(mats, got):
            al.append((u, v, 0.0) if raw.materials[m].kind == capi.RH_MAT_SHOWUV else orc.color_at(m, u, v))
        s["albedo"][dep] = np.array(al)
    return fold(s, w, h)


def assert_same(fe, e, what, rows=None):
    """Every buffer bit-identical (rows: the expectation's rows to compare against)."""
    for k in ("albedo", "normal", "depth", "hits"):
        got = np.asarray(fe[k] if isinstance(fe, dict) else getattr(fe, k))
        want = e[k] if rows is None else e[k][rows]
        assert got.shape == want.shape and got.tobytes() == want.tobytes(), (what, k, np.argwhere(got != want)[:5])


def host(fe):
    """A Features' buffers as numpy arrays (device buffers copied back; device hit counts as uint32)."""
    out = {}
    for k in ("albedo", "normal", "depth", "hits", "hit_ids"):
        v = getattr(fe, k)
        if v is not None and hasattr(v, "cpu"):
            v = v.cpu().numpy()
            if k == "hits":
                v = v.view(np.uint32)
        out[k] = v
    return out


def f64_offsets(w, h, spp, seed=7):
    off = rh.sample_offsets(w * h, spp, seed)
    return off, off[..., 0].copy(), off[..., 1].copy()


@pytest.mark.parametrize("name", SCENES + list(BUILT))
@pytest.mark.parametrize("w,h", SIZES)
def test_buffers_equal_the_oracle(name, w, h):
    sc, orc = scene(name)
    zero = np.zeros((w * h, 1))
    e = expected(sc, orc, w, h, zero, zero)
    fe = rh.renderFeatures(job(sc, w, h), want_hit_ids=True)
    assert_same(fe, e, (name, w, h, "no offsets"))
    assert np.array_equal(fe.hit_ids, e["ids"]), name
    assert (fe.hits > 0).any(), (name, "the view sees nothing")
    off, ox, oy = f64_offsets(w, h, 4)
    e4 = expected(sc, orc, w, h, ox, oy)
    assert_same(rh.renderFeatures(job(sc, w, h), spp=4, offsets=off), e4, (name, w, h, "F64, 4 spp"))


@pytest.mark.parametrize("name", ["cornellBox", "texture", "dragon_low", "built_perspective"])
def test_same_hits_and_ids_as_the_render(name):
    sc, orc = scene(name)
    w, h, spp = 203, 97, 4
    off, _, _ = f64_offsets(w, h, spp)
    img = rh.render(job(sc, w, h), spp=spp, offsets=off, want_hit_ids=True)
    fe = rh.renderFeatures(job(sc, w, h), spp=spp, offsets=off, want_hit_ids=True)
    assert np.array_equal(fe.hits, (img.hit_ids[..., 0] >= 0).sum(axis=2).astype(np.uint32)), name
    assert fe.hit_ids.tobytes() == img.hit_ids.tobytes(), name
    st = fe.stats
    assert st["rays_primary"] == w * h * spp and st["chunks"] == 1 and st["kernel_launches"] == 1 and st["ms_total"] > 0
    assert all(v == 0 for k, v in st.items() if k not in ("rays_primary", "chunks", "kernel_launches", "ms_total")), st


@pytest.mark.parametrize("name", ["outScene", "built_orthographic"])
def test_offset_modes_shards_and_buffers(name):
    import torch

    sc, orc = scene(name)
    w, h, spp = 203, 97, 4
    j = job(sc, w, h)
    # F32 and tiled offsets against their own expectation
    off32 = rh.sample_offsets(w * h, spp, 11, dtype=np.float32)
    e = expected(sc, orc, w, h, off32[..., 0].astype(np.float64), off32[..., 1].astype(np.float64))
    assert_same(rh.renderFeatures(j, spp=spp, offsets=off32), e, (name, "F32"))
    T = 5
    tile = rh.sample_offsets(T * T, spp, 12)
    rows, cols = np.divmod(np.arange(w * h), w)
    full = tile[(rows % T) * T + cols % T]
    e = expected(sc, orc, w, h, full[..., 0].copy(), full[..., 1].copy())
    assert_same(rh.renderFeatures(j, spp=spp, offsets=tile, offset_tile=T), e, (name, "tiled"))
    # SplitMix64: samples b .. b + spp - 1 of an 8-sample stream = the F64 slice of that stream
    stream = rh.sample_offsets(w * h, 8, 24)
    for b in (0, 3):
        sm = rh.renderFeatures(j, spp=spp, seed=24, stream_spp=8, stream_base=b, want_hit_ids=True)
        f64 = rh.renderFeatures(j, spp=spp, offsets=stream[:, b:b + spp], want_hit_ids=True)
        assert_same(host(sm), host(f64), (name, "splitmix", b))
        assert sm.hit_ids.tobytes() == f64.hit_ids.tobytes()
    # shards (with RH_FLAG_SHARD_OFFSETS too) against the rows of the unsharded call
    off, _, _ = f64_offsets(w, h, spp)
    whole = host(rh.renderFeatures(j, spp=spp, offsets=off, want_hit_ids=True))
    for G in (2, 3):
        bh = capi.lib().rh_default_band_height(h, G)
        for g in range(G):
            part = host(rh.renderFeatures(j, spp=spp, offsets=off, want_hit_ids=True, shard_index=g, shard_count=G))
            grows = np.array(rh.shard_global_rows(h, g, G, bh))
            real = grows >= 0
            assert_same({k: part[k][real] for k in part}, whole, (name, G, g), rows=grows[real])
            assert part["hit_ids"][real].tobytes() == whole["hit_ids"][grows[real]].tobytes()
            assert not part["hits"][~real].any() and np.isinf(part["depth"][~real]).all() and not part["albedo"][~real].any()
            compact = np.ascontiguousarray(off.reshape(h, w, spp, 2)[np.maximum(grows, 0)])
            sh = shard_call(sc, j, spp, compact, g, G, bh, len(grows))
            assert_same({k: sh[k][real] for k in sh}, whole, (name, G, g, "shard offsets"), rows=grows[real])
    # device outputs and device offsets against host ones
    dev = rh.renderFeatures(j, spp=spp, offsets=torch.from_numpy(off).cuda(), want_hit_ids=True, device=True)
    assert dev.albedo.is_cuda and dev.hits.is_cuda and dev.hit_ids.is_cuda
    d = host(dev)
    assert_same(d, whole, (name, "device"))
    assert d["hit_ids"].tobytes() == whole["hit_ids"].tobytes()
    assert_same(host(rh.renderFeatures(j, spp=spp, offsets=off, device=True)), whole, (name, "device outputs, host offsets"))
    # the exact walk: camera rays have no grazers
    assert_same(host(rh.renderFeatures(j, spp=spp, offsets=off, exact_boxes=True)), whole, (name, "exact boxes"))


def shard_call(sc, j, spp, compact, g, G, bh, rows):
    """rh_render_features of shard g of G with RH_FLAG_SHARD_OFFSETS (the shard's rows of the offsets only)."""
    L = capi.lib()
    o = capi.rh_render_opts()
    o.width, o.height, o.max_depth, o.spp = j.width, j.height, 3, spp
    o.offset_mode, o.offsets = capi.RH_OFFSETS_F64, compact.ctypes.data
    o.shard_index, o.shard_count, o.band_height, o.flags = g, G, bh, capi.RH_FLAG_SHARD_OFFSETS
    out = dict(albedo=np.empty((rows, j.width, 3)), normal=np.empty((rows, j.width, 3)), depth=np.empty((rows, j.width)),
               hits=np.empty((rows, j.width), dtype=np.uint32))
    ft = capi.rh_features()
    ft.albedo, ft.normal, ft.depth, ft.hits = (out[k].ctypes.data for k in ("albedo", "normal", "depth", "hits"))
    capi.check(L.rh_render_features(sc.device, C.byref(j.camera), C.byref(o), C.byref(ft), None, None))
    return out


def test_host_buffers_over_several_scratch_chunks():
    """1024 x 768 at 16 spp (12.6 M samples, six chunks of host scratch) with host offsets and outputs gives the bytes of
    the same frame with device offsets and outputs (one launch)."""
    import torch

    sc, _ = scene("cornellBox")
    j = job(sc, 1024, 768)
    off = rh.sample_offsets(1024 * 768, 16, 3)
    h = rh.renderFeatures(j, spp=16, offsets=off, want_hit_ids=True)
    d = rh.renderFeatures(j, spp=16, offsets=torch.from_numpy(off).cuda(), want_hit_ids=True, device=True)
    assert h.stats["chunks"] >= 3 and d.stats["chunks"] == 1, (h.stats["chunks"], d.stats["chunks"])
    assert h.stats["rays_primary"] == d.stats["rays_primary"] == 1024 * 768 * 16
    dd = host(d)
    assert_same(dd, host(h), "chunked host buffers")
    assert dd["hit_ids"].tobytes() == h.hit_ids.tobytes()


def test_scene_update_and_learned_state():
    w, h = 96, 64
    sc = load_scene("cornellBox")
    mats = sc.materials
    k = next(i for i in range(len(mats)) if mats[i].kind == capi.RH_MAT_DIFFUSE and mats[i].cmap_kind == capi.RH_CMAP_FLAT)
    before = rh.renderFeatures(job(sc, w, h))
    edited = sc.materials
    edited[k].cmap_kind, edited[k].size = capi.RH_CMAP_CHECKER, 0.3
    edited[k].color2[:] = (0.05, 0.6, 0.2)
    sc.update(materials=edited)
    after = rh.renderFeatures(job(sc, w, h))
    fresh = load_scene("cornellBox")
    fresh.update(materials=edited)  # before the device copy exists: a fresh rh_scene_create of the edited tables
    want = rh.renderFeatures(job(fresh, w, h))
    assert_same(host(after), host(want), "updated scene")
    assert after.albedo.tobytes() != before.albedo.tobytes()
    # the call leaves the scene's learned state alone: render, features, render == render, render
    a, b = load_scene("dragon_low"), load_scene("dragon_low")
    ja, jb = job(a, 203, 97), job(b, 203, 97)
    off, _, _ = f64_offsets(203, 97, 2)
    ra1 = rh.render(ja, spp=2, offsets=off)
    rh.renderFeatures(ja, spp=2, offsets=off)
    ra2 = rh.render(ja, spp=2, offsets=off)
    rb1 = rh.render(jb, spp=2, offsets=off)
    rb2 = rh.render(jb, spp=2, offsets=off)
    for x, y in ((ra1, rb1), (ra2, rb2)):
        assert x.pixels.tobytes() == y.pixels.tobytes()
        assert {k: v for k, v in x.stats.items() if not k.startswith("ms_")} == {k: v for k, v in y.stats.items() if not k.startswith("ms_")}


def test_argument_errors():
    import torch

    sc, _ = scene("cornellBox")
    L = capi.lib()
    w, h = 16, 8
    o = capi.rh_render_opts()
    o.width, o.height, o.max_depth, o.spp, o.shard_count = w, h, 3, 2, 1
    cam = sc.camera
    depth = np.empty((h, w))
    ft = capi.rh_features()
    ft.depth = depth.ctypes.data
    ids = np.empty((h, w, 2, 2), dtype=np.int32)

    def call(opts=o, feats=ft, ids_ptr=None, scene_=sc.device, camera=cam):
        return L.rh_render_features(scene_, C.byref(camera) if camera is not None else None, C.byref(opts) if opts is not None else None,
                                    C.byref(feats) if feats is not None else None, ids_ptr, None)

    assert call() == capi.RH_OK
    assert call(scene_=None) == call(camera=None) == call(opts=None) == call(feats=None) == capi.RH_ERR_ARG
    assert call(feats=capi.rh_features()) == capi.RH_ERR_ARG  # no output
    o.flags = capi.RH_FLAG_HIT_IDS
    assert call(feats=capi.rh_features(), ids_ptr=ids.ctypes.data) == capi.RH_OK  # hit ids alone are an output
    assert call() == capi.RH_ERR_ARG  # RH_FLAG_HIT_IDS without a buffer
    for bad in (capi.RH_FLAG_PEER_FRAMES, capi.RH_FLAG_COUNT, capi.RH_FLAG_PROFILE):
        o.flags = bad
        assert call() == capi.RH_ERR_ARG, bad
    o.flags = capi.RH_FLAG_SHADOW_POOLED | capi.RH_FLAG_SHADOW_SPLIT | capi.RH_FLAG_NO_LIGHT_MAPS
    o.chunk_samples = 5
    assert call() == capi.RH_OK  # accepted, no effect
    o.flags, o.chunk_samples = 0, 0
    o.max_depth = 31
    assert call() == capi.RH_ERR_ARG
    o.max_depth = 3
    # stream fields with another offset mode; past the end of the stream
    ft.stream_spp = 4
    assert call() == capi.RH_ERR_ARG
    seed = C.c_uint64(1)
    o.offset_mode, o.offsets = capi.RH_OFFSETS_SPLITMIX64, C.addressof(seed)
    ft.stream_base = 2
    assert call() == capi.RH_OK
    ft.stream_base = 3
    assert call() == capi.RH_ERR_ARG
    ft.stream_spp = 0  # = spp
    assert call() == capi.RH_ERR_ARG
    ft.stream_base = 0
    assert call() == capi.RH_OK
    o.offset_mode, o.offsets = capi.RH_OFFSETS_NONE, None
    # RH_FLAG_DEVICE_OUT: host pointers and misaligned device pointers
    o.flags = capi.RH_FLAG_DEVICE_OUT
    assert call() == capi.RH_ERR_ARG
    t = torch.empty(w * h + 1, dtype=torch.float64, device="cuda")
    ft.depth = t.data_ptr()
    assert call() == capi.RH_OK
    ft.depth = t.data_ptr() + 4
    assert call() == capi.RH_ERR_ARG
    ft.depth = t.data_ptr()
    o.flags = capi.RH_FLAG_DEVICE_OUT | capi.RH_FLAG_HIT_IDS
    assert call(ids_ptr=ids.ctypes.data) == capi.RH_ERR_ARG
    ti = torch.empty(h * w * 2 * 2 + 2, dtype=torch.int32, device="cuda")
    assert call(ids_ptr=ti.data_ptr() + 4) == capi.RH_ERR_ARG
    assert call(ids_ptr=ti.data_ptr()) == capi.RH_OK
    # the Python layer
    with pytest.raises(ValueError):
        rh.renderFeatures(job(sc, w, h), spp=2, offsets=torch.zeros((w * h, 2, 2), dtype=torch.float64).cuda())  # CUDA offsets, host outputs
    with pytest.raises(capi.RayHsError) as e:
        rh.renderFeatures(job(sc, w, h), spp=2, seed=1, stream_spp=3, stream_base=2)
    assert e.value.code == capi.RH_ERR_ARG
