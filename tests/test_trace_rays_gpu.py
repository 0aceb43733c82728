"""GPU tests of the radiance queries (rh_trace_rays / traceRay): camera rays against rh_render, every ray against the
oracle's traceRay (colours, hit ids, per-class ray counts) on every shipped pack and two built scenes, the variants that
must keep the colours (shadow schedule, light maps, device buffers, chunking), queue growth, the scene's render state,
and argument errors."""
import ctypes as C
import zlib

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import COUNT_NAMES, OracleScene, camera_rays
from rayhs_b200 import capi
from tests.test_ray_query_gpu import BUILT, CAM_H, CAM_W, MAX_GRAZING, adversarial_rays, geometry, incoherent_rays
from tests.util import ATOL, RTOL, SCENES, assert_parity, load_scene, to_int_c

pytestmark = pytest.mark.gpu


def has_transparent(sc):
    raw = sc.raw.contents
    return any(raw.materials[i].kind == capi.RH_MAT_TRANSPARENT for i in range(raw.n_materials))


def trace(sc, rays, max_depth, **kw):
    return rh.traceRay(sc, np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:]), max_depth, **kw)


def counts(stats):
    return {k: stats[k] for k in COUNT_NAMES}


def close(a, b):
    return np.isclose(a, b, rtol=RTOL, atol=ATOL, equal_nan=True).all(axis=1)


@pytest.fixture(scope="module", params=SCENES + list(BUILT))
def case(request):
    name = request.param
    sc = BUILT[name]() if name in BUILT else load_scene(name)
    return name, sc, OracleScene(sc.raw), geometry(sc)


def rays_of(name, sc, g):
    rng = np.random.RandomState(zlib.crc32(name.encode()) ^ 0x7ACE)
    return {"camera": camera_rays(sc.camera, CAM_W, CAM_H), "incoherent": incoherent_rays(g, rng),
            "adversarial": adversarial_rays(g, rng)}


@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("size", [(48, 32), (203, 97)])
def test_camera_rays_give_the_renders_bytes_and_hit_ids(name, size):
    sc = load_scene(name)
    w, h = size
    img = rh.render(rh.Rendering(sc, sc.camera, w, h, sc.max_depth), want_hit_ids=True)
    rays = camera_rays(sc.camera, w, h)
    r = trace(sc, rays, sc.max_depth, want_hit_ids=True)
    assert r.colors.shape == (w * h, 3) and r.colors.dtype == np.float64 and r.stats["rays_primary"] == w * h
    assert np.array_equal(r.hit_ids, img.hit_ids.reshape(-1, 2)), name
    got = to_int_c(r.colors).reshape(h, w, 3)
    if has_transparent(sc):  # forks of a Transparent hit add into one accumulator with atomics: 1-LSB wobble
        assert_parity(got, img.pixels, name)
    else:
        assert np.array_equal(got, img.pixels), (name, np.argwhere((got != img.pixels).any(axis=-1))[:5])
    for k in COUNT_NAMES:
        assert r.stats[k] == img.stats[k], (name, k)


@pytest.mark.parametrize("max_depth", [0, 1, "scene", 8])
def test_every_ray_equals_the_oracle(case, max_depth):
    name, sc, orc, g = case
    depth = sc.max_depth if max_depth == "scene" else max_depth
    for kind, rays in rays_of(name, sc, g).items():
        want, want_ids, want_counts = orc.trace_batch(rays, depth)
        what = (name, kind, depth)
        exact = trace(sc, rays, depth, want_hit_ids=True, exact_boxes=True)
        bad = np.flatnonzero(~close(exact.colors, want))
        assert len(bad) == 0, (what, "exact walk", bad[:10], exact.colors[bad[:3]], want[bad[:3]])
        assert np.array_equal(exact.hit_ids, want_ids), what
        assert counts(exact.stats) == want_counts, what
        # the default walk: the same except on rays whose closest hit (of the ray or of a ray it spawns) the float cull
        # decides differently — grazers (DESIGN §3), bounded as for rh_closest_intersection; camera rays have none
        got = trace(sc, rays, depth, want_hit_ids=True)
        graze = np.flatnonzero(~close(got.colors, want) | (got.hit_ids != want_ids).any(axis=1))
        assert len(graze) <= (0 if kind == "camera" else max(1, MAX_GRAZING * len(rays))), \
            (what, graze[:10], got.colors[graze[:3]], want[graze[:3]])
        if len(graze):
            keep = np.setdiff1d(np.arange(len(rays)), graze)
            got = trace(sc, rays[keep], depth)
            want_counts = orc.trace_batch(rays[keep], depth)[2]
        assert counts(got.stats) == want_counts, what
        if kind == "camera" and depth > 0:
            assert (want > 0).any(), (name, "the view is black")


def test_variants_keep_the_colours(case):
    """Shadow schedules, light maps, device buffers and chunking change how the work runs, not the colours."""
    import torch

    name, sc, orc, g = case
    rays = np.concatenate(list(rays_of(name, sc, g).values()))
    rng = np.random.RandomState(5)
    rays = np.concatenate([rays, rays[rng.randint(0, len(rays), 3 * 4096)]])  # several rows of 4096 rays
    depth = max(sc.max_depth, 2)
    base = trace(sc, rays, depth, want_hit_ids=True)
    forks = has_transparent(sc)

    def same(a, b, what):
        if forks:  # Transparent forks add with atomics: equal up to the last bits
            assert close(a, b).all(), (name, what)
        else:
            assert a.tobytes() == b.tobytes(), (name, what, np.flatnonzero((a != b).any(axis=1))[:10])

    for what, kw in (("pooled", dict(shadow="pooled")), ("split", dict(shadow="split")), ("no light maps", dict(light_maps=False)),
                     ("4096-ray chunks", dict(chunk_rays=4096)), ("3-row chunks", dict(chunk_rays=3 * 4096 + 17))):
        r = trace(sc, rays, depth, want_hit_ids=True, **kw)
        same(r.colors, base.colors, what)
        assert np.array_equal(r.hit_ids, base.hit_ids), (name, what)
        assert counts(r.stats) == counts(base.stats), (name, what)
        if "chunk_rays" in kw:
            assert r.stats["chunks"] > 1, (name, what)
    for n in (0, 1, 33, 4096, 4097, len(rays)):
        host = trace(sc, rays[:n], depth, want_hit_ids=True)
        o, d = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (rays[:n, :3], rays[:n, 3:]))
        dev = rh.traceRay(sc, o, d, depth, want_hit_ids=True)
        assert dev.colors.is_cuda and tuple(dev.colors.shape) == (n, 3) and dev.colors.dtype == torch.float64
        assert dev.hit_ids.is_cuda and tuple(dev.hit_ids.shape) == (n, 2)
        same(dev.colors.cpu().numpy(), host.colors, ("device", n))
        assert np.array_equal(dev.hit_ids.cpu().numpy(), host.hit_ids), (name, n)
        assert dev.stats["rays_primary"] == host.stats["rays_primary"] == n


def growth_scene():
    """Transparent and Diffuse spheres inside a box of six mirror planes: no ray leaves, and every Transparent hit
    forks into a reflection and a probe, so the secondary passes hold many times the primary rays."""
    from tests.util import RawScene

    rng = np.random.RandomState(17)
    mats = [{"kind": "transparent", "ior": 1.5}, {"kind": "mirror", "ior": 8.0},
            {"kind": "diffuse", "color1": (0.8, 0.6, 0.4)}, {"kind": "emmit", "color1": (1.5, 1.5, 1.5)}]
    grid = np.linspace(-0.75, 0.75, 4)
    objs = []
    for i, (x, y, z) in enumerate(np.array(np.meshgrid(grid, grid, grid)).reshape(3, -1).T):
        c = np.array([x, y, z]) + rng.uniform(-0.05, 0.05, 3)
        objs.append({"kind": "sphere", "center": tuple(c), "radius": 0.17, "material": 3 if i == 21 else (2 if i % 5 == 0 else 0)})
    for axis in range(3):
        for s in (-1, 1):
            n = np.zeros(3)
            n[axis] = -s
            t = np.roll(n, 1)
            objs.append({"kind": "plane", "point": tuple(-n * 1.2), "normal": tuple(n), "tangent": tuple(t), "material": 1})
    lights = [{"kind": "point", "vec": (0.05, 0.02, -0.03), "color": (3, 3, 3), "radius": 1.0}]
    return RawScene(objs, mats, lights, camera={"position": (0, 0, -1.1)}, size=(64, 64, 8))


def growth_rays(n, seed=3):
    rng = np.random.RandomState(seed)
    o = rng.uniform(-1.1, 1.1, (n, 3))
    d = rng.normal(size=(n, 3))
    return np.concatenate([o, d], axis=1)


def test_queue_growth_retries_and_keeps_the_colours():
    sc = growth_scene()
    n = 1 << 20
    rays = growth_rays(n)
    r = trace(sc, rays, 8, want_hit_ids=True)
    assert r.stats["queue_factor"] > 2, r.stats
    assert r.stats["rays_reflect"] + r.stats["rays_probe"] > 3 * n, r.stats
    idx = np.unique(np.concatenate([np.random.RandomState(4).randint(0, n, 1500), [0, 1, 4095, 4096, n - 1]]))
    want, want_ids, _ = OracleScene(sc.raw).trace_batch(rays[idx], 8)
    assert close(r.colors[idx], want).all(), np.flatnonzero(~close(r.colors[idx], want))[:10]
    assert np.array_equal(r.hit_ids[idx], want_ids)
    assert (want > 0).any()


def test_trace_rays_leaves_the_scenes_render_state_alone():
    """A render, an overflowing traceRay batch, the same render again: same bytes, queue factor and shadow schedule."""
    sc = growth_scene()
    job = rh.Rendering(sc, sc.camera, 256, 256, 0)  # (no secondary rays: the render's own queues never grow)
    first = rh.render(job)
    r = trace(sc, growth_rays(1 << 20), 8)
    assert r.stats["queue_factor"] > max(2, first.stats["queue_factor"]), (r.stats["queue_factor"], first.stats["queue_factor"])
    second = rh.render(job)
    assert_parity(second.pixels, first.pixels)  # (Transparent forks: the 1-LSB wobble)
    for k in ("queue_factor", "shadow_split", "chunks", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert second.stats[k] == first.stats[k], k


def test_argument_errors():
    import torch

    sc = load_scene("cornellBox")
    L = capi.lib()
    dev = sc.device
    rays = np.zeros((4, 6))
    rays[:, 5] = 1
    col = np.empty((4, 3))
    ids = np.empty((4, 2), dtype=np.int32)

    def call(opts=None, r=rays.ctypes.data, n=4, c=col.ctypes.data, i=None, **kw):
        o = opts or capi.rh_trace_opts()
        for k, v in kw.items():
            setattr(o, k, v)
        return L.rh_trace_rays(dev, r, n, C.byref(o), c, i, None)

    assert call() == capi.RH_OK
    for bad in (capi.RH_FLAG_PROFILE, capi.RH_FLAG_COUNT, capi.RH_FLAG_PEER_FRAMES, capi.RH_FLAG_DEVICE_OFFSETS,
                capi.RH_FLAG_SHARD_OFFSETS, 1 << 20):
        assert call(flags=bad) == capi.RH_ERR_ARG, bad
    for d in (-1, 31, 1000):
        assert call(max_depth=d) == capi.RH_ERR_ARG, d
    assert call(max_depth=30) == capi.RH_OK
    assert call(r=None) == capi.RH_ERR_ARG and call(c=None) == capi.RH_ERR_ARG
    assert call(r=None, n=0, c=None) == capi.RH_OK
    assert call(flags=capi.RH_FLAG_HIT_IDS) == capi.RH_ERR_ARG
    assert call(flags=capi.RH_FLAG_HIT_IDS, i=ids.ctypes.data) == capi.RH_OK
    assert L.rh_trace_rays(dev, rays.ctypes.data, 4, None, col.ctypes.data, None, None) == capi.RH_ERR_ARG
    assert L.rh_trace_rays(None, rays.ctypes.data, 4, C.byref(capi.rh_trace_opts()), col.ctypes.data, None, None) == capi.RH_ERR_ARG
    # device flag with host memory, and misaligned device buffers
    D = capi.RH_FLAG_DEVICE_OUT
    assert call(flags=D) == capi.RH_ERR_ARG
    t = torch.zeros(4 * 6 + 2, dtype=torch.float64, device="cuda")
    t[5::6] = 1
    c = torch.empty(4 * 3 + 1, dtype=torch.float64, device="cuda")
    i = torch.empty(4 * 2 + 2, dtype=torch.int32, device="cuda")
    assert call(flags=D, r=t.data_ptr(), c=c.data_ptr()) == capi.RH_OK
    assert call(flags=D, r=t.data_ptr() + 8, c=c.data_ptr()) == capi.RH_ERR_ARG
    assert call(flags=D, r=t.data_ptr(), c=c.data_ptr() + 4) == capi.RH_ERR_ARG
    assert call(flags=D | capi.RH_FLAG_HIT_IDS, r=t.data_ptr(), c=c.data_ptr(), i=i.data_ptr() + 4) == capi.RH_ERR_ARG
    assert call(flags=D | capi.RH_FLAG_HIT_IDS, r=t.data_ptr(), c=c.data_ptr(), i=ids.ctypes.data) == capi.RH_ERR_ARG
    assert call(flags=D | capi.RH_FLAG_HIT_IDS, r=t.data_ptr(), c=c.data_ptr() + 8, i=i.data_ptr() + 8) == capi.RH_OK
    # the Python layer: shapes, dtypes, a mix of host and device inputs, and the library's checks surface as errors
    o = np.zeros((3, 3))
    for bad_o, bad_d in ((o.astype(np.float32), o), (o, o[:2]), (o, torch.zeros(3, 3, dtype=torch.float64).cuda()),
                         (torch.zeros(3, 3).cuda(), torch.zeros(3, 3).cuda())):
        with pytest.raises(ValueError):
            rh.traceRay(sc, bad_o, bad_d, 3)
    for kw in (dict(max_depth=31), dict(max_depth=-1)):
        with pytest.raises(capi.RayHsError) as e:
            rh.traceRay(sc, o, o, **kw)
        assert e.value.code == capi.RH_ERR_ARG
