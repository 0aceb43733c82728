"""GPU tests of sphere lights (RH_LIGHT_SPHERE): renders of packs whose point lights became sphere lights, mixed scenes of
point, sphere and directional lights, and balls placed against each shadow shortcut, held to the sphere-light oracle
(tests/sphere_light_oracle.py: bytes, linear colours, hit ids and ray counts) under both shadow schedules, exact boxes and
no light maps; the light-table limits (12 / 13 and 32 / 33 lights); radius 0; every shading entry point against its own
definition; scene updates against a fresh rh_scene_create; the point lights' tables beside sphere lights; bad radii."""
import ctypes as C
import math

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi
from tests.lens_oracle import camera_rays
from tests.sphere_light_oracle import SphereOracle
from tests.test_trace_rays_gpu import has_transparent
from tests.util import assert_oracle_exact, assert_parity, load_scene, render_linear

pytestmark = pytest.mark.gpu

W, H, SPP, SEED = 32, 20, 4, 24
RAYS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
P, S, D = capi.RH_LIGHT_POINT, capi.RH_LIGHT_SPHERE, capi.RH_LIGHT_DIRECTIONAL


def light(kind, vec, color=(1.0, 1.0, 1.0), radius=0.1):
    return capi.rh_light(kind=kind, vec=tuple(float(x) for x in vec), color=tuple(float(x) for x in color), radius=float(radius))


def with_lights(name, lights):
    sc = load_scene(name)
    sc.update(lights=list(lights))
    return sc


def as_spheres(name, radius=None):
    """The pack with its point lights turned into sphere lights (of their own radius, or `radius`); transform, which has
    only directional lights, gains a sphere light."""
    sc = load_scene(name)
    out = []
    for L in sc.lights:
        if L.kind == P:
            L.kind = S
            if radius is not None:
                L.radius = radius
        out.append(L)
    if name == "transform":
        out.append(light(S, (0.5, 1.5, 2.0), (3, 3, 3), 0.4 if radius is None else radius))
    sc.update(lights=out)
    return sc


def job(sc, w=W, h=H, cam=None):
    return rh.Rendering(sc, sc.camera if cam is None else cam, w, h, sc.max_depth)


def same(sc, a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    if has_transparent(sc) and a.dtype == np.uint8:
        assert_parity(a, b, str(what))
    else:
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), (what, int((a != b).sum()))


def assert_oracle(sc, img, w, h, spp, offsets, what, cam=None):
    ref = SphereOracle(sc.raw).render(sc.camera if cam is None else cam, w, h, sc.max_depth, spp=spp, offsets=offsets)
    assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"]), what
    assert_oracle_exact(img.pixels, img.linear, ref, str(what))
    got = tuple(img.stats[k] for k in RAYS)
    want = tuple(ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow"))
    assert got == want, (what, got, want)
    return ref


def check_scene(sc, what, w=W, h=H, spp=SPP):
    """The render against the oracle, and rh_render under both schedules, exact boxes and no light maps: the same bytes."""
    j = job(sc, w, h)
    img = render_linear(j, spp=spp, seed=SEED)
    assert_oracle(sc, img, w, h, spp, rh.sample_offsets(w * h, spp, SEED), what)
    for kw in (dict(shadow="pooled"), dict(shadow="split"), dict(exact_boxes=True), dict(light_maps=False)):
        r = rh.render(j, spp=spp, seed=SEED, want_hit_ids=True, **kw)
        same(sc, r.pixels, img.pixels, (what, kw))
        assert np.array_equal(r.hit_ids, img.hit_ids), (what, kw)
        assert tuple(r.stats[k] for k in RAYS) == tuple(img.stats[k] for k in RAYS), (what, kw)
    return img


# ---------------------------------------------------------------- 1. packs and mixed scenes against the oracle
@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "texture", "transform"])
def test_packs_with_sphere_lights_equal_the_oracle(name):
    img = check_scene(as_spheres(name), name)
    hard = render_linear(job(load_scene(name)), spp=SPP, seed=SEED)
    if name != "transform":
        assert not np.array_equal(img.linear, hard.linear), name  # (the balls soften the shadows)


def mixed(n, kinds=(P, S, D)):
    """n lights inside the Cornell box, cycling through `kinds`, dim enough that the sum stays below white."""
    rng = np.random.RandomState(n)
    out = []
    for i in range(n):
        k = kinds[i % len(kinds)]
        if k == D:
            out.append(light(D, (rng.uniform(-0.5, 0.5), -1.0, rng.uniform(-0.5, 0.5)), (0.04, 0.04, 0.05), 0))
        else:
            out.append(light(k, (rng.uniform(-0.7, 0.7), rng.uniform(0.2, 0.9), rng.uniform(-0.2, 0.9)), (2.0, 1.8, 1.6), rng.uniform(0.05, 0.3)))
    return out


@pytest.mark.parametrize("n", [3, 12, 13, 32, 33])
def test_mixed_scenes_and_the_light_limits(n):
    """12 / 13: the lit-bit and staged-light limits; 32 / 33: the masks of a queued hit (shadow_simple_kernel beyond)."""
    for name in ("cornellBox", "dragon_low"):
        check_scene(with_lights(name, mixed(n)), (name, n), 24, 16, 2)


# ---------------------------------------------------------------- 2. balls against each shortcut
def mesh_box(sc):
    r = sc.raw.contents
    for i in range(r.n_objects):
        o = r.objects[i]
        if o.kind == capi.RH_OBJ_MESH:
            pos = np.ctypeslib.as_array(o.positions, shape=(o.n_verts, 3))
            return pos.min(axis=0), pos.max(axis=0)
    raise AssertionError("no mesh")


def objects(sc, kind):
    r = sc.raw.contents
    return [r.objects[i] for i in range(r.n_objects) if r.objects[i].kind == kind]


def test_adversarial_balls():
    # a centre outside the mesh's root box whose ball overlaps it (the light-side bits must not cull the mesh)
    sc = load_scene("dragon_low")
    lo, hi = mesh_box(sc)
    mid = 0.5 * (lo + hi)
    c = np.array([mid[0], hi[1] + 0.05, mid[2]])
    check_scene(with_lights("dragon_low", [light(S, c, (2, 2, 2), 0.3), light(P, (0.0, 0.9, 0.75), (50, 50, 50), 0.1)]), "root box")
    # a ball crossing an occluding plane: the samples behind the wall are shadowed (the plane sides must not skip it)
    sc = load_scene("cornellBox")
    planes = objects(sc, capi.RH_OBJ_PLANE)
    assert planes
    for pl in planes[:3]:
        c = np.array(pl.a) + 0.02 * np.array(pl.b)
        check_scene(with_lights("cornellBox", [light(S, c, (3, 3, 3), 0.25), light(P, (0.0, 0.9, 0.75), (20, 20, 20), 0.1)]),
                    ("plane", tuple(pl.a)))
    # a ball overlapping an occluding sphere
    spheres = objects(sc, capi.RH_OBJ_SPHERE)
    assert spheres
    s0 = spheres[0]
    c = np.array(s0.a) + np.array([0.0, s0.b[0] * 1.1, 0.0])
    check_scene(with_lights("cornellBox", [light(S, c, (3, 3, 3), 0.5 * s0.b[0]), light(P, (0.0, 0.9, 0.75), (20, 20, 20), 0.1)]),
                "sphere")
    # hit points inside the ball
    check_scene(with_lights("cornellBox", [light(S, (0.0, 0.0, 0.5), (1, 1, 1), 1.5)]), "inside")
    check_scene(with_lights("dragon_low", [light(S, mid, (1, 1, 1), float(np.abs(hi - lo).max()))]), "inside mesh")


@pytest.mark.parametrize("name", ["cornellBox", "dragon_low"])
def test_radius_zero_gives_the_point_lights_bytes(name):
    zero = as_spheres(name, radius=0.0)
    pt = load_scene(name)
    lights = pt.lights
    for L in lights:
        if L.kind == P:
            L.radius = 0.0
    pt.update(lights=list(lights))
    a = rh.render(job(zero), spp=SPP, seed=SEED, want_hit_ids=True)
    b = rh.render(job(pt), spp=SPP, seed=SEED, want_hit_ids=True)
    assert a.pixels.tobytes() == b.pixels.tobytes() and np.array_equal(a.hit_ids, b.hit_ids)
    assert tuple(a.stats[k] for k in RAYS) == tuple(b.stats[k] for k in RAYS)


# ---------------------------------------------------------------- 3. every shading entry point
@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "texture"])
def test_entry_points_match_their_definitions(name):
    import torch

    sc = as_spheres(name)
    forks = has_transparent(sc)
    j = job(sc)
    plain = rh.render(j, spp=SPP, seed=SEED, want_hit_ids=True)
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
    same(sc, img.pixels, want, (name, "adaptive"))
    # views with per-view seeds: each view is its own render
    cams = [sc.camera, sc.camera]
    vs = rh.renderViews(j, cams, spp=SPP, seeds=[SEED, 7], want_hit_ids=True, linear=True)
    for v, sd in enumerate((SEED, 7)):
        r = rh.render(j, spp=SPP, seed=sd, want_hit_ids=True)
        same(sc, vs.pixels[v], r.pixels, (name, "view", v))
        assert np.array_equal(vs.hit_ids[v], r.hit_ids), (name, "view ids", v)
    # light groups: the beauty is the render's, the groups sum to it and relight; one light alone is the oracle's frame
    # of the scene whose other lights are black (the light indices, and so the samples, stay)
    lgs = rh.renderLightGroups(j, spp=SPP, seed=SEED, want_hit_ids=True)
    same(sc, lgs.image, plain.pixels, (name, "light groups"))
    total = lgs.groups.sum(axis=0) + lgs.rest
    assert np.allclose(total, ref_linear(j), rtol=1e-9, atol=1e-12), name
    n_l = len(sc.lights)
    assert np.allclose(lgs.relight(np.ones((n_l, 3))), total, rtol=1e-12, atol=1e-12)
    off = rh.sample_offsets(W * H, SPP, SEED)
    for l in range(n_l):
        lights = sc.lights
        for k in range(n_l):
            if k != l:
                lights[k].color[:] = (0.0, 0.0, 0.0)
        one = load_scene(name)
        one.update(lights=list(lights))
        want = SphereOracle(one.raw).render(one.camera, W, H, one.max_depth, spp=SPP, offsets=off)["rgb_f64"]
        assert np.allclose(lgs.groups[l] + lgs.rest, want, rtol=1e-9, atol=1e-12), (name, l)
    # caller-built rays (rh_trace_rays): the oracle's traceRay with sphere lights
    rays = camera_rays(sc.camera, W, H)
    rad = rh.traceRay(sc, rays[:, :3].copy(), rays[:, 3:].copy(), sc.max_depth, want_hit_ids=True)
    col, ids, cnt = SphereOracle(sc.raw).trace_batch(rays, sc.max_depth)
    assert np.array_equal(rad.hit_ids, ids), name
    assert np.allclose(rad.colors, col, rtol=1e-9, atol=1e-12, equal_nan=True), name
    for k in RAYS:
        assert rad.stats[k] == cnt[k], (name, k)
    # rh_multi_render: one GPU, and two where present
    for n_gpus in (1, 2):
        if n_gpus > torch.cuda.device_count():
            continue
        try:
            multi = rh.render_multi(j, n_gpus, spp=SPP, seed=SEED)
        finally:
            rh.multi_shutdown([sc])
        same(sc, multi.pixels, plain.pixels, (name, "multi", n_gpus))
        for k in RAYS:
            assert multi.stats[k] == plain.stats[k], (name, n_gpus, k)


def ref_linear(j):
    return render_linear(j, spp=SPP, seed=SEED).linear


# ---------------------------------------------------------------- 4. updates and light tables
def tables(sc):
    t = sc.light_tables()
    return t["index"].tobytes(), t["maps"].view(np.uint32).tobytes(), None if t["lit"] is None else t["lit"].tobytes(), t["res"]


def info4(sc):
    info = (C.c_uint32 * 4)()
    capi.check(capi.lib().rh_scene_light_tables(sc.device, info, None, None, None))
    return list(info)


@pytest.mark.parametrize("name", ["dragon_low", "cornellBox"])
def test_updates_equal_a_fresh_create(name):
    base = load_scene(name).lights
    pts = [i for i, L in enumerate(base) if L.kind == P]

    def edit(kind_of, radius_of):
        out = []
        for i, L in enumerate(base):
            L2 = capi.rh_light.from_buffer_copy(L)
            if i in pts:
                L2.kind, L2.radius = kind_of(i), radius_of(i, L.radius)
            out.append(L2)
        return out

    steps = [edit(lambda i: S, lambda i, r: r),                                 # point -> sphere
             edit(lambda i: S, lambda i, r: 3 * r),                             # radius edit of sphere lights
             edit(lambda i: S if i == pts[0] else P, lambda i, r: 3 * r),        # sphere -> point (one stays)
             edit(lambda i: P, lambda i, r: r)]                                  # all back to points
    sc = load_scene(name)
    sc.device
    for k, lights in enumerate(steps):
        info = sc.update(lights=lights)
        if k == 1:
            assert info["colours_only"] == 0, info  # a sphere light's radius is geometry
        if k == 2:
            assert info["maps_rasterised"] > 0 or name == "cornellBox", info
        fresh = with_lights(name, lights)
        assert tables(sc) == tables(fresh), (name, k)
        assert info4(sc) == info4(fresh), (name, k)
        a = rh.render(job(sc), spp=SPP, seed=SEED, want_hit_ids=True)
        b = rh.render(job(fresh), spp=SPP, seed=SEED, want_hit_ids=True)
        assert a.pixels.tobytes() == b.pixels.tobytes() and np.array_equal(a.hit_ids, b.hit_ids), (name, k)
        fresh.close()


@pytest.mark.parametrize("setup", ["device", "host"])
def test_point_light_tables_are_those_without_the_sphere_lights(setup, monkeypatch):
    if setup == "host":
        monkeypatch.setenv("RAYHS_B200_SETUP", "host")
    else:
        monkeypatch.delenv("RAYHS_B200_SETUP", raising=False)
    base = list(load_scene("dragon_low").lights)
    spheres = [light(S, (0.2, 0.5, 0.3), (5, 5, 5), 0.2), light(S, (-0.3, 0.1, 0.4), (5, 5, 5), 0.15)]
    a, b = with_lights("dragon_low", base + spheres), with_lights("dragon_low", base)
    ta, tb = a.light_tables(), b.light_tables()
    n = len(base)
    assert ta["res"] == tb["res"] and ta["maps"].view(np.uint32).tobytes() == tb["maps"].view(np.uint32).tobytes()
    assert ta["index"][:n].tobytes() == tb["index"][:n].tobytes()
    assert (ta["index"][n:] == 0xFFFFFFFF).all()
    assert ta["lit"] is not None and tb["lit"] is not None and ta["lit"].tobytes() == tb["lit"].tobytes()
    assert len(ta["maps"]) > 0
    check_scene(a, ("tables", setup), 24, 16, 2)


BAD_RADII = [-0.1, -math.inf, math.inf, math.nan]


@pytest.mark.parametrize("radius", BAD_RADII)
def test_bad_radius_is_an_argument_error(radius):
    lights = list(load_scene("cornellBox").lights) + [light(S, (0, 0.5, 0.5), (1, 1, 1), radius)]
    sc = with_lights("cornellBox", lights)
    with pytest.raises(capi.RayHsError) as e:
        sc.device
    assert e.value.code == capi.RH_ERR_ARG and "radius" in str(e.value)
    ok = load_scene("cornellBox")
    ok.device
    before = rh.render(job(ok), spp=1).pixels
    with pytest.raises(capi.RayHsError) as e:
        ok.update(lights=lights)
    assert e.value.code == capi.RH_ERR_ARG
    assert rh.render(job(ok), spp=1).pixels.tobytes() == before.tobytes()  # the scene is unchanged
    # the edges that are valid: radius 0 and -0; a point light keeps the value-domain behaviour of odd radii
    for r in (0.0, -0.0):
        with_lights("cornellBox", lights[:-1] + [light(S, (0, 0.5, 0.5), (1, 1, 1), r)]).device
    with_lights("cornellBox", lights[:-1] + [light(P, (0, 0.5, 0.5), (1, 1, 1), radius)]).device
