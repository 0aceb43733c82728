"""GPU tests of the value domain: built scenes with non-finite and extreme material, light, texture and normal values
(tests/value_cases.py), extreme sample offsets and caller rays, against the oracle.  Stricter than assert_parity: NaN
and +-inf positions equal, finite linear colours bit for bit where every term has weight 1 (else within the radiance
queries' rtol), every RGB8 byte equal (up to pixels within that rtol of a k/255 boundary), hit ids, the five ray counts
and negative_channels equal, under both shadow schedules and without light maps."""
import math

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import COUNT_NAMES, OracleScene, camera_rays
from tests.util import ATOL, RTOL, load_scene
from tests import value_cases as vc

pytestmark = pytest.mark.gpu

VARIANTS = [dict(shadow="pooled"), dict(shadow="split"), dict(shadow="pooled", light_maps=False)]
ORC_COUNTS = ("primary", "reflect", "probe", "exit", "shadow")


def first(mask, k=8):
    return np.argwhere(mask)[:k].tolist()


def assert_linear(got, want, exact, what):
    """NaN and +-inf at the same places (same signs); finite values bit for bit when `exact`, else within RTOL / ATOL."""
    got, want = np.asarray(got).reshape(-1, 3), np.asarray(want).reshape(-1, 3)
    for name, f in (("NaN", np.isnan), ("+inf", np.isposinf), ("-inf", np.isneginf)):
        bad = f(got) != f(want)
        assert not bad.any(), (what, name, bad.sum(), [(i, got[i[0]].tolist(), want[i[0]].tolist()) for i in first(bad, 4)])
    fin = np.isfinite(want)
    bad = fin & ((got != want) if exact else ~np.isclose(got, want, rtol=RTOL, atol=ATOL))
    assert not bad.any(), (what, "finite", bad.sum(), [(i, got[i[0]].tolist(), want[i[0]].tolist()) for i in first(bad, 4)])


def assert_bytes(got, ref, what):
    """Every byte equal, except on pixels with an oracle channel within RTOL of a k/255 boundary (listed on failure)."""
    bad = (got != ref["rgb_u8"]).any(axis=-1)
    if not bad.any():
        return
    v = 255 * ref["rgb_f64"]
    near = (np.isfinite(v) & (np.abs(v - np.round(v)) <= RTOL * np.abs(v) + 255 * ATOL)).any(axis=-1)
    assert not (bad & ~near).any(), (what, "bytes", first(bad & ~near), "(near k/255:", first(bad & near), ")")


def negative_pixels(ref):
    return int((ref["rgb_int"] < 0).any(axis=-1).sum())


def check(rs, depth, exact, spp=1, offsets=None, seed=None, what=""):
    """Every comparison of the module for one scene and max_depth; returns the oracle's render."""
    w, h = rs.width, rs.height
    job = rh.Rendering(rs, rs.camera, w, h, depth)
    if seed is not None:
        offsets_ref = rh.sample_offsets(w * h, spp, seed)
    else:
        offsets_ref = None if offsets is None else np.asarray(offsets, dtype=np.float64)
    ref = OracleScene(rs.raw).render(rs.camera, w, h, depth, spp=spp, offsets=offsets_ref)
    want_counts = tuple(ref["rays"][k] for k in ORC_COUNTS)
    neg = negative_pixels(ref)
    for kw in VARIANTS:
        tag = (what, depth, kw)
        src = dict(seed=seed) if seed is not None else dict(offsets=offsets)
        img = rh.render(job, spp=spp, want_hit_ids=True, **src, **kw)
        assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"]), (tag, "hit ids")
        assert tuple(img.stats[k] for k in COUNT_NAMES) == want_counts, (tag, "ray counts")
        assert img.stats["negative_channels"] == neg, (tag, "negative_channels", img.stats["negative_channels"], neg)
        assert_bytes(img.pixels, ref, tag)
        acc = rh.Accumulator(job)
        a = acc.add(spp, offsets=offsets, **kw) if seed is None else acc.add(spp, offsets=offsets_ref, **kw)
        acc.close()
        assert_linear(a.linear, ref["rgb_f64"], exact, (tag, "accumulate linear"))
        assert a.stats["negative_channels"] == neg, (tag, "accumulate negative_channels")
        assert_bytes(a.pixels, ref, (tag, "accumulate"))
        if spp == 1 and offsets is None and seed is None:
            rays = camera_rays(rs.camera, w, h)
            r = rh.traceRay(rs, np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:]), depth, want_hit_ids=True, **kw)
            assert_linear(r.colors, ref["rgb_f64"], exact, (tag, "traceRay"))
            assert np.array_equal(r.hit_ids, ref["hit_ids"].reshape(-1, 2)), (tag, "traceRay hit ids")
            assert tuple(r.stats[k] for k in COUNT_NAMES) == want_counts, (tag, "traceRay ray counts")
    src = dict(seed=seed) if seed is not None else dict(offsets=offsets)
    shards = [rh.render(job, spp=spp, shard_index=i, shard_count=2, band_height=8, **src) for i in range(2)]
    assert sum(s.stats["negative_channels"] for s in shards) == neg, (what, depth, "2-shard negative_channels")
    return ref


CASES = vc.cases()


@pytest.mark.parametrize("name,factory,depths,exact", CASES, ids=[c[0] for c in CASES])
def test_value_case_equals_the_oracle(name, factory, depths, exact):
    rs = factory()
    for depth in depths:
        check(rs, depth, exact or depth == 0, what=name)


def test_the_cases_reach_the_values_they_are_about():
    """The case table is not vacuous: the oracle's frames hold NaN, +-inf and negative channels where intended."""
    def frame(name, depth=0):
        f = dict((c[0], c[1]) for c in CASES)[name]()
        return OracleScene(f.raw).render(f.camera, f.width, f.height, depth)
    for sign in "+-":
        r = frame(f"lambert_diffuse_flat_{sign}")
        assert np.isnan(r["rgb_f64"][..., 0]).any()   # 0 * inf in the culled pairs
    assert np.isnan(frame("mirror_ior_-1.0", 0)["rgb_f64"]).any() and np.isnan(frame("mirror_ior_-1.0", 3)["rgb_f64"]).any()
    assert np.isinf(frame("light_radius_minus_distance")["rgb_f64"]).any()
    assert negative_pixels(frame("toint_showuv")) > 100 and negative_pixels(frame("toint_emmit")) > 0


# ---------------------------------------------------------------- sample offsets
def departure(hits):
    """The rays of DESIGN §3's documented departure: the reference's closest hit has time NaN or +inf (a NaN ray
    passes the reference's triangle test and wins GHC's minimumBy; a plane accepts time = +inf), where the wavefront
    reports a miss."""
    return (hits["object"] >= 0) & ~np.isfinite(hits["t"])


def offsets_frame(dtype, values):
    rng = np.random.RandomState(17)
    off = rng.uniform(0, 1, size=(vc.W * vc.H, 4, 2))
    pick = rng.randint(0, len(values), size=off.shape)
    use = rng.uniform(size=off.shape) < 0.3
    off[use] = np.array(values)[pick[use]]
    return off.astype(dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_far_sample_offsets(dtype):
    """+-1e6 and -0.0 offsets in a 4-spp frame: camera rays far off the image."""
    rs = vc.lit_stage(vc.point())
    check(rs, 0, True, spp=4, offsets=offsets_frame(dtype, [1e6, -1e6, -0.0, 0.25, 0.75]), what=str(dtype))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_non_finite_sample_offsets(dtype):
    """NaN and +-inf offsets make NaN and infinite camera rays: every sample's hit id is the oracle's, except the
    documented departure (the oracle's hit time NaN or +inf), where the wavefront reports a miss."""
    rs = vc.lit_stage(vc.point())
    w, h, spp = rs.width, rs.height, 4
    off = offsets_frame(dtype, [math.nan, math.inf, -math.inf, 0.5])
    off64 = off.astype(np.float64).reshape(h, w, spp, 2)
    orc = OracleScene(rs.raw)
    ref = orc.render(rs.camera, w, h, 0, spp=spp, offsets=off64)
    rays = np.array([np.concatenate(orc.ray_from_pixel(rs.camera, w, h, x + off64[y, x, k, 0], y + off64[y, x, k, 1]))
                     for y in range(h) for x in range(w) for k in range(spp)])
    dep = departure(orc.closest_batch(rays)).reshape(h, w, spp)
    assert dep.any() and not dep.all()
    for kw in VARIANTS:
        ids = rh.render(rh.Rendering(rs, rs.camera, w, h, 0), spp=spp, offsets=off, want_hit_ids=True, **kw).hit_ids.reshape(h, w, spp, 2)
        assert np.array_equal(ids[~dep], ref["hit_ids"][~dep]), kw
        assert (ids[dep] == -1).all(), kw


def test_splitmix_offsets_on_a_value_scene():
    check(vc.MATERIALS["nan"][0](*vc.MATERIALS["nan"][1]), 0, True, spp=4, seed=99, what="splitmix")


# ---------------------------------------------------------------- progressive calls
def test_accumulator_keeps_the_oracles_nan_and_inf_pattern_over_calls():
    rs = vc.lambert(-1, "plastic", "checker")
    w, h, spp = rs.width, rs.height, 2
    job = rh.Rendering(rs, rs.camera, w, h, 2)
    stream = rh.sample_offsets(w * h, 2 * spp, 5).reshape(w * h, 2 * spp, 2)
    ref = OracleScene(rs.raw).render(rs.camera, w, h, 2, spp=2 * spp, offsets=stream)
    acc = rh.Accumulator(job)
    acc.add(spp, offsets=np.ascontiguousarray(stream[:, :spp]))
    img = acc.add(spp, offsets=np.ascontiguousarray(stream[:, spp:]))
    acc.close()
    assert_linear(img.linear, ref["rgb_f64"], False, "two accumulate calls")
    assert img.stats["negative_channels"] == negative_pixels(ref)
    assert_bytes(img.pixels, ref, "two accumulate calls")


# ---------------------------------------------------------------- caller rays
EDGE = [math.nan, math.inf, -math.inf, 5e-324, 2.0 ** 100, 2.0 ** -100, 1e300, -0.0]


def edge_rays(sc, n=2000, seed=4):
    rays = camera_rays(sc.camera, 40, 30)
    rng = np.random.RandomState(seed)
    rays = rays[rng.randint(0, len(rays), n)].copy()
    pick = rng.randint(0, len(EDGE), size=rays.shape)
    use = rng.uniform(size=rays.shape) < 0.15
    rays[use] = np.array(EDGE)[pick[use]]
    return rays


@pytest.mark.parametrize("which", ["cornellBox", "lambert", "mesh_nan"])
def test_caller_rays_with_extreme_components(which):
    """closestIntersection and traceRay of rays with NaN, +-inf, subnormal, 2^+-100 and 1e300 components against the
    oracle: equal on every ray outside the documented departure, a miss on the rays inside it.  (mesh_nan's NaN vertex
    normals reflect into NaN rays, which are inside it: its radiance is compared without reflections.)"""
    sc = {"cornellBox": lambda: load_scene("cornellBox"), "lambert": lambda: vc.lambert(1, "diffuse", "flat"),
          "mesh_nan": lambda: vc.NORMALS["mesh_nan"][0](*vc.NORMALS["mesh_nan"][1])}[which]()
    rays = edge_rays(sc)
    want = OracleScene(sc.raw).closest_batch(rays)
    dep = departure(want)
    assert dep.any() and not dep.all()
    hits = rh.closestIntersection(sc, np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:]))
    got = np.stack([hits.object, hits.tri], axis=1)
    assert np.array_equal(got[~dep], np.stack([want["object"], want["tri"]], axis=1)[~dep]), which
    assert (got[dep] == -1).all(), which
    keep = rays[~dep]
    orc = OracleScene(sc.raw)
    for depth in ((0,) if which == "mesh_nan" else (0, 2)):
        colors, ids, counts = orc.trace_batch(keep, depth)
        for kw in VARIANTS:
            r = rh.traceRay(sc, np.ascontiguousarray(keep[:, :3]), np.ascontiguousarray(keep[:, 3:]), depth, want_hit_ids=True, **kw)
            assert np.array_equal(r.hit_ids, ids), (which, depth, kw)
            assert_linear(r.colors, colors, False, (which, depth, kw))
            assert {k: r.stats[k] for k in COUNT_NAMES} == counts, (which, depth, kw)


# ---------------------------------------------------------------- the documented departure (DESIGN §3)
@pytest.mark.parametrize("bounces", [9, 10])
def test_product_order_departure_is_the_documented_one(bounces):
    """A ray zigzags between two Mirror planes with ior = nextafter(-1, 0): r0 = (2 / 2^-53)^2 = 2^108, at normal incidence
    fresnel = r0 and l.n = 1, so every bounce has the factor 2^108, exactly.  It then hits an emitter of 2^-1000.  The
    reference nests 2^108 * (1 * (... * 2^-1000)), the wavefront forms (2^108)^bounces first: 9 bounces give 2^-28 on
    both sides, bit for bit; at 10 the weight 2^1080 overflows and the wavefront gives +inf where the reference gives 2^80."""
    ior = math.nextafter(-1.0, 0.0)
    mats = [{"kind": "mirror", "ior": ior}, {"kind": "emmit", "color1": (2.0 ** -1000, 2.0 ** -1000, 0.0)}]
    objs = [{"kind": "plane", "point": (0, 0, 0), "normal": (0, 0, 1), "tangent": (1, 0, 0), "material": 0},
            {"kind": "plane", "point": (0, 0, 2), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 0},
            {"kind": "sphere", "center": (2.0 * bounces, 0, 1), "radius": 0.3, "material": 1}]
    rs = vc.scene(objs, mats, [])
    rays = np.array([[0.0, 0.0, 1.0, 1.0, 0.0, -1.0]])
    want, _, counts = OracleScene(rs.raw).trace_batch(rays, bounces)
    assert counts["rays_reflect"] == bounces
    assert want[0, 0] == 2.0 ** (108 * bounces - 1000)
    got = rh.traceRay(rs, rays[:, :3], rays[:, 3:], bounces).colors
    if bounces == 9:
        assert got[0, 0] == want[0, 0] and got[0, 2] == 0, got
    else:
        assert np.isposinf(got[0, 0]) and np.isnan(got[0, 2]), got   # inf * 0 in blue


@pytest.mark.parametrize("kind", ["plastic", "transparent"])
@pytest.mark.parametrize("max_depth", [10, 11, 12])
def test_black_under_an_overflowed_weight_is_absorbed_by_the_addition(kind, max_depth):
    """The corridor above with a lit Plastic (or Transparent) sphere in place of the emitter: the weight of the sphere's
    hit has overflowed to inf after 10 bounces of 2^108, but every factor is finite.  At maxDepth (10) fresnel * black
    is +-0 and Plastic's diff + 0 keeps diff, so the reference gives inf * diff = [-inf, inf, inf], as does w * diff;
    deeper, the sphere's reflection child starts a new chain of finite factors whose black ends add nothing either."""
    ior = math.nextafter(-1.0, 0.0)
    mats = [{"kind": "mirror", "ior": ior}, {"kind": kind, "ior": 1.5, "color1": (-0.5, 0.6, 0.7)}]
    objs = [{"kind": "plane", "point": (0, 0, 0), "normal": (0, 0, 1), "tangent": (1, 0, 0), "material": 0},
            {"kind": "plane", "point": (0, 0, 2), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 0},
            {"kind": "sphere", "center": (20.0, 0, 1), "radius": 0.3, "material": 1}]
    rs = vc.scene(objs, mats, [vc.point(vec=(19.4, 0, 1), color=(1, 1, 1))])
    rays = np.array([[0.0, 0.0, 1.0, 1.0, 0.0, -1.0]])
    want, ids, counts = OracleScene(rs.raw).trace_batch(rays, max_depth)
    if kind == "plastic" and max_depth == 10:
        assert np.isneginf(want[0, 0]) and np.isposinf(want[0, 1:]).all(), want
    for kw in VARIANTS:
        r = rh.traceRay(rs, rays[:, :3], rays[:, 3:], max_depth, want_hit_ids=True, **kw)
        assert_linear(r.colors, want, False, (kind, max_depth, kw))
        assert np.array_equal(r.hit_ids, ids) and {k: r.stats[k] for k in COUNT_NAMES} == counts, (kind, max_depth, kw)
