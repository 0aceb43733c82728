"""CPU tests of sphere lights (RH_LIGHT_SPHERE, beside rh_light in include/rayhs_b200.h): a numpy restatement of the light
sample written from the header against tests/sphere_light_oracle.cpp, the sample's properties, the sphere-light oracle
pinned to the plain oracle on every shipped pack, the JSON type, the update planner's classes for the new kind, and the
Python helper."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from rayhs_b200 import capi
from tests import lens_oracle
from tests.sphere_light_oracle import SphereOracle
from tests.util import GOLDEN, SCENES, load_scene, temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U64 = np.uint64
MASK = (1 << 64) - 1


# ---------------------------------------------------------------- the sample, restated from the header
def mix64(z):
    z = (z ^ (z >> U64(30))) * U64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> U64(27))) * U64(0x94D049BB133111EB)
    return z ^ (z >> U64(31))


def uniform(key, k):
    z = key + (U64(k) + U64(1)) * U64(0x9E3779B97F4A7C15)
    return (mix64(z) >> U64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def sample(center, r, li, p):
    """L' [n, 3] of the light (centre, radius r, index li) for shading points p [n, 3], and whether a triple was taken."""
    p = np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 3)
    bits = p.view(U64)
    with np.errstate(over="ignore"):
        key = bits[:, 0] ^ mix64(bits[:, 1] ^ mix64(bits[:, 2] ^ mix64(np.full(len(p), li, dtype=U64))))
        abc = np.zeros((len(p), 3))
        taken = np.zeros(len(p), dtype=bool)
        for j in range(16):
            t = np.stack([2 * uniform(key, 3 * j + c) - 1 for c in range(3)], axis=1)
            ok = ~taken & ((t[:, 0] * t[:, 0] + t[:, 1] * t[:, 1]) + t[:, 2] * t[:, 2] < 1)
            abc[ok] = t[ok]
            taken |= ok
    c = np.asarray(center, dtype=np.float64)
    return np.stack([c[k] + r * abc[:, k] for k in range(3)], axis=1), taken


def sphere_scene(name, radius=None, which=None):
    """The pack with its point lights (or the ones listed in `which`) turned into sphere lights of their own radius (or
    `radius`), before the device copy."""
    sc = load_scene(name)
    lights = sc.lights
    for i, L in enumerate(lights):
        if L.kind == capi.RH_LIGHT_POINT and (which is None or i in which):
            L.kind = capi.RH_LIGHT_SPHERE
            if radius is not None:
                L.radius = radius
    sc.update(lights=list(lights))
    return sc


def test_restatement_equals_the_oracle_sample_bit_for_bit():
    sc = sphere_scene("cornellBox")
    orc = SphereOracle(sc.raw)
    rng = np.random.RandomState(7)
    p = np.concatenate([rng.uniform(-3, 3, (2000, 3)), rng.normal(0, 1e-3, (500, 3)),
                        np.array([[0.0, -0.0, 0.0], [1e300, -1e-300, 5.0], [np.inf, 0, 0], [np.nan, 1, 2]])])
    for li, L in enumerate(sc.lights):
        want, _ = sample(L.vec, L.radius, li, p)
        got = orc.sphere_points(li, p)
        assert got.tobytes() == want.tobytes(), li
    # known answers: the first draws of a fixed point (their bits pin the hash and the stream)
    want, taken = sample((1.0, 2.0, 3.0), 0.5, 3, [[0.25, -0.5, 1.0]])
    L = capi.rh_light(kind=capi.RH_LIGHT_SPHERE, vec=(1.0, 2.0, 3.0), color=(1, 1, 1), radius=0.5)
    raw = capi.rh_raw_scene.from_buffer_copy(sc.raw.contents)
    arr = (capi.rh_light * 4)(L, L, L, L)
    raw.lights, raw.n_lights = C.cast(arr, C.POINTER(capi.rh_light)), 4
    got = SphereOracle(C.pointer(raw)).sphere_points(3, [[0.25, -0.5, 1.0]])
    assert taken[0] and got.tobytes() == want.tobytes()
    assert np.abs(got - np.array([1.0, 2.0, 3.0])).max() > 0  # (a draw, not the centre)


def test_samples_lie_in_the_closed_ball_fill_it_and_do_not_depend_on_call_order():
    c, r = np.array([0.5, -1.25, 2.0]), 0.75
    rng = np.random.RandomState(11)
    p = rng.uniform(-5, 5, (40000, 3))
    s, taken = sample(c, r, 1, p)
    d = np.sqrt(((s - c) ** 2).sum(axis=1))
    assert (d <= r * (1 + 1e-15)).all()
    assert taken.mean() > 0.999  # only (1 - pi/6)^16 ~ 7e-6 of the points keep the centre
    # uniform in the ball: the fraction within r/2 is 1/8, the mean of each coordinate 0
    assert abs((d[taken] < r / 2).mean() - 0.125) < 0.01
    assert np.abs((s[taken] - c).mean(axis=0)).max() < 0.01 * r
    # deterministic, per point and light: reversed order, single calls and other light indices
    s2, _ = sample(c, r, 1, p[::-1])
    assert s2[::-1].tobytes() == s.tobytes()
    assert sample(c, r, 1, p[123:124])[0].tobytes() == s[123:124].tobytes()
    assert not np.array_equal(sample(c, r, 2, p)[0], s)


def test_no_draw_falls_back_to_the_centre():
    rng = np.random.RandomState(5)
    c, r = (1.5, -2.0, 0.25), 2.0
    for _ in range(40):
        p = rng.uniform(-1, 1, (200000, 3))
        s, taken = sample(c, r, 0, p)
        if not taken.all():
            break
    else:
        pytest.fail("no point without a draw found")
    q = p[~taken][:1]
    assert s[~taken][0].tolist() == list(c)
    sc = load_scene("cornellBox")
    raw = capi.rh_raw_scene.from_buffer_copy(sc.raw.contents)
    arr = (capi.rh_light * 1)(capi.rh_light(kind=capi.RH_LIGHT_SPHERE, vec=c, color=(1, 1, 1), radius=r))
    raw.lights, raw.n_lights = C.cast(arr, C.POINTER(capi.rh_light)), 1
    assert SphereOracle(C.pointer(raw)).sphere_points(0, q)[0].tolist() == list(c)


# ---------------------------------------------------------------- the sphere-light oracle
@pytest.mark.parametrize("name", [s for s in SCENES if s != "dragon_full"] + ["dragon_full"])
def test_sphere_oracle_is_the_oracle_without_sphere_lights(name):
    """On every shipped pack (none has a sphere light) the restated shading renders the oracle's frames: colours, bytes,
    hit ids and ray counts per class, with and without offsets, and the seeded sample."""
    sc = load_scene(name)
    assert all(L.kind != capi.RH_LIGHT_SPHERE for L in sc.lights)
    orc, sph = OracleScene(sc.raw), SphereOracle(sc.raw)
    w, h, spp = (9, 7, 2) if name == "dragon_full" else (17, 11, 3)
    off = np.random.RandomState(3).uniform(-0.5, 0.5, (w * h, spp, 2))
    for n, o in ((1, None), (spp, off)):
        want, got = orc.render(sc.camera, w, h, sc.max_depth, spp=n, offsets=o), sph.render(sc.camera, w, h, sc.max_depth, spp=n, offsets=o)
        for k in ("rgb_f64", "rgb_u8", "hit_ids"):
            assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).reshape(np.shape(got[k])).tobytes(), (name, n, k)
        assert got["rays"] == want["rays"], (name, n)
    want = orc.render_sample(sc.camera, w, h, sc.max_depth, spp=spp, seed=24, rows=(1, None, 3), cols=(0, None, 2))
    got = sph.render_sample(sc.camera, w, h, sc.max_depth, spp, 24, rows=(1, None, 3), cols=(0, None, 2))
    for k in ("rgb_f64", "rgb_u8", "hit_ids"):
        assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), (name, "sample", k)
    assert got["rays"] == want["rays"]


@pytest.mark.parametrize("name", ["cornellBox", "dragon_superlow"])
def test_sphere_oracle_radius_zero_is_the_point_light_and_a_ball_softens(name):
    point = load_scene(name)
    zero, ball = sphere_scene(name, radius=0.0), sphere_scene(name)
    w, h, spp = 24, 16, 4
    off = np.random.RandomState(1).uniform(-0.5, 0.5, (w * h, spp, 2))
    # radius 0: the falloff of every sphere light is then 0 too, as for the point light of radius 0
    pz = load_scene(name)
    lights = pz.lights
    for L in lights:
        if L.kind == capi.RH_LIGHT_POINT:
            L.radius = 0.0
    pz.update(lights=list(lights))
    a = SphereOracle(zero.raw).render(zero.camera, w, h, zero.max_depth, spp, off)
    b = OracleScene(pz.raw).render(pz.camera, w, h, pz.max_depth, spp=spp, offsets=off)
    assert a["rgb_f64"].tobytes() == b["rgb_f64"].tobytes() and a["rays"] == b["rays"]
    c = SphereOracle(ball.raw).render(ball.camera, w, h, ball.max_depth, spp, off)
    d = OracleScene(point.raw).render(point.camera, w, h, point.max_depth, spp=spp, offsets=off)
    assert c["rays"] == d["rays"]
    assert not np.array_equal(c["rgb_f64"], d["rgb_f64"])


# ---------------------------------------------------------------- front end, planner, Python
def test_json_sphere_light_parses_and_survives_a_pack(tmp_path):
    with open(os.path.join(GOLDEN, "cli_scene.json")) as f:
        scene = json.load(f)
    scene["scene"]["lights"] = [
        {"type": "sphere", "position": {"x": 0.5, "y": 1.5, "z": -0.25}, "color": {"r": 0.9, "g": 0.8, "b": 0.7}, "radius": 0.375},
        {"type": "point", "position": {"x": 1, "y": 2, "z": 3}, "color": {"r": 1, "g": 1, "b": 1}, "radius": 2}]
    p = tmp_path / "sphere.json"
    p.write_text(json.dumps(scene))
    sc = rh.Scene.from_json(str(p), str(tmp_path))
    L = sc.lights
    assert L[0].kind == capi.RH_LIGHT_SPHERE == 2 and L[1].kind == capi.RH_LIGHT_POINT
    assert tuple(L[0].vec) == (0.5, 1.5, -0.25) and tuple(L[0].color) == (0.9, 0.8, 0.7) and L[0].radius == 0.375
    pack = str(tmp_path / "sphere.pack")
    sc.save_pack(pack)
    assert [bytes(x) for x in rh.Scene.from_pack(pack).lights] == [bytes(x) for x in L]
    scene["scene"]["lights"] = [{"type": "sphere", "position": {"x": 0, "y": 0, "z": 0}, "color": {"r": 1, "g": 1, "b": 1}}]
    p.write_text(json.dumps(scene))
    with pytest.raises(capi.RayHsError):
        rh.Scene.from_json(str(p), str(tmp_path))


@pytest.fixture(scope="module")
def planner():
    srcs = [os.path.join(ROOT, "tests", "scene_update_driver.cpp"), os.path.join(ROOT, "rayhs_b200", "csrc", "scene_update.h"),
            os.path.join(ROOT, "include", "rayhs_b200.h")]
    L = temp_library("scene_update", srcs, ["-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared"])
    L.su_classify.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    L.su_lit_mask.restype = C.c_uint32
    L.su_lit_mask.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    L.su_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    return L


def test_update_classes_of_sphere_lights(planner):
    COLOURS, TABLES = 1, 3
    mats = (capi.rh_material * 1)(capi.rh_material(kind=capi.RH_MAT_DIFFUSE))
    objm = (C.c_int32 * 1)(0)

    def lights(*specs):
        return (capi.rh_light * len(specs))(*[capi.rh_light(kind=k, vec=v, color=(1, 1, 1), radius=r) for k, v, r in specs])

    P, S = capi.RH_LIGHT_POINT, capi.RH_LIGHT_SPHERE

    def cls(a, b):
        return planner.su_classify(mats, mats, 1, a, len(a), b, len(b), objm, 1)

    base = lights((P, (0, 1, 0), 0.5), (S, (1, 1, 0), 0.25))
    assert cls(base, lights((P, (0, 1, 0), 0.75), (S, (1, 1, 0), 0.25))) == COLOURS  # a point light's radius is colour
    assert cls(base, lights((P, (0, 1, 0), 0.5), (S, (1, 1, 0), 0.5))) == TABLES  # a sphere light's radius is geometry
    assert cls(base, lights((S, (0, 1, 0), 0.5), (S, (1, 1, 0), 0.25))) == TABLES  # point -> sphere
    assert cls(base, lights((P, (0, 1, 0), 0.5), (P, (1, 1, 0), 0.25))) == TABLES  # sphere -> point
    assert planner.su_lit_mask(base, 2, lights((S, (0, 1, 0), 0.5), (S, (1, 1, 0), 0.5)), 2) == 0b11
    assert planner.su_lit_mask(base, 2, lights((P, (0, 1, 0), 0.9), (S, (1, 1, 0), 0.25)), 2) == 0
    # maps: a sphere light has none; one that becomes a point light is rasterised, a point light that stays keeps its map
    old_index = (C.c_uint32 * 16)(*([0] + [0xFFFFFFFF] * 15))
    steps = (C.c_uint32 * 64)()
    n = planner.su_plan(old_index, base, 2, lights((P, (0, 1, 0), 0.5), (P, (1, 1, 0), 0.25)), 2, 1, 16, steps)
    assert n == 2 and list(steps[:8]) == [0, 0, 0, 0, 0, 1, 1, 0xFFFFFFFF]
    n = planner.su_plan(old_index, base, 2, lights((S, (0, 1, 0), 0.5), (S, (1, 1, 0), 0.25)), 2, 1, 16, steps)
    assert n == 0


def test_python_constant_and_helper_match_the_header():
    with open(os.path.join(ROOT, "include", "rayhs_b200.h")) as f:
        header = f.read()
    enum = re.search(r"enum \{ RH_LIGHT_DIRECTIONAL = 0, RH_LIGHT_POINT = 1, RH_LIGHT_SPHERE = (\d+) \};", header)
    assert enum and int(enum.group(1)) == capi.RH_LIGHT_SPHERE
    L = rh.sphereLight((0.5, -1, 2), np.array([1.0, 0.5, 0.25]), 0.125)
    assert isinstance(L, capi.rh_light) and L.kind == capi.RH_LIGHT_SPHERE
    assert tuple(L.vec) == (0.5, -1.0, 2.0) and tuple(L.color) == (1.0, 0.5, 0.25) and L.radius == 0.125
    sc = load_scene("cornellBox")
    sc.update(lights=list(sc.lights) + [L])
    assert bytes(sc.raw.contents.lights[len(sc.lights) - 1]) == bytes(L)
    assert bytes(sc.flat.contents.lights[len(sc.lights) - 1]) == bytes(L)
