"""CPU tests of the thin-lens camera (RH_PROJ_THIN_LENS, rh_camera in include/rayhs_b200.h): a numpy restatement of the
lens ray, written from the header's rule, against the tests' C++ restatement on the oracle (tests/lens_oracle.py) bit for
bit, and that restatement's renders against the oracle's own for the reference's cameras; radius 0 against the perspective
rays; where the lens origins lie and how they are distributed; sharpness at the focus plane; the JSON `thinLens`
projection, the pack round trip, and the Python constant and helper."""
import json
import math
import os
import re

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from oracle.orc import camera_rays as oracle_camera_rays
from rayhs_b200 import capi
from tests import lens_oracle
from tests.lens_oracle import camera_rays
from tests.util import GOLDEN, SCENES, load_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = np.uint64(0x9E3779B97F4A7C15)


# ---------------------------------------------------------------- the rule, restated in numpy
def mix64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z ^ (z >> np.uint64(30))
        z = z * np.uint64(0xBF58476D1CE4E5B9)
        z = z ^ (z >> np.uint64(27))
        z = z * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def uniform(key, k):
    """Value k of the SplitMix64 stream seeded with key, as a double in [0, 1)."""
    with np.errstate(over="ignore"):
        z = mix64(key + (np.uint64(k) + np.uint64(1)) * GAMMA)
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def lens_point(px, py):
    """(a, b, attempts): the lens point of each image position and the attempts it took (17: none succeeded)."""
    px, py = np.asarray(px, dtype=np.float64), np.asarray(py, dtype=np.float64)
    key = px.view(np.uint64) ^ mix64(py.view(np.uint64))
    a, b = np.zeros_like(px), np.zeros_like(px)
    tries = np.full(px.shape, 17)
    todo = np.ones(px.shape, dtype=bool)
    for j in range(16):
        x = 2 * uniform(key, 2 * j) - 1
        y = 2 * uniform(key, 2 * j + 1) - 1
        take = todo & ((x * x) + (y * y) < 1)
        a[take], b[take], tries[take] = x[take], y[take], j + 1
        todo &= ~take
    return a, b, tries


def normalize(v):
    return (1 / np.sqrt(v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1] + v[..., 2] * v[..., 2]))[..., None] * v


def cross(a, b):
    return np.array([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]])


def look_at(cam):
    """Rows of lookAt(position, target, up): the columns right, up, forward."""
    pos, tgt, tup = np.array(cam.position[:]), np.array(cam.target[:]), np.array(cam.up[:])
    forward = normalize(tgt - pos)
    right = normalize(cross(tup, forward))
    up = cross(forward, right)
    return np.stack([right, up, forward], axis=1), pos


def apply(m, v):
    return np.stack([m[r, 0] * v[..., 0] + m[r, 1] * v[..., 1] + m[r, 2] * v[..., 2] for r in range(3)], axis=-1)


def lens_rays(cam, w, h, xy):
    """rays [n, 6] of the thin-lens camera at image positions xy [n, 2] (the header's steps 1-5)."""
    px, py = xy[:, 0].astype(np.float64), xy[:, 1].astype(np.float64)
    w, h = float(w), float(h)
    aspect = w / h
    apw, aph = (w, w / aspect) if aspect > 1 else (aspect * h, h)
    f = 0.5 * h / (math.tan(0.5) * cam.fovy)
    vx = apw * (px - (w / 2)) / w
    vy = aph * ((-py) + (h / 2)) / h
    d = normalize(np.stack([vx, vy, np.full_like(vx, f)], axis=-1))
    m, p = look_at(cam)
    R, F = cam.proj_width, cam.proj_height
    if R == 0:
        return np.concatenate([np.zeros_like(d) + p, apply(m, d)], axis=1)
    a, b, _ = lens_point(px, py)
    L = np.stack([R * a, R * b, np.zeros_like(a)], axis=-1)
    s = F / d[:, 2]
    P = np.stack([s * d[:, 0], s * d[:, 1], s * d[:, 2]], axis=-1)
    e = normalize(P - L)
    return np.concatenate([apply(m, L) + p, apply(m, e)], axis=1)


# ---------------------------------------------------------------- cameras and image positions
def lens(cam, R, F, fovy=None):
    c = rh.thinLens(cam, R, F)
    if fovy is not None:
        c.fovy = fovy
    elif not c.fovy > 0:
        c.fovy = 1.0  # (an orthographic pack camera)
    return c


def positions(w, h, n_off=2, seed=0):
    """Every pixel of a w x h frame with n_off seeded offsets each (x at column 0 may be negative), plus the corners and
    the edge rows at +-0.5."""
    rng = np.random.RandomState(seed)
    rows, cols = np.divmod(np.arange(h * w), w)
    xy = [np.stack([cols + rng.uniform(-0.5, 0.5, cols.size), rows + rng.uniform(-0.5, 0.5, rows.size)], axis=1) for _ in range(n_off)]
    edges = [(-0.5, -0.5), (w - 0.5, h - 0.5), (-0.5, h - 0.5), (w - 0.5, -0.5), (0, 0), (-0.25, h - 1), (w / 2, h / 2)]
    xy.append(np.array(edges, dtype=np.float64))
    out = np.concatenate(xy)
    assert (out[:, 0] < 0).any()
    return out


CASES = [(0.05, 4.0, None, 16, 9), (0.3, 1.5, 0.7, 9, 16), (1e-3, 10.0, 1.2, 13, 13), (2.0, 0.25, 0.4, 40, 3), (0.12, 3.3, None, 1, 7)]


@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("R,F,fovy,w,h", CASES)
def test_restatement_equals_the_oracle_bit_for_bit(name, R, F, fovy, w, h):
    cam = lens(load_scene(name).camera, R, F, fovy)
    xy = positions(w, h, seed=w * h)
    got, want = camera_rays(cam, w, h, xy), lens_rays(cam, w, h, xy)
    assert got.tobytes() == want.tobytes(), (name, int((got != want).sum()))


@pytest.mark.parametrize("name", SCENES)
def test_radius_zero_is_the_perspective_camera(name):
    sc = load_scene(name)
    for w, h in ((16, 9), (9, 16)):
        for F in (0.5, 7.0):
            c = lens(sc.camera, 0.0, F)
            persp = capi.rh_camera.from_buffer_copy(c)
            persp.projection = capi.RH_PROJ_PERSPECTIVE
            xy = positions(w, h)
            got = camera_rays(c, w, h, xy)
            assert got.tobytes() == camera_rays(persp, w, h, xy).tobytes(), (name, w, h, F)
            assert got.tobytes() == lens_rays(c, w, h, xy).tobytes()
            c.proj_width = -0.0  # (-0 is >= 0 and == 0: a radius of 0 too)
            assert camera_rays(c, w, h, xy).tobytes() == got.tobytes()


@pytest.mark.parametrize("name", ["cornellBox", "transform", "outScene"])
def test_the_lens_oracle_is_the_oracle_for_the_references_cameras(name):
    """For orthographic and perspective cameras tests/lens_oracle.py casts the oracle's rays and renders the oracle's
    frames: colours, bytes, hit ids and ray counts, with and without offsets, and the seeded row sample."""
    sc = load_scene(name)
    orc = OracleScene(sc.raw)
    w, h, spp = 19, 11, 3
    ortho = capi.rh_camera.from_buffer_copy(sc.camera)
    ortho.projection = capi.RH_PROJ_ORTHOGRAPHIC
    for cam in (sc.camera, ortho):
        xy = positions(w, h)
        assert camera_rays(cam, w, h, xy).tobytes() == oracle_camera_rays(cam, w, h, xy).tobytes()
        off = np.random.RandomState(3).uniform(-0.5, 0.5, (w * h, spp, 2))
        for n, o in ((1, None), (spp, off)):
            want, got = orc.render(cam, w, h, sc.max_depth, spp=n, offsets=o), lens_oracle.render(orc, cam, w, h, sc.max_depth, spp=n, offsets=o)
            for k in ("rgb_f64", "rgb_u8", "hit_ids"):
                assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).reshape(np.shape(got[k])).tobytes(), (name, n, k)
            assert got["rays"] == want["rays"], (name, n)
        want = orc.render_sample(cam, w, h, sc.max_depth, spp=spp, seed=24, rows=(1, None, 4), cols=(2, None, 3))
        got = lens_oracle.render_sample(orc, cam, w, h, sc.max_depth, spp, 24, rows=(1, None, 4), cols=(2, None, 3))
        for k in ("rows", "cols", "rgb_f64", "rgb_u8", "hit_ids"):
            assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), (name, "sample", k)
        assert got["rays"] == want["rays"]
    seeded = lens_oracle.splitmix_offsets(24, np.arange(w * h), spp)
    import rayhs_b200 as rh_

    assert seeded.tobytes() == rh_.sample_offsets(w * h, spp, 24).tobytes()


def camera_space(cam, rays):
    m, p = look_at(cam)
    return (rays[:, :3] - p) @ m, rays[:, 3:] @ m  # m is orthonormal: m^T (x - p), m^T d


N_DIST = 1_000_000


def test_lens_points_cover_the_disk_uniformly():
    sc = load_scene("cornellBox")
    R, F, w, h = 0.4, 3.0, 1000, 1000
    cam = lens(sc.camera, R, F)
    xy = positions(w, h, n_off=1, seed=5)[:N_DIST]
    rays = camera_rays(cam, w, h, xy)
    o, _ = camera_space(cam, rays)
    # the origins lie in the plane of the right and up axes through the position, within R of it
    assert np.abs(o[:, 2]).max() <= 1e-12 * R
    r2 = o[:, 0] ** 2 + o[:, 1] ** 2
    assert r2.max() <= R * R * (1 + 1e-12)
    # a uniform disk of radius R: mean 0 (sd R/2 per axis), E[r^2] = R^2/2 (sd R^2/sqrt(12)); 6 sigma
    n = len(xy)
    assert n == N_DIST
    for k in range(2):
        assert abs(o[:, k].mean()) <= 6 * (R / 2) / math.sqrt(n), k
    assert abs(r2.mean() - R * R / 2) <= 6 * (R * R / math.sqrt(12)) / math.sqrt(n)
    # each quadrant holds a quarter, and the annuli hold their areas' shares
    for sx in (-1, 1):
        for sy in (-1, 1):
            q = ((sx * o[:, 0] > 0) & (sy * o[:, 1] > 0)).mean()
            assert abs(q - 0.25) <= 6 * math.sqrt(0.25 * 0.75 / n)
    for lo, hi in ((0, 0.25), (0.25, 0.5), (0.5, 0.75), (0.75, 1.0)):
        share = ((r2 >= lo * R * R) & (r2 < hi * R * R)).mean()
        assert abs(share - (hi - lo)) <= 6 * math.sqrt((hi - lo) * (1 - hi + lo) / n), (lo, hi)
    # the 16-attempt rule: how many attempts the samples needed (a fall-back to the centre has probability 0.2146^16)
    a, b, tries = lens_point(xy[:, 0], xy[:, 1])
    print(f"lens attempts over {n} samples: max {int(tries.max())}, mean {tries.mean():.4f}")
    assert tries.max() <= 16 and abs(tries.mean() - 4 / math.pi) < 0.01
    tol = 1e-12 * (1 + np.abs(np.array(cam.position)).max())
    assert np.allclose(o[:, 0], R * a, rtol=0, atol=tol) and np.allclose(o[:, 1], R * b, rtol=0, atol=tol)


@pytest.mark.parametrize("name", ["cornellBox", "dragon_low", "transform"])
@pytest.mark.parametrize("R,F", [(0.05, 2.0), (0.5, 0.75), (1.5, 12.0)])
def test_every_lens_ray_meets_the_focus_plane_where_the_pinhole_ray_does(name, R, F):
    sc = load_scene(name)
    w, h = 24, 17
    c = lens(sc.camera, R, F)
    persp = capi.rh_camera.from_buffer_copy(c)
    persp.projection = capi.RH_PROJ_PERSPECTIVE
    xy = positions(w, h, n_off=3, seed=11)
    o, d = camera_space(c, camera_rays(c, w, h, xy))
    _, d0 = camera_space(persp, camera_rays(persp, w, h, xy))
    t = (F - o[:, 2]) / d[:, 2]
    hit = o + t[:, None] * d
    want = (F / d0[:, 2])[:, None] * d0
    err = np.linalg.norm(hit - want, axis=1) / np.linalg.norm(want, axis=1)
    assert err.max() <= 1e-12, (name, R, F, float(err.max()))
    assert np.abs(o[:, :2]).max() > 0.1 * R  # (the origins do move)


# ---------------------------------------------------------------- front end, packs, Python
def lens_json(tmp_path, projection):
    with open(os.path.join(GOLDEN, "cli_scene.json")) as f:
        scene = json.load(f)
    scene["camera"]["projection"] = projection
    p = tmp_path / "lens.json"
    p.write_text(json.dumps(scene))
    return str(p)


def test_json_thin_lens_parses_and_survives_a_pack(tmp_path):
    path = lens_json(tmp_path, {"type": "thinLens", "fovy": 0.75, "aperture": 0.125, "focusDistance": 2.5})
    sc = rh.Scene.from_json(path, str(tmp_path))
    c = sc.camera
    assert c.projection == capi.RH_PROJ_THIN_LENS == 2
    assert (c.fovy, c.proj_width, c.proj_height) == (0.75, 0.125, 2.5)
    assert tuple(c.position) == (0.3, 0.4, -2.5)
    pack = str(tmp_path / "lens.pack")
    sc.save_pack(pack)
    back = rh.Scene.from_pack(pack)
    assert bytes(back.camera) == bytes(c)
    w, h = 12, 7
    rows, cols = np.divmod(np.arange(w * h), w)
    assert camera_rays(back.camera, w, h).tobytes() == lens_rays(c, w, h, np.stack([cols, rows], axis=1)).tobytes()
    for bad in ({"type": "thinLens", "fovy": 0.75, "aperture": 0.125}, {"type": "thinLens", "aperture": 0.1, "focusDistance": 1}):
        with pytest.raises(capi.RayHsError):
            rh.Scene.from_json(lens_json(tmp_path, bad), str(tmp_path))


def test_python_constant_and_helper_match_the_header():
    with open(os.path.join(ROOT, "include", "rayhs_b200.h")) as f:
        header = f.read()
    enum = re.search(r"enum \{ RH_PROJ_ORTHOGRAPHIC = 0, RH_PROJ_PERSPECTIVE = 1, RH_PROJ_THIN_LENS = (\d+) \};", header)
    assert enum and int(enum.group(1)) == capi.RH_PROJ_THIN_LENS
    cam = load_scene("cornellBox").camera
    before = bytes(cam)
    c = rh.thinLens(cam, 0.25, 3.5)
    assert bytes(cam) == before  # a copy
    assert c.projection == capi.RH_PROJ_THIN_LENS and (c.proj_width, c.proj_height) == (0.25, 3.5)
    for k in ("position", "target", "up"):
        assert tuple(getattr(c, k)) == tuple(getattr(cam, k))
    assert c.fovy == cam.fovy and c.near_ == cam.near_
