"""GPU tests of the batched ray queries (rh_closest_intersection / rh_shadow_intersection) against the oracle, ray by
ray: every shipped pack plus two built scenes (> 64 objects: tables read from global memory; 1 000 spheres: the sphere
tree), with the camera rays of the scene's view, seeded incoherent rays and an adversarial set (axis-aligned and
zero-component directions, unnormalised directions, rays through mesh vertices, along edges and in triangle planes,
origins inside spheres and on planes, rays parallel to planes)."""
import zlib

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi
from tests.query_oracle import BatchOracle
from tests.util import SCENES, RawScene, load_scene

pytestmark = pytest.mark.gpu

# Sphere uv goes through CUDA's atan / acos, which are within 2 ulp of the exact value (CUDA C Programming Guide,
# double-precision mathematical functions), against glibc's < 1 ulp; the product with 1/pi rounds once more on both
# sides.  So a sphere's u and v may differ from the oracle's by at most this many ulp of the larger of the two.
SPHERE_UV_ULP = 8
CAM_W, CAM_H = 48, 32


def many_objects_scene():
    rng = np.random.RandomState(9)
    mats = [{"kind": k, "ior": 1.5, "color1": tuple(rng.uniform(0.2, 1, 3))} for k in ("diffuse", "plastic", "mirror")] * 30
    mats.append({"kind": "emmit", "color1": (2, 2, 2)})
    objs = [{"kind": "sphere", "center": tuple(rng.uniform(-1, 1, 3)), "radius": float(rng.uniform(0.03, 0.12)),
             "material": 90 if i % 11 == 0 else i % 90} for i in range(150)]
    objs.append({"kind": "plane", "point": (0, -1.2, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0})
    lights = [{"kind": "point", "vec": (0, 3, -2), "color": (60, 60, 60), "radius": 0.5},
              {"kind": "directional", "vec": (0.3, 2.0, -0.5), "color": (0.5, 0.5, 0.5)}]
    return RawScene(objs, mats, lights, camera={"position": (0, 0, -4)}, size=(CAM_W, CAM_H, 3))


BUILT = {"many_objects": many_objects_scene, "spheres_1000": lambda: rh.Scene.synthetic(20000, 1000)}


@pytest.fixture(scope="module", params=SCENES + list(BUILT))
def case(request):
    name = request.param
    sc = BUILT[name]() if name in BUILT else load_scene(name)
    orc = BatchOracle(sc.raw)
    return name, sc, orc, geometry(sc)


def geometry(sc):
    """Kinds, meshes (vertex positions, index triples), spheres, planes and lights of the raw scene."""
    raw = sc.raw.contents
    g = dict(kinds=[], verts=[], tris=[], spheres=[], planes=[], lights=[])
    for i in range(raw.n_objects):
        o = raw.objects[i]
        g["kinds"].append(o.kind)
        if o.kind == capi.RH_OBJ_MESH and o.n_indices >= 3:
            pos = np.ctypeslib.as_array(o.positions, shape=(o.n_verts, 3)).copy()
            idx = np.ctypeslib.as_array(o.indices, shape=(o.n_indices,))[: o.n_indices // 3 * 3].reshape(-1, 3).astype(np.int64)
            g["verts"].append(pos)
            g["tris"].append(pos[idx])
        elif o.kind == capi.RH_OBJ_SPHERE:
            g["spheres"].append((np.array(o.a[:]), o.b[0]))
        elif o.kind == capi.RH_OBJ_PLANE:
            g["planes"].append((np.array(o.a[:]), np.array(o.b[:]), np.array(o.c[:])))
    for i in range(raw.n_lights):
        g["lights"].append((raw.lights[i].kind, np.array(raw.lights[i].vec[:])))
    pts = [v for v in g["verts"]] + [np.array([c - r, c + r]) for c, r in g["spheres"]]
    pts = np.concatenate(pts) if pts else np.array([[-1.0, -1, -1], [1, 1, 1]])
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    pad = 0.1 * (hi - lo) + 1e-3
    g["lo"], g["hi"] = lo - pad, hi + pad
    g["tris"] = np.concatenate(g["tris"]) if g["tris"] else np.zeros((0, 3, 3))
    g["verts"] = np.concatenate(g["verts"]) if g["verts"] else np.zeros((0, 3))
    return g


def unit(rng, n):
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def camera_rays(sc, orc):
    return np.array([np.concatenate(orc.ray_from_pixel(sc.camera, CAM_W, CAM_H, x, y)) for y in range(CAM_H) for x in range(CAM_W)])


def incoherent_rays(g, rng, n=4096):
    return np.concatenate([rng.uniform(g["lo"], g["hi"], (n, 3)), unit(rng, n)], axis=1)


def adversarial_rays(g, rng, k=256):
    lo, hi = g["lo"], g["hi"]
    O = lambda: rng.uniform(lo, hi, (k, 3))  # noqa: E731
    sets = []
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    sets.append((O(), axes[rng.randint(0, 6, k)]))                      # axis-aligned
    d = unit(rng, k)
    d[np.arange(k), rng.randint(0, 3, k)] = 0.0                          # one zero component
    sets.append((O(), d))
    sets.append((O(), unit(rng, k) * 1e-3))                               # unnormalised
    sets.append((O(), unit(rng, k) * 1e3))
    if len(g["tris"]):
        t = g["tris"][rng.randint(0, len(g["tris"]), k)]
        a, b, c = t[:, 0], t[:, 1], t[:, 2]
        o = O()
        sets.append((o, g["verts"][rng.randint(0, len(g["verts"]), k)] - o))  # through a vertex
        sets.append((a - 0.5 * (b - a), b - a))                           # along an edge, through both end points
        e = (b - a) + 0.3 * (c - a)
        sets.append((a - e, e))                                          # in the triangle's plane, through it
    if g["spheres"]:
        s = [g["spheres"][i] for i in rng.randint(0, len(g["spheres"]), k)]
        ctr = np.array([c for c, _ in s])
        rad = np.array([r for _, r in s])[:, None]
        sets.append((ctr + 0.5 * rad * unit(rng, k), unit(rng, k)))         # origins inside spheres
        sets.append((ctr.copy(), unit(rng, k)))                              # from the centre
    for p, n, t in g["planes"]:
        bt = np.cross(t, n)
        uv = rng.uniform(-2, 2, (k, 2))
        on = p + uv[:, :1] * t + uv[:, 1:] * bt
        sets.append((on, unit(rng, k)))                                      # origins on the plane
        dirs = uv[:, :1] * t + uv[:, 1:] * bt
        sets.append((O(), dirs))                                             # parallel to the plane
        sets.append((on + n, np.repeat(t[None], k, axis=0)))                 # parallel, above it
    o = np.concatenate([s[0] for s in sets])
    d = np.concatenate([s[1] for s in sets])
    keep = np.linalg.norm(d, axis=1) > 0
    return np.concatenate([o[keep], d[keep]], axis=1)


def all_rays(name, sc, orc, g):
    rng = np.random.RandomState(zlib.crc32(name.encode()))
    return {"camera": camera_rays(sc, orc), "incoherent": incoherent_rays(g, rng), "adversarial": adversarial_rays(g, rng)}


def query(sc, rays, **kw):
    return rh.closestIntersection(sc, np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:]), **kw)


def rec_bytes(rec):
    return np.ascontiguousarray(rec).view(np.uint8).reshape(len(rec), rec.dtype.itemsize)


def assert_same_hits(got, want, kinds, what):
    """Ids equal; t, p, n and mesh / plane uv bit-identical; sphere uv within SPHERE_UV_ULP."""
    assert np.array_equal(got["object"], want["object"]), (what, np.flatnonzero(got["object"] != want["object"])[:10])
    assert np.array_equal(got["tri"], want["tri"]), what
    gb, wb = rec_bytes(got), rec_bytes(want)
    sphere = np.array([want["object"][i] >= 0 and kinds[want["object"][i]] == capi.RH_OBJ_SPHERE for i in range(len(want))], dtype=bool)
    uv = slice(56, 72)
    rest = np.r_[0:56, 72:80]
    bad = np.flatnonzero((gb[:, rest] != wb[:, rest]).any(axis=1))
    assert len(bad) == 0, (what, bad[:10], got[bad[:3]], want[bad[:3]])
    bad = np.flatnonzero((gb[~sphere][:, uv] != wb[~sphere][:, uv]).any(axis=1))
    assert len(bad) == 0, (what, "mesh / plane uv", bad[:10])
    a, b = got["uv"][sphere], want["uv"][sphere]
    ok = (a == b) | (np.isnan(a) & np.isnan(b)) | (np.abs(a - b) <= SPHERE_UV_ULP * np.spacing(np.maximum(np.abs(a), np.abs(b))))
    assert ok.all(), (what, "sphere uv", a[~ok.all(axis=1)][:5], b[~ok.all(axis=1)][:5])


def shadow_rays_from(hits, lights):
    """accumDiffuse's shadow rays (RayHs.hs:89-97): rayEps p ld from every hit towards every light (Light.hs:12-17)."""
    p = hits["p"][hits["object"] >= 0]
    out = []
    for kind, v in lights:
        if kind == capi.RH_LIGHT_DIRECTIONAL:
            ld = np.repeat(v[None], len(p), axis=0)
        else:
            w = v - p
            d = np.sqrt(w[:, 0] * w[:, 0] + w[:, 1] * w[:, 1] + w[:, 2] * w[:, 2])
            ld = (1 / d)[:, None] * w
        out.append(np.concatenate([p + 0.000001 * ld, ld], axis=1))
    return out


# The default walk culls with conservative float boxes; the reference's double box test can reject a box that a ray
# grazes (a hit within an ulp of the box face), and then the float cull finds a hit the reference does not (DESIGN.md
# §3).  RH_FLAG_EXACT_BOXES walks the reference's own tree with its own box test and must agree on every ray; the default
# walk must agree with it except on at most this share of the rays of a set (all of them adversarial grazers).
MAX_GRAZING = 1 / 500


def grazing_rows(a, b):
    return np.flatnonzero((rec_bytes(a) != rec_bytes(b)).any(axis=1)) if a.dtype.names else np.flatnonzero(a != b)


def test_closest_hits_equal_the_oracle_and_the_exact_walk(case):
    name, sc, orc, g = case
    for kind, rays in all_rays(name, sc, orc, g).items():
        want = orc.closest_batch(rays)
        exact = query(sc, rays, exact_boxes=True).records
        assert_same_hits(exact, want, g["kinds"], (name, kind, "exact walk"))
        got = query(sc, rays).records
        graze = grazing_rows(got, exact)
        assert len(graze) <= max(1, MAX_GRAZING * len(rays)), (name, kind, graze[:10], rays[graze[:3]])
        keep = np.setdiff1d(np.arange(len(rays)), graze)
        assert_same_hits(got[keep], want[keep], g["kinds"], (name, kind))
        if kind == "camera":
            assert (want["object"] >= 0).any(), (name, "the view sees nothing")
            assert len(graze) == 0, (name, "a camera ray grazes")


def test_shadows_equal_the_oracle_for_every_light(case):
    name, sc, orc, g = case
    assert g["lights"], name
    rays = all_rays(name, sc, orc, g)
    hits = orc.closest_batch(np.concatenate([rays["camera"], rays["incoherent"]]))
    from_hits = shadow_rays_from(hits, g["lights"])
    for li in range(len(g["lights"])):
        for kind, r in (("random", np.concatenate([rays["incoherent"], rays["adversarial"]])), ("from hits", from_hits[li])):
            o, d = np.ascontiguousarray(r[:, :3]), np.ascontiguousarray(r[:, 3:])
            want = orc.shadow_batch(li, r)
            exact = rh.shadowIntersection(sc, li, o, d, exact_boxes=True)
            assert exact.dtype == np.bool_ and np.array_equal(exact, want), (name, li, kind, np.flatnonzero(exact != want)[:10])
            got = rh.shadowIntersection(sc, li, o, d)
            graze = grazing_rows(got, exact)
            assert len(graze) <= max(1, MAX_GRAZING * len(r)), (name, li, kind, graze[:10])
            if kind == "from hits":
                assert len(graze) == 0, (name, li, "a shadow ray from a hit grazes")


def test_query_agrees_with_the_renders_primary_hit_ids(case):
    name, sc, orc, g = case
    img = rh.render(rh.Rendering(sc, sc.camera, CAM_W, CAM_H, 0), want_hit_ids=True)
    ids = img.hit_ids.reshape(CAM_H * CAM_W, 2)
    h = query(sc, camera_rays(sc, orc))
    assert np.array_equal(ids[:, 0], h.object) and np.array_equal(ids[:, 1], h.tri), name


def test_device_path_returns_the_host_bytes_at_every_size(case):
    import torch

    name, sc, orc, g = case
    rays = all_rays(name, sc, orc, g)["incoherent"]
    for n in (0, 1, 33, len(rays)):
        r = rays[:n]
        host = query(sc, r)
        o, d = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (r[:, :3], r[:, 3:]))
        dev = rh.closestIntersection(sc, o, d)
        assert dev.records.is_cuda and dev.t.is_cuda and tuple(dev.p.shape) == (n, 3) and tuple(dev.uv.shape) == (n, 2)
        assert np.array_equal(dev.records.cpu().numpy().reshape(-1), rec_bytes(host.records).reshape(-1)), (name, n)
        assert np.array_equal(dev.object.cpu().numpy(), host.object) and np.array_equal(dev.t.cpu().numpy(), host.t)
        for li in range(len(g["lights"])):
            hs = rh.shadowIntersection(sc, li, r[:, :3].copy(), r[:, 3:].copy())
            ds = rh.shadowIntersection(sc, li, o, d)
            assert ds.is_cuda and ds.dtype == torch.bool and np.array_equal(ds.cpu().numpy(), hs), (name, li, n)


def test_more_rays_than_one_launch_and_one_host_chunk():
    """2^24 + 5 incoherent rays on dragon_full: several host chunks and two device launches; the device and host paths
    give the same bytes, and a seeded sample (including the rays around the chunk and launch edges) matches the oracle."""
    import torch

    sc = load_scene("dragon_full")
    orc = BatchOracle(sc.raw)
    g = geometry(sc)
    n = (1 << 24) + 5
    rng = np.random.RandomState(2024)
    o = rng.uniform(g["lo"], g["hi"], (n, 3))
    d = rng.normal(size=(n, 3))
    host = rh.closestIntersection(sc, o, d)
    dev = rh.closestIntersection(sc, torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda())
    assert np.array_equal(dev.records.cpu().numpy().reshape(-1), rec_bytes(host.records).reshape(-1))
    edges = np.array([k * (1 << 21) + j for k in range(1, 9) for j in (-2, -1, 0, 1)] + [n - 3, n - 2, n - 1])
    idx = np.unique(np.concatenate([rng.randint(0, n, 6000), edges]))
    want = orc.closest_batch(np.concatenate([o[idx], d[idx]], axis=1))
    assert_same_hits(host.records[idx], want, g["kinds"], "dragon_full, 2^24 + 5 rays")
    assert (want["object"] >= 0).sum() > 100
    li = 0
    hs = rh.shadowIntersection(sc, li, o, d)
    ds = rh.shadowIntersection(sc, li, torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda())
    assert np.array_equal(ds.cpu().numpy(), hs)
    assert np.array_equal(hs[idx], orc.shadow_batch(li, np.concatenate([o[idx], d[idx]], axis=1)))


def test_argument_errors():
    import torch

    sc = load_scene("cornellBox")
    L = capi.lib()
    rays = np.zeros((4, 6))
    rays[:, 5] = 1
    hits = np.empty(4, dtype=rh.HIT_DTYPE)
    occ = np.empty(4, dtype=np.uint8)
    n_lights = sc.flat.contents.n_lights
    dev = sc.device
    assert L.rh_shadow_intersection(dev, n_lights, rays.ctypes.data, 4, occ.ctypes.data, 0) == capi.RH_ERR_ARG
    assert L.rh_shadow_intersection(dev, n_lights - 1, rays.ctypes.data, 4, occ.ctypes.data, 0) == capi.RH_OK
    for bad in (capi.RH_FLAG_HIT_IDS, capi.RH_FLAG_PROFILE, capi.RH_FLAG_COUNT, 1 << 20):
        assert L.rh_closest_intersection(dev, rays.ctypes.data, 4, hits.ctypes.data, bad) == capi.RH_ERR_ARG
        assert L.rh_shadow_intersection(dev, 0, rays.ctypes.data, 4, occ.ctypes.data, bad) == capi.RH_ERR_ARG
    assert L.rh_closest_intersection(dev, None, 4, hits.ctypes.data, 0) == capi.RH_ERR_ARG
    assert L.rh_closest_intersection(dev, rays.ctypes.data, 4, None, 0) == capi.RH_ERR_ARG
    assert L.rh_shadow_intersection(dev, 0, None, 4, occ.ctypes.data, 0) == capi.RH_ERR_ARG
    assert L.rh_shadow_intersection(dev, 0, rays.ctypes.data, 4, None, 0) == capi.RH_ERR_ARG
    assert L.rh_closest_intersection(dev, None, 0, None, 0) == capi.RH_OK
    assert L.rh_closest_intersection(None, rays.ctypes.data, 4, hits.ctypes.data, 0) == capi.RH_ERR_ARG
    # device flag with host memory, and a misaligned device buffer
    assert L.rh_closest_intersection(dev, rays.ctypes.data, 4, hits.ctypes.data, capi.RH_FLAG_DEVICE_OUT) == capi.RH_ERR_ARG
    t = torch.zeros(4 * 6 + 1, dtype=torch.float64, device="cuda")
    out = torch.empty(4 * 80 + 16, dtype=torch.uint8, device="cuda")
    assert L.rh_closest_intersection(dev, t.data_ptr() + 8, 4, out.data_ptr(), capi.RH_FLAG_DEVICE_OUT) == capi.RH_ERR_ARG
    assert L.rh_closest_intersection(dev, t.data_ptr(), 4, out.data_ptr() + 8, capi.RH_FLAG_DEVICE_OUT) == capi.RH_ERR_ARG
    assert L.rh_closest_intersection(dev, t.data_ptr(), 4, out.data_ptr(), capi.RH_FLAG_DEVICE_OUT) == capi.RH_OK
    # the Python layer: shapes, dtypes, a mix of host and device inputs
    o = np.zeros((3, 3))
    for bad_o, bad_d in ((o.astype(np.float32), o), (o, o[:2]), (o[:, :2], o[:, :2]), (o, torch.zeros(3, 3, dtype=torch.float64).cuda()),
                         (torch.zeros(3, 3).cuda(), torch.zeros(3, 3).cuda()), (torch.zeros(3, 3, dtype=torch.float64), o)):
        with pytest.raises(ValueError):
            rh.closestIntersection(sc, bad_o, bad_d)
        with pytest.raises(ValueError):
            rh.shadowIntersection(sc, 0, bad_o, bad_d)
    with pytest.raises(capi.RayHsError) as e:
        rh.shadowIntersection(sc, n_lights, o, o)
    assert e.value.code == capi.RH_ERR_ARG
