"""CPU tests of the batched ray queries: the rh_hit layout of the header against the ctypes / numpy mirrors, loud
failure without a device, and the oracle's batch queries (oracle/batch.cpp: orc_closest_batch / orc_shadow_batch)
against the oracle's one-ray entry point and against hand-derived answers."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import HIT_DTYPE as ORC_HIT_DTYPE, OracleScene
from rayhs_b200 import capi
from tests.util import RawScene, load_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["t", "p", "n", "uv", "object", "tri"]


def test_rh_hit_layout_matches_the_header():
    """sizeof / offsetof from a C program compiled against the header equal the ctypes and numpy mirrors (80 bytes)."""
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){' + \
        'printf("size %zu\\n", sizeof(rh_hit));' + "".join(f'printf("{f} %zu\\n", offsetof(rh_hit, {f}));' for f in FIELDS) + \
        "return 0;}"
    exe = os.path.join(ROOT, "build", "abi_rh_hit")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    out = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert out["size"] == C.sizeof(capi.rh_hit) == rh.HIT_DTYPE.itemsize == ORC_HIT_DTYPE.itemsize == 80
    for f in FIELDS:
        assert out[f] == getattr(capi.rh_hit, f).offset == rh.HIT_DTYPE.fields[f][1] == ORC_HIT_DTYPE.fields[f][1], f


def test_queries_without_a_device_fail_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    rays = np.zeros((4, 6))
    hits = np.empty(4, dtype=rh.HIT_DTYPE)
    occ = np.empty(4, dtype=np.uint8)
    assert L.rh_closest_intersection(None, rays.ctypes.data, 4, hits.ctypes.data, 0) == capi.RH_ERR_STATE
    assert L.rh_shadow_intersection(None, 0, rays.ctypes.data, 4, occ.ctypes.data, 0) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()


def test_closest_batch_equals_the_one_ray_entry_point():
    sc = load_scene("cornellBox")
    orc = OracleScene(sc.raw)
    rng = np.random.RandomState(3)
    cam = [np.concatenate(orc.ray_from_pixel(sc.camera, 64, 48, x, y)) for y in range(0, 48, 2) for x in range(0, 64, 2)]
    o = rng.uniform(-3, 3, (2000, 3))
    d = rng.normal(size=(2000, 3))
    d[::7, rng.randint(0, 3)] = 0.0  # zero components
    rays = np.concatenate([np.array(cam), np.concatenate([o, d], axis=1)])
    got = OracleScene(sc.raw).closest_batch(rays, threads=4)
    hits = 0
    for i, r in enumerate(rays):
        one = orc.closest(r[:3], r[3:])
        if one is None:
            assert got["object"][i] == -1 and got["tri"][i] == -1 and got["t"][i] == math.inf, i
            assert not got["p"][i].any() and not got["n"][i].any() and not got["uv"][i].any(), i
            continue
        hits += 1
        assert (got["object"][i], got["tri"][i]) == (one["object"], one["tri"]), i
        for k in ("p", "n", "uv"):
            assert got[k][i].tobytes() == one[k].tobytes(), (i, k)
        assert got["t"][i].tobytes() == np.float64(one["t"]).tobytes(), i
    assert hits > 1000


SPHERE = {"kind": "sphere", "center": (0, 0, 0), "radius": 1.0}


def test_closest_batch_hand_derived_answers():
    rs = RawScene([SPHERE, {"kind": "plane", "point": (0, -2, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0)}],
                  [{"kind": "diffuse"}], [])
    orc = OracleScene(rs.raw)
    rays = np.array([[0, 0, -5, 0, 0, 1],     # from outside at the centre: t = distance - 1
                     [0, 0, 0, 0, 0, 1],      # from the centre: the far root
                     [0, 0, 0.5, 0, 0, 2],    # from inside, direction of length 2: far root at z = 1, t = 0.25
                     [5, -1, 0, 1, 0, 0],     # parallel to the plane, beside the sphere: a miss
                     [0, -3, 0, 1, 0, 0]])    # parallel to the plane, below it: a miss
    h = orc.closest_batch(rays)
    assert h["t"][0] == 4.0 and h["object"][0] == 0 and h["tri"][0] == -1
    assert tuple(h["p"][0]) == (0, 0, -1) and tuple(h["n"][0]) == (0, 0, -1)
    assert h["t"][1] == 1.0 and tuple(h["p"][1]) == (0, 0, 1) and tuple(h["n"][1]) == (0, 0, 1)
    assert h["t"][2] == 0.25 and tuple(h["p"][2]) == (0, 0, 1)
    for i in (3, 4):
        assert h["t"][i] == math.inf and h["object"][i] == -1 and h["tri"][i] == -1, i


def test_shadow_batch_hand_derived_answers():
    ray = np.array([[0, 0, 0, 0, 0, 1]])
    # the only blocker is an emitter: isOccluder (RayHs.hs:81-82) drops it
    emitter = RawScene([{"kind": "sphere", "center": (0, 0, 3), "radius": 0.5}], [{"kind": "emmit", "color1": (1, 1, 1)}],
                       [{"kind": "point", "vec": (0, 0, 6)}])
    assert not OracleScene(emitter.raw).shadow_batch(0, ray)[0]
    # the same sphere as a diffuse object does block
    diffuse = RawScene([{"kind": "sphere", "center": (0, 0, 3), "radius": 0.5}], [{"kind": "diffuse"}],
                       [{"kind": "point", "vec": (0, 0, 6)}])
    assert OracleScene(diffuse.raw).shadow_batch(0, ray)[0]
    # a blocker behind a point light is not in front of it (inFrontOfLight, RayHs.hs:84-87) ...
    behind = [{"kind": "sphere", "center": (0, 0, 5), "radius": 0.5}]
    point = RawScene(behind, [{"kind": "diffuse"}], [{"kind": "point", "vec": (0, 0, 2)}])
    assert not OracleScene(point.raw).shadow_batch(0, ray)[0]
    # ... while for a directional light every hit counts
    directional = RawScene(behind, [{"kind": "diffuse"}], [{"kind": "directional", "vec": (0, 0, 1)}])
    assert OracleScene(directional.raw).shadow_batch(0, ray)[0]
    # two lights in one scene: the index selects the light
    both = RawScene(behind, [{"kind": "diffuse"}], [{"kind": "point", "vec": (0, 0, 2)}, {"kind": "directional", "vec": (0, 0, 1)}])
    assert OracleScene(both.raw).shadow_batch(0, np.repeat(ray, 3, axis=0)).tolist() == [False] * 3
    assert OracleScene(both.raw).shadow_batch(1, np.repeat(ray, 3, axis=0)).tolist() == [True] * 3


def test_python_layer_rejects_bad_shapes_and_dtypes_before_any_call():
    """The checks run before the library is reached, so they hold without a device."""
    o = np.zeros((5, 3))
    for bad_o, bad_d in ((o.astype(np.float32), o), (o, o[:4]), (o[:, :2], o[:, :2]), (o.reshape(-1), o.reshape(-1)),
                         (o, o.tolist())):
        with pytest.raises(ValueError):
            rh.closestIntersection(None, bad_o, bad_d)
        with pytest.raises(ValueError):
            rh.shadowIntersection(None, 0, bad_o, bad_d)
