"""CPU tests of the radiance queries (rh_trace_rays / traceRay): the rh_trace_opts layout of the header against the
ctypes mirror, loud failure without a device, argument checks of the Python layer, and the batch oracle of the GPU
tests (oracle/batch.cpp: orc_trace_batch) against hand-derived answers and against the oracle's own render."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene, camera_rays
from rayhs_b200 import capi
from tests.util import SCENES, RawScene, load_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PI_INV = 1 / np.pi  # oracle.cpp piInv (Math.hs:11-12)


def test_rh_trace_opts_layout_matches_the_header():
    fields = [f for f, _ in capi.rh_trace_opts._fields_]
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){' + \
        'printf("size %zu\\n", sizeof(rh_trace_opts));' + \
        "".join(f'printf("{f} %zu\\n", offsetof(rh_trace_opts, {f}));' for f in fields) + "return 0;}"
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "abi_rh_trace_opts")
        with open(exe + ".c", "w") as f:
            f.write(src)
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
        out = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert out["size"] == C.sizeof(capi.rh_trace_opts) == 16
    for f in fields:
        assert out[f] == getattr(capi.rh_trace_opts, f).offset, f


def test_trace_rays_without_a_device_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    rays = np.zeros((4, 6))
    colors = np.empty((4, 3))
    o = capi.rh_trace_opts()
    assert L.rh_trace_rays(None, rays.ctypes.data, 4, C.byref(o), colors.ctypes.data, None, None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()


def test_python_layer_rejects_bad_shapes_and_dtypes_before_any_call():
    """The checks run before the library is reached, so they hold without a device."""
    o = np.zeros((5, 3))
    for bad_o, bad_d in ((o.astype(np.float32), o), (o, o[:4]), (o[:, :2], o[:, :2]), (o.reshape(-1), o.reshape(-1)),
                         (o, o.tolist()), (o, o.astype(np.int64))):
        with pytest.raises(ValueError):
            rh.traceRay(None, bad_o, bad_d, 3)
    for bad_chunk in (-1, 1 << 32):
        with pytest.raises(ValueError):
            rh.traceRay(None, o, o, 3, chunk_rays=bad_chunk)


PLANE = {"kind": "plane", "point": (0, 0, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0}
CD = np.array([0.5, 0.25, 0.75])
# a point light 2 above the plane's origin: distance 2, radius 2, so the falloff is 1 / (1 + 2/2)^2 = 1/4 (Light.hs:12-17)
LIGHT = {"kind": "point", "vec": (0, 2, 0), "color": (4, 2, 8), "radius": 2.0}
LC = 0.25 * np.array(LIGHT["color"])
# onto the plane's origin from (1, 1, 0): t = 1, p = 0, n = (0, 1, 0); the light is straight above p, l = (0, 1, 0)
RAY = np.array([[1.0, 1, 0, -1, -1, 0]])


def trace(raw_scene, rays, max_depth):
    return OracleScene(raw_scene.raw).trace_batch(rays, max_depth)


def test_trace_batch_diffuse_plane_under_a_point_light():
    sc = RawScene([PLANE], [{"kind": "diffuse", "color1": tuple(CD)}], [LIGHT])
    col, ids, counts = trace(sc, RAY, 3)
    # irradiance of Diffuse (RayHs.hs:111-113): 0.2 cd + accumDiffuse, one unshadowed light: max(l.n, 0) / pi * cd * lc
    want = 0.2 * CD + (0 + max(1.0, 0) * PI_INV * (CD * LC))
    assert col[0].tolist() == want.tolist()
    assert ids[0].tolist() == [0, -1]
    assert counts == {"rays_primary": 1, "rays_reflect": 0, "rays_probe": 0, "rays_exit": 0, "rays_shadow": 1}


def test_trace_batch_occluded_light_drops_its_term():
    # a sphere between p and the light (beside the primary ray, which passes 0.71 from its centre) blocks the shadow ray
    blocker = {"kind": "sphere", "center": (0, 1, 0), "radius": 0.25, "material": 0}
    sc = RawScene([PLANE, blocker], [{"kind": "diffuse", "color1": tuple(CD)}], [LIGHT])
    col, ids, counts = trace(sc, RAY, 3)
    assert col[0].tolist() == (0.2 * CD).tolist()
    assert ids[0].tolist() == [0, -1] and counts["rays_shadow"] == 1


def test_trace_batch_emitter_mirror_and_miss():
    sc = RawScene([{"kind": "sphere", "center": (0, 0, 3), "radius": 1.0, "material": 0},
                   {"kind": "sphere", "center": (0, 0, -3), "radius": 1.0, "material": 1},
                   PLANE | {"material": 1}],
                  [{"kind": "emmit", "color1": (2.0, 0.5, 3.0)}, {"kind": "mirror", "ior": 1.5}], [LIGHT])
    rays = np.array([[0, 0.5, 0, 0, 0, 1],     # onto the emitter: its colour (RayHs.hs:121)
                     [0, 0, 0, 0, 0, -1],      # head-on onto the mirror sphere (in the plane: parallel to it)
                     [0, 0.5, 0, 0, 1, 0]])    # up, away from everything: a miss is black (RayHs.hs:149-154)
    col, ids, counts = trace(sc, rays, 0)
    assert col[0].tolist() == [2.0, 0.5, 3.0] and ids[0].tolist() == [0, -1]
    # a Mirror at max_depth 0: fresnel x specular, and specular is black at the depth limit (RayHs.hs:99-104, 145-146)
    assert col[1].tolist() == [0, 0, 0] and ids[1].tolist() == [1, -1]
    assert col[2].tolist() == [0, 0, 0] and ids[2].tolist() == [-1, -1]
    assert counts == {"rays_primary": 3, "rays_reflect": 0, "rays_probe": 0, "rays_exit": 0, "rays_shadow": 0}
    # one level deeper the mirror reflects the ray straight back onto the emitter: fresnel at normal incidence is r0
    # (Material.hs:22-29) and dot(reflected, n) = 1
    col1, _, counts1 = trace(sc, rays[1:2], 1)
    q = (1.0 - 1.5) / (1.0 + 1.5)
    f = q * q + (1 - q * q) * 0.0
    assert col1[0].tolist() == [f * 2.0, f * 0.5, f * 3.0]
    assert counts1 == {"rays_primary": 1, "rays_reflect": 1, "rays_probe": 0, "rays_exit": 0, "rays_shadow": 0}


W, H = 48, 32


@pytest.mark.parametrize("name", SCENES)
def test_trace_batch_equals_the_oracle_render_at_one_sample(name):
    """Pixel-centre camera rays through orc_trace_batch give the oracle render's rgb_f64, hit ids and ray counts
    bit for bit: the same traceRay, called per pixel by rayTrace (RayHs.hs:156-166)."""
    sc = load_scene(name)
    ref = OracleScene(sc.raw).render(sc.camera, W, H, sc.max_depth)
    orc = OracleScene(sc.raw)
    col, ids, counts = orc.trace_batch(camera_rays(sc.camera, W, H), sc.max_depth)
    assert col.tobytes() == ref["rgb_f64"].reshape(-1, 3).tobytes(), name
    assert np.array_equal(ids, ref["hit_ids"].reshape(-1, 2)), name
    assert [counts[k] for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")] == \
        [ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow")], name
