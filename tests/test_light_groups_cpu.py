"""CPU tests of the light groups (rh_render_light_groups / renderLightGroups): the entry point is exported and bound,
rh_light_groups' layout in the header equals the ctypes mirror, the chunk planner's per-sample byte count, the Python
layer's argument checks and output shapes with the library stubbed, and LightGroups.relight against numpy."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host
from tests.test_render_plan_cpu import B200_MEM, BENCH_ROW, BENCH_ROWS, CASES, SMALL_MEM, plan
from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["group_of_light", "n_groups", "reserved_", "out"]


def test_symbol_is_exported_and_bound():
    L = capi.lib()
    args = capi.SIGNATURES["rh_render_light_groups"][1]
    assert L.rh_render_light_groups.argtypes == args
    assert len(args) == 7 and args[3]._type_ is capi.rh_light_groups and args[6]._type_ is capi.rh_stats
    assert rh.renderLightGroups is host.renderLightGroups and rh.LightGroups is host.LightGroups


def test_rh_light_groups_layout_matches_the_header():
    """sizeof / offsetof from a C program compiled against the header equal the ctypes mirror (24 bytes)."""
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){' + \
        'printf("size %zu\\n", sizeof(rh_light_groups));' + \
        "".join(f'printf("{f} %zu\\n", offsetof(rh_light_groups, {f}));' for f in FIELDS) + "return 0;}"
    exe = os.path.join(ROOT, "build", "abi_rh_light_groups")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    out = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([exe], text=True).splitlines())}
    assert out["size"] == C.sizeof(capi.rh_light_groups) == 24
    for f in FIELDS:
        assert out[f] == getattr(capi.rh_light_groups, f).offset, f


def test_without_a_device_the_call_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    o = capi.rh_render_opts()
    o.width, o.height, o.spp = 4, 4, 1
    out = np.empty((2, 4, 4, 3))
    lg = capi.rh_light_groups()
    lg.n_groups, lg.out = 1, out.ctypes.data
    assert L.rh_render_light_groups(None, None, C.byref(o), C.byref(lg), None, None, None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()


# ---------------------------------------------------------------- chunk plan
_plan_lib = None


def lg_plan(rows_local, row_samples, chunk_samples, mem, host_offsets, bytes_per_sample):
    global _plan_lib
    if _plan_lib is None:
        _plan_lib = temp_library("light_groups_plan", [os.path.join(ROOT, "tests", "light_groups_plan_driver.cpp"),
                                                       os.path.join(ROOT, "rayhs_b200", "csrc", "render_plan.h")],
                                 ["-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared"])
        _plan_lib.lg_plan.restype = C.c_int
        _plan_lib.lg_plan.argtypes = [C.c_int, C.c_ulonglong, C.c_int, C.c_ulonglong, C.c_int, C.c_ulonglong, C.c_int,
                                      C.POINTER(C.c_int)]
        _plan_lib.lg_default_bytes_per_sample.restype = C.c_ulonglong
    rows = np.zeros(8192, np.int32)
    n = _plan_lib.lg_plan(rows_local, row_samples, chunk_samples, mem, int(host_offsets), bytes_per_sample, len(rows),
                          rows.ctypes.data_as(C.POINTER(C.c_int)))
    assert 0 < n <= len(rows)
    return rows[:n].tolist()


def default_bytes():
    lg_plan(1, 1, 0, B200_MEM, False, 0)
    return int(_plan_lib.lg_default_bytes_per_sample())


@pytest.mark.parametrize("name", sorted(n for n, c in CASES.items() if c[5] is None))
def test_the_default_byte_count_keeps_todays_plans(name):
    rows_local, row_samples, chunk_samples, mem, host_offsets, _, _ = CASES[name]
    want = plan(*CASES[name])[0]
    assert lg_plan(rows_local, row_samples, chunk_samples, mem, host_offsets, 0) == want
    assert lg_plan(rows_local, row_samples, chunk_samples, mem, host_offsets, default_bytes()) == want


@pytest.mark.parametrize("n_groups", [1, 3, 16])
@pytest.mark.parametrize("mem", [B200_MEM, SMALL_MEM])
@pytest.mark.parametrize("host_out", [False, True])
def test_group_scratch_stays_within_the_budget(n_groups, mem, host_out):
    """Every chunk's scratch (the render's bytes per sample plus 24 per group and sample, plus 24 per group and pixel
    of host output) fits 45 % of the device memory, halved per lane when the frame has several chunks."""
    group = 24 * (n_groups + 1)
    per_sample = default_bytes() + group * (2 if host_out else 1)
    for spp in (1, 16):
        rows = lg_plan(BENCH_ROWS, 3840 * spp, 0, mem, False, per_sample)
        budget = 0.45 * mem / (2 if len(rows) > 1 else 1)
        assert sum(rows) == BENCH_ROWS
        for r in rows:
            assert r * 3840 * spp * (default_bytes() + group) + (r * 3840 * group if host_out else 0) <= budget
    # the bench frame (3840 x 2160 x 16 spp) is one chunk for the render; with more per-sample bytes it splits sooner
    assert len(lg_plan(BENCH_ROWS, BENCH_ROW, 0, B200_MEM, False, default_bytes())) == 1
    assert len(lg_plan(BENCH_ROWS, BENCH_ROW, 0, B200_MEM, False, default_bytes() + 24 * 17 * 2)) > 1


# ---------------------------------------------------------------- Python layer
class _FakeLib:
    """Stands in for librayhs_b200.so: records the rh_render_light_groups call and fills the outputs with markers."""

    def __init__(self):
        self.calls = []

    def rh_default_band_height(self, h, g):
        return h if g <= 1 else 4

    def rh_shard_rows(self, h, g, bh):
        n_bands = (h + bh - 1) // bh
        return (n_bands + g - 1) // g * bh

    def rh_render_light_groups(self, scene, cam, opts, lg, rgb, ids, stats):
        o, g = opts._obj, lg._obj
        n_lights = _Job.scene.raw.contents.n_lights
        self.calls.append(dict(scene=scene, size=(o.width, o.height, o.spp), mode=o.offset_mode, offsets=o.offsets,
                               shard=(o.shard_index, o.shard_count, o.band_height), chunk=o.chunk_samples, flags=o.flags,
                               map=list((C.c_uint8 * max(n_lights, 1)).from_address(g.group_of_light))[:n_lights],
                               n_groups=g.n_groups, reserved=g.reserved_, out=g.out, rgb=rgb, ids=ids))
        stats._obj.rays_primary = 11
        return 0


class _Raw:
    n_lights = 3


class _Job:
    class scene:
        device = "scene-handle"

        class raw:
            contents = _Raw

    camera = capi.rh_camera()
    width, height, maxDepth = 10, 6, 3


@pytest.fixture
def fake(monkeypatch):
    L = _FakeLib()
    monkeypatch.setattr(host, "lib", lambda: L)
    _Raw.n_lights = 3
    return L


def test_shapes_and_the_default_groups(fake):
    lgs = rh.renderLightGroups(_Job, spp=2, seed=5, want_hit_ids=True)
    assert lgs.groups.shape == (3, 6, 10, 3) and lgs.rest.shape == (6, 10, 3) and lgs.groups.dtype == np.float64
    assert lgs.image.shape == (6, 10, 3) and lgs.image.dtype == np.uint8
    assert lgs.hit_ids.shape == (6, 10, 2, 2) and lgs.hit_ids.dtype == np.int32
    assert lgs.stats["rays_primary"] == 11
    (c,) = fake.calls
    assert c["map"] == [0, 1, 2] and c["n_groups"] == 3 and c["reserved"] == 0
    assert c["out"] == lgs.groups.ctypes.data and lgs.rest.ctypes.data == c["out"] + 3 * 6 * 10 * 3 * 8
    assert c["rgb"] == lgs.image.ctypes.data and c["ids"] == lgs.hit_ids.ctypes.data
    assert c["mode"] == capi.RH_OFFSETS_SPLITMIX64 and c["flags"] == capi.RH_FLAG_HIT_IDS and c["size"] == (10, 6, 2)


def test_groups_flags_and_shards(fake):
    lgs = rh.renderLightGroups(_Job, groups=[1, 1, 0], rgb=False, shadow="split", exact_boxes=True, light_maps=False,
                               chunk_samples=40, shard_index=1, shard_count=2, band_height=2, profile=True)
    assert lgs.groups.shape == (2, 4, 10, 3) and lgs.image is None and lgs.hit_ids is None
    c = fake.calls[-1]
    assert c["map"] == [1, 1, 0] and c["n_groups"] == 2 and c["rgb"] is None and c["ids"] is None
    assert c["shard"] == (1, 2, 2) and c["chunk"] == 40
    assert c["flags"] == (capi.RH_FLAG_SHADOW_SPLIT | capi.RH_FLAG_EXACT_BOXES | capi.RH_FLAG_NO_LIGHT_MAPS | capi.RH_FLAG_PROFILE)
    rh.renderLightGroups(_Job, groups=[0, 0, 5])  # empty groups 1 .. 4 are images of zeros
    assert fake.calls[-1]["n_groups"] == 6
    off = np.zeros((60, 2, 2))
    rh.renderLightGroups(_Job, spp=2, offsets=off)
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_F64 and fake.calls[-1]["offsets"] == off.ctypes.data
    rh.renderLightGroups(_Job, spp=2, offsets=off.astype(np.float32))
    assert fake.calls[-1]["mode"] == capi.RH_OFFSETS_F32
    _Raw.n_lights = 0
    lgs = rh.renderLightGroups(_Job)
    assert lgs.groups.shape == (1, 6, 10, 3) and fake.calls[-1]["n_groups"] == 1 and fake.calls[-1]["map"] == []


def test_argument_checks(fake):
    for kw in (dict(groups=[0, 1]), dict(groups=[0, 1, 2, 3]), dict(groups=[0, 16, 1]), dict(groups=[0, -1, 1]),
               dict(spp=2, offsets=np.zeros((60, 1, 2))), dict(spp=2, offsets=np.zeros((60, 2, 2)), seed=3)):
        with pytest.raises(ValueError):
            rh.renderLightGroups(_Job, **kw)
    assert not fake.calls  # rejected before the library is reached


def test_relight_against_numpy():
    rng = np.random.RandomState(3)
    groups, rest = rng.normal(size=(4, 5, 7, 3)), rng.normal(size=(5, 7, 3))
    lgs = rh.LightGroups(groups, rest)
    k = rng.uniform(0, 2, (4, 3))
    want = rest.copy()
    for y in range(5):
        for x in range(7):
            for c in range(3):
                s = k[0, c] * groups[0, y, x, c]
                for g in range(1, 4):
                    s = s + k[g, c] * groups[g, y, x, c]
                want[y, x, c] = s + rest[y, x, c]
    assert np.array_equal(lgs.relight(k), want)
    assert np.array_equal(lgs.relight(np.ones((4, 3))), groups[0] + groups[1] + groups[2] + groups[3] + rest)
    for bad in (np.ones((3, 3)), np.ones((4,)), np.ones((4, 3, 1))):
        with pytest.raises(ValueError):
            lgs.relight(bad)
