"""CPU tests of scene updates (rh_scene_update / rh_multi_scene_update / Scene.update): the bindings and the struct
layout, loud failure without a device, Scene.update on the description alone (raw and flat, checked with the oracle),
Python-side argument errors, and the update planner (rayhs_b200/csrc/scene_update.h, compiled alone through
tests/scene_update_driver.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rayhs_b200 import capi
from tests.util import RawScene, load_scene, temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "scene_update_driver.cpp"), os.path.join(ROOT, "rayhs_b200", "csrc", "scene_update.h"),
           os.path.join(ROOT, "include", "rayhs_b200.h")]
FLAGS = ["-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared"]
NONE, COLOURS, EMITTERS, TABLES = 0, 1, 2, 3
EMPTY = 0xFFFFFFFF


def test_update_info_layout_and_prototypes():
    assert C.sizeof(capi.rh_update_info) == 24
    offsets = {n: getattr(capi.rh_update_info, n).offset for n, _ in capi.rh_update_info._fields_}
    assert offsets == {"colours_only": 0, "occluders_rebuilt": 4, "maps_rasterised": 8, "maps_kept": 12, "lit_queries": 16}
    src = ('#include <stddef.h>\n#include <stdio.h>\n#include "rayhs_b200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu\\n",'
           'sizeof(rh_update_info), offsetof(rh_update_info, colours_only), offsetof(rh_update_info, occluders_rebuilt),'
           'offsetof(rh_update_info, maps_rasterised), offsetof(rh_update_info, maps_kept), offsetof(rh_update_info, lit_queries));'
           'return 0;}')
    exe = os.path.join(ROOT, "build", "update_info_layout")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    assert [int(x) for x in subprocess.check_output([exe], text=True).split()] == [24, 0, 4, 8, 12, 16]
    L = capi.lib()
    for name in ("rh_scene_update", "rh_multi_scene_update"):
        assert getattr(L, name).argtypes == capi.SIGNATURES[name][1]
        assert capi.SIGNATURES[name][1][1] is C.POINTER(capi.rh_material)
        assert capi.SIGNATURES[name][1][3] is C.POINTER(capi.rh_light)
        assert capi.SIGNATURES[name][1][5] is C.POINTER(capi.rh_update_info)


def test_without_a_device_the_calls_fail_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    assert L.rh_init(-1) == capi.RH_ERR_CUDA
    assert b"no CPU fallback" in L.rh_last_error()
    assert L.rh_scene_update(None, None, 0, None, 0, None) == capi.RH_ERR_ARG
    assert b"rh_scene_update: null scene" in L.rh_last_error()
    assert L.rh_multi_scene_update(None, None, 0, None, 0, None) == capi.RH_ERR_ARG
    sc = load_scene("cornellBox")
    with pytest.raises(capi.RayHsError):
        sc.device


def _edited_tables(sc):
    mats, lights = sc.materials, sc.lights
    mats[0].color1[:] = (0.25, 0.5, 0.75)
    if mats[0].kind == capi.RH_MAT_DIFFUSE:
        mats[0].kind = capi.RH_MAT_MIRROR
    lights[0].vec[0] += 0.5
    new_light = capi.rh_light.from_buffer_copy(lights[0])
    new_light.kind = capi.RH_LIGHT_DIRECTIONAL
    new_light.vec[:] = (0.3, -1.0, 0.2)
    new_light.color[:] = (0.2, 0.2, 0.2)
    return mats, list(lights) + [new_light]


def test_update_before_the_device_edits_raw_and_flat():
    from oracle.orc import OracleScene

    sc = load_scene("cornellBox")
    n_objects = sc.raw.contents.n_objects
    mats, lights = _edited_tables(sc)
    info = sc.update(materials=mats, lights=lights)
    assert info == {"colours_only": 0, "occluders_rebuilt": 0, "maps_rasterised": 0, "maps_kept": 0, "lit_queries": 0}
    assert not sc._dev
    for view in (sc.raw.contents, sc.flat.contents):
        assert view.n_lights == len(lights) and view.n_materials == len(mats)
        assert [bytes(view.lights[i]) for i in range(len(lights))] == [bytes(x) for x in lights]
        assert [bytes(view.materials[i]) for i in range(len(mats))] == [bytes(x) for x in mats]
    assert sc.raw.contents.n_objects == n_objects
    assert [bytes(x) for x in sc.materials] == [bytes(x) for x in mats]
    assert [bytes(x) for x in sc.lights] == [bytes(x) for x in lights]

    # the oracle fed the updated Scene.raw renders what it renders for a raw scene edited here
    base = load_scene("cornellBox")
    edited = capi.rh_raw_scene.from_buffer_copy(base.raw.contents)
    m_arr = (capi.rh_material * len(mats))(*mats)
    l_arr = (capi.rh_light * len(lights))(*lights)
    edited.materials = C.cast(m_arr, C.POINTER(capi.rh_material))
    edited.lights = C.cast(l_arr, C.POINTER(capi.rh_light))
    edited.n_lights = len(lights)
    w, h = 40, 30
    a = OracleScene(sc.raw).render(sc.camera, w, h, sc.max_depth)
    b = OracleScene(C.pointer(edited)).render(base.camera, w, h, base.max_depth)
    before = OracleScene(base.raw).render(base.camera, w, h, base.max_depth)
    assert np.array_equal(a["rgb_u8"], b["rgb_u8"]) and np.array_equal(a["hit_ids"], b["hit_ids"])
    assert a["rays"] == b["rays"]
    assert not np.array_equal(a["rgb_u8"], before["rgb_u8"])


def test_update_keeps_a_table_given_as_none_and_can_remove_every_light():
    sc = load_scene("cornellBox")
    mats = sc.materials
    sc.update(lights=[])
    assert sc.raw.contents.n_lights == 0 and sc.flat.contents.n_lights == 0 and len(sc.lights) == 0
    assert [bytes(x) for x in sc.materials] == [bytes(x) for x in mats]
    sc.update()
    assert len(sc.lights) == 0


def test_python_side_argument_errors():
    sc = load_scene("cornellBox")
    mats = sc.materials
    with pytest.raises(ValueError, match="materials"):
        sc.update(materials=list(mats)[:-1])
    with pytest.raises(TypeError):
        sc.update(lights=[mats[0]])
    with pytest.raises(TypeError):
        sc.update(materials=[1, 2, 3])
    assert [bytes(x) for x in sc.materials] == [bytes(x) for x in mats]


# ---------------------------------------------------------------------------------------------- the planner
@pytest.fixture(scope="module")
def planner():
    L = temp_library("scene_update", SOURCES, FLAGS)
    L.su_classify.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    L.su_lit_mask.restype = C.c_uint32
    L.su_lit_mask.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    L.su_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    return L


def mat(kind=capi.RH_MAT_DIFFUSE, c=(0.5, 0.5, 0.5), ior=1.5):
    m = capi.rh_material()
    m.kind, m.ior, m.texture = kind, ior, -1
    m.color1[:] = c
    return m


def light(kind=capi.RH_LIGHT_POINT, vec=(0, 5, 0), color=(1, 1, 1)):
    x = capi.rh_light()
    x.kind = kind
    x.vec[:], x.color[:] = vec, color
    return x


def arr(kind, rows):
    return (kind * max(len(rows), 1))(*rows)


def classify(L, om, nm, ol, nl, obj_mat):
    o = (C.c_int32 * max(len(obj_mat), 1))(*obj_mat)
    return L.su_classify(arr(capi.rh_material, om), arr(capi.rh_material, nm), len(om), arr(capi.rh_light, ol), len(ol),
                         arr(capi.rh_light, nl), len(nl), o, len(obj_mat))


def plan(L, old_index, ol, nl, n_meshes):
    cap = 64
    out = (C.c_uint32 * (4 * cap))()
    idx = None if old_index is None else (C.c_uint32 * len(old_index))(*old_index)
    n = L.su_plan(idx, arr(capi.rh_light, ol), len(ol), arr(capi.rh_light, nl), len(nl), n_meshes, cap, out)
    return [tuple(out[4 * k:4 * k + 4]) for k in range(n)]


def index_of(n_lights, entries):
    """light_map_index of n_lights lights: entries {(light, mesh): map}."""
    idx = [EMPTY] * (8 * n_lights)
    for (li, m), k in entries.items():
        idx[li * 8 + m] = k
    return idx


P0, P1, P2 = light(vec=(0, 5, 0)), light(vec=(3, 5, 0)), light(vec=(-3, 5, 1))
D0 = light(kind=capi.RH_LIGHT_DIRECTIONAL, vec=(0, -1, 0))


def test_classes(planner):
    m = [mat(), mat(capi.RH_MAT_MIRROR), mat(capi.RH_MAT_EMMIT)]
    objs = [0, 1, 2, 0]
    assert classify(planner, m, m, [P0, P1], [P0, P1], objs) == NONE
    recoloured = [mat(c=(0.1, 0.2, 0.3)), m[1], m[2]]
    brighter = light(vec=(0, 5, 0), color=(2, 2, 2))
    brighter.radius = 3.0
    assert classify(planner, m, recoloured, [P0, P1], [brighter, P1], objs) == COLOURS
    assert classify(planner, m, [mat(ior=1.33), m[1], m[2]], [P0], [P0], objs) == TABLES  # ior decides refraction
    assert classify(planner, m, [mat(capi.RH_MAT_PLASTIC), m[1], m[2]], [P0], [P0], objs) == TABLES
    assert classify(planner, m, m, [P0, P1], [P0, light(vec=(3, 6, 0))], objs) == TABLES  # one light moved
    assert classify(planner, m, m, [P0, P1], [P0], objs) == TABLES                         # a light removed
    assert classify(planner, m, m, [P0], [P0, P1], objs) == TABLES                         # a light added
    assert classify(planner, m, m, [P0, P1], [P1, P0], objs) == TABLES                     # reordered
    assert classify(planner, m, [m[0], mat(capi.RH_MAT_EMMIT), m[2]], [P0], [P0], objs) == EMITTERS
    assert classify(planner, m, [m[0], m[1], mat()], [P0], [P0], objs) == EMITTERS
    # a material no object uses may become an emitter without changing the emitter set
    assert classify(planner, m, [m[0], mat(capi.RH_MAT_EMMIT), m[2]], [P0], [P0], [0, 2]) == TABLES


def test_lit_mask(planner):
    L = planner
    assert L.su_lit_mask(arr(capi.rh_light, [P0, P1, P2]), 3, arr(capi.rh_light, [P0, light(vec=(3, 6, 0)), P2]), 3) == 0b010
    assert L.su_lit_mask(arr(capi.rh_light, [P0, P1]), 2, arr(capi.rh_light, [P0, P1, D0]), 3) == 0b100
    # removed: index 1 holds another light now, index 2 none (its bits are only cleared)
    assert L.su_lit_mask(arr(capi.rh_light, [P0, P1, P2]), 3, arr(capi.rh_light, [P0, P2]), 2) == 0b110
    assert L.su_lit_mask(arr(capi.rh_light, [P0, P1]), 2, arr(capi.rh_light, []), 0) == 0b11
    assert L.su_lit_mask(arr(capi.rh_light, [P0, P1]), 2, arr(capi.rh_light, [P1, P0]), 2) == 0b11
    moved_to_dir = light(kind=capi.RH_LIGHT_DIRECTIONAL, vec=(0, 5, 0))
    assert L.su_lit_mask(arr(capi.rh_light, [P0]), 1, arr(capi.rh_light, [moved_to_dir]), 1) == 0b1
    many = [light(vec=(i, 5, 0)) for i in range(14)]
    assert L.su_lit_mask(arr(capi.rh_light, []), 0, arr(capi.rh_light, many), 14) == 0x0FFF


def test_plan_one_light_moved(planner):
    # two meshes; map of (P1, mesh 0) was not worth having
    old = index_of(3, {(0, 0): 0, (2, 0): 1, (0, 1): 2, (1, 1): 3, (2, 1): 4})
    moved = light(vec=(3, 6, 0))
    assert plan(planner, old, [P0, P1, P2], [P0, moved, P2], 2) == [
        (0, 0, 0, 0), (0, 1, 1, EMPTY), (0, 2, 0, 1),
        (1, 0, 0, 2), (1, 1, 1, EMPTY), (1, 2, 0, 4)]


def test_plan_lights_added_removed_and_reordered(planner):
    old = index_of(2, {(0, 0): 0, (1, 0): 1})
    # added: a point light after a directional one; the old lights keep their maps
    assert plan(planner, old, [P0, P1], [P0, D0, P1, P2], 1) == [(0, 0, 0, 0), (0, 2, 0, 1), (0, 3, 1, EMPTY)]
    # removed: the remaining light takes its map from its old index
    assert plan(planner, old, [P0, P1], [P1], 1) == [(0, 0, 0, 1)]
    # reordered: the maps move with their lights
    assert plan(planner, old, [P0, P1], [P1, P0], 1) == [(0, 0, 0, 1), (0, 1, 0, 0)]
    # a duplicate position takes over each old map at most once
    assert plan(planner, index_of(1, {(0, 0): 0}), [P0], [P0, P0], 1) == [(0, 0, 0, 0), (0, 1, 1, EMPTY)]
    # a point light that became directional has no map; one that became a point light is rasterised
    assert plan(planner, old, [P0, P1], [light(kind=capi.RH_LIGHT_DIRECTIONAL, vec=(0, 5, 0)), P1], 1) == [(0, 1, 0, 1)]


def test_plan_usefulness_flip_keeps_the_old_verdict(planner):
    # an old map that was not worth having stays so for the same light and triangles (no raster, no map); a moved
    # light's maps are built anew whatever their old verdict
    old = index_of(2, {(1, 0): 0})
    assert plan(planner, old, [P0, P1], [P0, P1], 1) == [(0, 0, 0, EMPTY), (0, 1, 0, 0)]
    assert plan(planner, old, [P0, P1], [light(vec=(0, 4, 0)), P1], 1) == [(0, 0, 1, EMPTY), (0, 1, 0, 0)]


def test_plan_without_reusable_tables_rasterises_every_pair(planner):
    # emitter set changed, another resolution or no old tables: nothing to carry over
    assert plan(planner, None, [P0, P1], [P0, P1], 2) == [
        (0, 0, 1, EMPTY), (0, 1, 1, EMPTY), (1, 0, 1, EMPTY), (1, 1, 1, EMPTY)]
    assert plan(planner, None, [P0], [D0], 3) == []
